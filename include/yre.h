/* yre.h -- C ABI of libyre.so, the B200 (sm_100a) kernels behind the yolo-re detection
 * inference hot path.
 *
 * The reference (ariaghora/yolo-re) is pure Python/PyTorch and has no FFI of its own; the
 * "interface each entry point replaces" is therefore the torch / torchvision call the
 * reference makes at the cited file:line (paths relative to the reference checkout).
 * INTEGRATION.md shows the ctypes binding a maintainer of the reference would add.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless stated;
 *   - every call is asynchronous on the caller's stream (cudaStream_t passed as void*);
 *   - returns 0 (YRE_OK) or a negative YRE_E* code; text via yre_last_error() (thread-local);
 *   - nothing here falls back to the CPU, cuDNN, cuBLAS or torch: an unsupported request
 *     fails with YRE_EUNSUPPORTED.
 *
 * Data layout: activations are channels-last ("NHWC") with an explicit channel window so that
 * chunk()/cat() of the reference (blocks/gelan.py:59-62, blocks/csp.py:60, blocks/common.py:33)
 * become zero-copy views of one wider buffer.
 *
 * Activation types: YRE_BF16 (the default product precision), YRE_F16 (IEEE half: 3 more significant bits than bf16,
 * but finite only up to +-65504 -- larger results are stored as +-inf, not saturated -- and normal only down to 2^-14)
 * and YRE_F32 (the validation precision).  Every kernel accumulates in fp32 whichever 16-bit type it reads and writes.
 * The two 16-bit types never mix within one call: an op whose 16-bit operands disagree fails with YRE_EUNSUPPORTED.
 */
#ifndef YRE_H
#define YRE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define YRE_VERSION 200

typedef void* yre_stream_t; /* cudaStream_t */

enum { YRE_OK = 0, YRE_EINVAL = -1, YRE_ECUDA = -2, YRE_EUNSUPPORTED = -3, YRE_ENOMEM = -4 };
enum { YRE_BF16 = 0, YRE_F32 = 1, YRE_F16 = 2 };
enum { YRE_ACT_NONE = 0, YRE_ACT_SILU = 1 };
enum { YRE_NHWC = 0, YRE_PHASE4 = 1 };
enum { YRE_ENGINE_AUTO = 0, YRE_ENGINE_FFMA = 1, YRE_ENGINE_TCGEN05 = 2 };

/* A channel window [c_off, c_off+C) of a channels-last activation buffer.
 *   YRE_NHWC   : element (b,y,x,c) at ((b*H + y)*W + x)*C_total + c_off + c
 *   YRE_PHASE4 : the logical HxW map stored as 4 parity planes so that a stride-2 3x3 conv
 *                becomes unit-stride per tap:  plane p = (y&1)*2 + (x&1), Hp=(H+1)/2, Wp=(W+1)/2,
 *                element at (((p*B + b)*Hp + y/2)*Wp + x/2)*C_total + c_off + c; cells of a plane
 *                that have no source pixel (odd H or W) hold zeros.                              */
typedef struct yre_view {
    void*   ptr;
    int32_t dtype;    /* YRE_BF16 | YRE_F16 | YRE_F32 */
    int32_t layout;   /* YRE_NHWC | YRE_PHASE4 */
    int32_t B, H, W;  /* logical extent */
    int32_t C_total;  /* channels of the physical buffer (pixel pitch) */
    int32_t c_off;    /* first channel of the window */
    int32_t C;        /* channels in the window */
} yre_view;

/* ---- library ---------------------------------------------------------------------------- */
int         yre_version(void);
const char* yre_last_error(void);
/* 0 if the CURRENT cuda device is sm_100 (B200); YRE_EUNSUPPORTED otherwise. */
int         yre_device_check(void);

/* ---- K1: fused convolution ----------------------------------------------------------------
 * Replaces Conv.forward = act(bn(conv(x)))              src/yolo/blocks/conv.py:88-89
 *          RepConv.forward (3x3 + 1x1 branches)          src/yolo/blocks/conv.py:140-141
 *          RepNBottleneck.forward residual               src/yolo/blocks/bottleneck.py:49-51
 *          head nn.Conv2d (bias, no BN/act)              src/yolo/heads/detect.py:52,61
 *          CBLinear.forward                              src/yolo/blocks/auxiliary.py:61-62
 * with BN folded into (w, bias) by the host, RepConv's 1x1 folded into the 3x3 centre tap and
 * grouped convs expanded to block-diagonal dense weights.
 *   y = [res +] act(conv(x, w) + bias),   kernel k in {1,3}, pad k/2, stride in {1,2}.
 * w: [Cout][k][k][Cin], same dtype as x.  bias: fp32 [Cout] (may be NULL).
 * y and res are x's 16-bit type or fp32 (a bf16 x with an fp16 y or res, or the reverse, is YRE_EUNSUPPORTED).
 * engine: YRE_ENGINE_TCGEN05 = implicit-GEMM on tcgen05/TMEM with TMA-staged operands
 * (x/w bf16 or fp16, of the same type; fp32 accumulation; Cin%32==0, Cout%16==0, stride-2 needs a YRE_PHASE4 input);
 * YRE_ENGINE_FFMA = fp32-accurate SIMT implicit GEMM (the fp32 validation mode and the
 * fallback for shapes tcgen05 does not take); YRE_ENGINE_AUTO picks tcgen05 when eligible.
 *
 * xu (optional, xu.ptr != NULL; 1x1 stride-1 convs only): a HALF-resolution view [B][H/2][W/2] whose 2x nearest-neighbour
 * upsample supplies the FIRST xu.C input channels, x the remaining x.C -- i.e. the conv reads
 * cat([Upsample(2, nearest)(xu), x], dim=channels) without that tensor ever being written:
 *   nn.Upsample + Concat + the consumer's 1x1 conv   src/yolo/model/parser.py:159-171, src/yolo/blocks/common.py:32-33,
 *                                                     src/yolo/blocks/gelan.py:58 (conv_in of the neck's RepNCSPELAN4)
 * w is then [Cout][1][1][xu.C + x.C].  On the tcgen05 engine the upsample is a TMA addressing mode (a tensor map over xu
 * whose two duplicated dimensions have global stride 0); results are bit-identical to running the conv on the
 * materialised concat. */
typedef struct yre_conv_desc {
    yre_view    x, y, res;  /* res.ptr == NULL: no residual; res has y's shape */
    const void* w;
    const float* bias;
    int32_t     k, stride, act, engine;
    yre_view    xu;         /* xu.ptr == NULL: plain conv */
} yre_conv_desc;
int yre_conv(const yre_conv_desc* d, yre_stream_t s);
/* Host-only query: the string yre_plan_op_variant reports for d on the tcgen05 engine of a device with num_sms SMs.  No
 * device is touched and no pointer is dereferenced.  d is validated as yre_conv validates it; beyond that, of the
 * pointers only whether res.ptr and xu.ptr are NULL changes the result (address alignment is not checked).
 * YRE_EUNSUPPORTED, with the reason in yre_last_error(), when the engine does not take the shape or its tile does not fit
 * shared memory. */
int yre_conv_tc_describe(const yre_conv_desc* d, int32_t num_sms, char* out, int32_t cap);
/* Host-only query, like yre_conv_tc_describe: the work schedule the tcgen05 kernel walks for the first n (1 <= n <= y.B)
 * images of d on a device with num_sms SMs -- what a plan compiled for d.y.B images launches in yre_plan_run_batch(n).
 * The tiling (tw x th x tb pixels x images by block_n channels) is the one chosen for all y.B images; n only shortens
 * the walk to the first tiles_b = ceil(n / tb) image tiles and sizes the persistent grid for them.  Work item w of
 * CTA (pair) c, for w = c, c + G, c + 2G ... (G = grid, or grid / 2 CTA pairs), decodes images outermost:
 *   YRE_TC_GENERIC, YRE_TC_HALO_WS: tile w -> N tile w % tiles_n, M tile m = w / tiles_n;
 *   YRE_TC_GENERIC_CTA2: unit w -> N tile w % tiles_n, M tiles 2 (w / tiles_n) + {0, 1} (one per CTA of the pair);
 *   YRE_TC_HALO_STREAM: unit w -> N tile w / upn, M tiles npair (w % upn) + {0 .. npair-1};
 * M tile m -> x tile m % tiles_x, y tile (m / tiles_x) % tiles_y, image tile m / (tiles_x tiles_y).  ybx = 1: the tile's
 * pixel rows run (y, image, x) (8 x 8 pixels of two images). */
enum { YRE_TC_GENERIC = 0, YRE_TC_GENERIC_CTA2 = 1, YRE_TC_HALO_WS = 2, YRE_TC_HALO_STREAM = 3 };
typedef struct yre_tc_schedule {
    int32_t kind, ybx;
    int32_t tw, th, tb, block_n;
    int32_t tiles_x, tiles_y, tiles_b, tiles_n;
    int32_t mtiles;   /* tiles_x * tiles_y * tiles_b */
    int32_t npair, upn;
    int32_t work;     /* tiles (GENERIC, HALO_WS) or units (GENERIC_CTA2, HALO_STREAM) */
    int32_t grid;     /* CTAs launched */
} yre_tc_schedule;
int yre_conv_tc_schedule(const yre_conv_desc* d, int32_t num_sms, int32_t n, yre_tc_schedule* out);

/* ---- K2: first conv straight from the image ------------------------------------------------------
 * Replaces layers.stem1 (Conv 3x3 s2 on the input image; configs/models/gelan-c.yaml stem1,
 * src/yolo/blocks/conv.py:88-89).  x_nchw: fp32 [B][Cin<=4][H][W]; w: fp32 [Cout][3][3][Cin];
 * y may be YRE_NHWC or YRE_PHASE4, bf16, fp16 or fp32 (a 16-bit y rounds image and weights to that type for the
 * tensor-core kernels; the products are exact and accumulate in fp32).
 * x_u8_hwc (optional; when non-NULL it is the input and x_nchw is ignored): uint8 [B][H][W][3] frames in BGR
 * order (cv2.imread layout), Cin must be 3.  Fuses what the reference does on the host before model()
 * (scripts/detect.py:223-227): BGR->RGB, HWC->CHW, .float() / 255 (fp32 division, round to nearest). */
typedef struct yre_stem_desc {
    const float* x_nchw;
    int32_t      B, Cin, H, W;
    yre_view     y;
    const float* w;
    const float* bias;
    int32_t      stride, act;
    const uint8_t* x_u8_hwc;
} yre_stem_desc;
int yre_stem_conv(const yre_stem_desc* d, yre_stream_t s);

/* ---- K3: ADown pre-pool ----------------------------------------------------------------------
 * Replaces F.avg_pool2d(x,2,1,0) -> chunk(2,1) -> [ . | F.max_pool2d(.,3,2,1) ]
 *                                                        src/yolo/blocks/downsample.py:41-44
 * avg_lo: first C/2 channels of the (H-1)x(W-1) average map (YRE_PHASE4 or YRE_NHWC);
 * max_hi: max_pool(3,2,1) of the last C/2 channels of that map, NHWC [B,Ho,Wo,C/2].
 * x, avg_lo and max_hi share one dtype (bf16, fp16 or fp32).  The 16-bit types average with packed 16-bit adds
 * (three extra roundings to the storage type); fp32 sums in torch's order. */
int yre_adown_prepool(const yre_view* x, const yre_view* avg_lo, const yre_view* max_hi, yre_stream_t s);

/* ---- K4: SPPELAN pooling pyramid --------------------------------------------------------------
 * Replaces three chained nn.MaxPool2d(5,1,2)             src/yolo/blocks/sppelan.py:44-47
 * (== windows 5 / 9 / 13 of the same input).  x and the outputs share one dtype (bf16, fp16 or fp32); exact. */
int yre_spp_maxpool(const yre_view* x, const yre_view* y5, const yre_view* y9, const yre_view* y13, yre_stream_t s);

/* ---- K5: nearest x2 upsample into a concat slice ----------------------------------------------
 * Replaces nn.Upsample(scale_factor=2, mode="nearest") + Concat
 *                                  src/yolo/model/parser.py:159-171, src/yolo/blocks/common.py:32-33 */
int yre_upsample2x(const yre_view* x, const yre_view* y, yre_stream_t s);   /* x, y: one dtype; exact */

/* ---- K8: CBFuse (yolov9-c auxiliary branch) ----------------------------------------------------
 * Replaces CBFuse.forward: sum_i nearest_resize(src_i -> target size) + target
 *                                                        src/yolo/blocks/auxiliary.py:100-110 */
/* all views share one dtype (bf16, fp16 or fp32); the sum runs in fp32 and is rounded once to y's type */
int yre_cbfuse_sum(const yre_view* srcs, int32_t n_src, const yre_view* target, const yre_view* y, yre_stream_t s);

/* ---- layout conversion at the API boundary ----------------------------------------------------
 * the view may be bf16, fp16 or fp32: nchw_to_view rounds to nearest even (fp16 overflows to +-inf), view_to_nchw is exact */
int yre_nchw_to_view(const float* x_nchw, const yre_view* y, yre_stream_t s);  /* fp32 NCHW -> view  */
int yre_view_to_nchw(const yre_view* x, float* y_nchw, yre_stream_t s);        /* view -> fp32 NCHW  */

/* ---- K6: DFL decode + class scoring -----------------------------------------------------------
 * Replaces DetectDFL.forward tail                        src/yolo/heads/detect.py:93-108
 *          DFL.forward                                   src/yolo/heads/dfl.py:46-50
 *          make_anchors / dist2bbox                      src/yolo/heads/anchor.py:26-40, 57-64
 * raw[l]: NHWC view [B,Hl,Wl,64+nc] (fp32 or bf16) = cat(box logits, class logits) of level l;
 * dfl_w: the 16 HOST values of layers.detect.dfl.conv.weight (held by value so that the launch
 * neither syncs nor reads host memory later); y: fp32 [B][A][4+nc], A = sum Hl*Wl, row =
 * (cx,cy,w,h in pixels, sigmoid class scores).  The reference's [B,4+nc,A] is its transpose. */
typedef struct yre_decode_desc {
    yre_view     raw[8];
    float        stride[8];
    int32_t      levels, nc;
    float        dfl_w[16];
    float*       y;
} yre_decode_desc;
int yre_dfl_decode_score(const yre_decode_desc* d, yre_stream_t s);
/* K6 for segmentation heads (upstream YOLOv9's Segment on DetectDFL): dec is decoded exactly as yre_dfl_decode_score
 * decodes it, and the same launch writes mc: fp32 [B][A][nm], row a = the nm mask coefficients of anchor a, read from
 * mask[l] at the anchor's pixel.  mask[l]: fp32 NHWC view [B,Hl,Wl,nm] of level l's mask tower output, with raw[l]'s
 * extent.  So the coefficients of a kept detection are mc[b][keep_anchor[b][j]].  nm must be 32; anything else, or a
 * mask view of another dtype, layout or extent, fails with YRE_EINVAL before the launch. */
typedef struct yre_decode_masks_desc {
    yre_decode_desc dec;
    yre_view        mask[8];
    int32_t         nm;
    float*          mc;
} yre_decode_masks_desc;
int yre_dfl_decode_score_masks(const yre_decode_masks_desc* d, yre_stream_t s);

/* ---- K7: batched class-aware NMS --------------------------------------------------------------
 * Replaces non_max_suppression                           src/yolo/utils/nms.py:19-94
 *          torchvision.ops.nms via _nms                   src/yolo/utils/nms.py:97-104
 * pred: fp32 [B][A][4+nc] contiguous.  classes: device int32 [n_classes] or NULL.
 * out: fp32 [B][max_det][6] rows (x1,y1,x2,y2,conf,cls) in descending score order;
 * counts: int32 [B]; keep_anchor: int64 [B][max_det] (anchor index of every kept row).
 * Results are bit-identical to the reference given the same pred.  No pre-NMS top-k cap. */
typedef struct yre_nms_desc {
    const float*   pred;
    int32_t        B, A, nc;
    float          conf_thres;  /* strict >, compared in fp32 (nms.py:57) */
    double         iou_thres;   /* fp32 IoU compared against this as a DOUBLE, as torchvision's CPU kernel does */
    int32_t        max_det;
    const int32_t* classes;
    int32_t        n_classes;   /* < 0: no class filter */
    int32_t        agnostic;
    float*         out;
    int32_t*       counts;
    int64_t*       keep_anchor;
    void*          workspace;
    size_t         workspace_bytes;
    /* optional (may be NULL): fp32 [B][5] = (pad_w, pad_h, gain, orig_w, orig_h) per image.  When given, the kept
     * boxes are written mapped back to the original image -- scale_boxes (scripts/detect.py:74-109) fused into the
     * output pass with the arithmetic of yre_scale_boxes: clamp((v - pad) / gain, 0, orig), fp32, true division.
     * Suppression itself always runs on the un-scaled boxes, as in the reference. */
    const float*   scale;
} yre_nms_desc;
size_t yre_nms_workspace_bytes(int32_t B, int32_t A);
int    yre_nms_batched(const yre_nms_desc* d, yre_stream_t s);
/* Only the candidate pass of yre_nms_batched (counters reset + filter / argmax / compaction into the workspace):
 * the HBM-bound stage on its own, for stage timing (bench.py roofline.stages) and profiling.  d->out / counts /
 * keep_anchor are not touched. */
int    yre_nms_filter_only(const yre_nms_desc* d, yre_stream_t s);

/* Multi-label NMS: upstream YOLOv9's non_max_suppression(..., multi_label=True) candidate set, which its val.py uses for
 * every published mAP (val.py: `non_max_suppression(preds, conf_thres, iou_thres, labels=lb, multi_label=True, ...)`;
 * utils/general.py: `i, j = (x[:, 5:mi] > conf_thres).nonzero(as_tuple=False).T`), on top of yolo-re's algorithm.
 * Extends nms.py:54-59 (first-max class per anchor, strict >, class filter): every (anchor a, class c) with
 * score[a][c] > conf_thres (and c in classes, when given) is a candidate, in the order (a ascending, then c).  Everything
 * after that is nms.py:61-92 unchanged: xyxy boxes, the class offset c * (max_coord + 1) with max_coord over the candidate
 * boxes, agnostic, a stable descending score sort (ties -> lower (a, c)), greedy IoU, keep[:max_det] with no pre-NMS cap.
 * Not upstream's max_wh = 7680 offset, max_nms = 30000 cap or unstable argsort.
 * Same descriptor and outputs as yre_nms_batched; keep_anchor is the anchor index, so several rows may share one anchor.
 * The workspace holds pow2ceil(A * nc) keys per image.  A * nc above 2^30 fails with YRE_EUNSUPPORTED (the workspace
 * size is then 0), as does an nc whose 32 rows do not fit the filter's 48 KB of shared memory (nc > 380). */
size_t yre_nms_multi_label_workspace_bytes(int32_t B, int32_t A, int32_t nc);
int    yre_nms_batched_multi_label(const yre_nms_desc* d, yre_stream_t s);
/* the candidate pass of yre_nms_batched_multi_label on its own (stage timing, as yre_nms_filter_only) */
int    yre_nms_multi_label_filter_only(const yre_nms_desc* d, yre_stream_t s);

/* ---- K8/K9: the steps either side of the path (SURVEY.md 8f row 1) -----------------------------------
 * K8 replaces letterbox                                  scripts/detect.py:40-71
 *             cv2.resize(INTER_LINEAR) on uint8          (OpenCV; 8-bit fixed point, bit-exact restatement)
 *             BGR->RGB, HWC->CHW, .float() / 255         scripts/detect.py:223-227
 * src: uint8 [h][w][3] (cv2.imread layout, rows `row_pitch` bytes apart) on the DEVICE.
 * The destination is an out_h x out_w rectangle (S x S when out_h = out_w = 0, the square letterbox):
 * out_mode YRE_LB_F32_CHW: dst = float [3][out_h][out_w], channel order reversed (RGB), value / 255 -- the tensor the
 *                          reference feeds to model(); YRE_LB_U8_HWC: dst = uint8 [out_h][out_w][3], what letterbox()
 *                          returns.
 * The geometry (un-padded size, padding, destination extent) comes from yre_letterbox_geometry_rect, which mirrors
 * the reference's Python arithmetic including round-half-to-even. */
enum { YRE_LB_F32_CHW = 0, YRE_LB_U8_HWC = 1 };
typedef struct yre_letterbox_desc {
    const uint8_t* src;
    int32_t        h, w;
    int64_t        row_pitch;
    int32_t        new_shape;        /* S */
    int32_t        new_w, new_h;     /* resized, un-padded size */
    int32_t        top, left;        /* padding before the image */
    uint8_t        color[4];         /* pad colour in SOURCE channel order (114,114,114), 4th byte unused */
    int32_t        out_mode;
    void*          dst;
    int32_t        out_h, out_w;     /* destination extent; 0, 0 = new_shape x new_shape */
} yre_letterbox_desc;
/* host helper: letterbox geometry for a target (new_h, new_w) from the source (d->h, d->w).
 *   r = min(new_h / h, new_w / w); the resized size is round(w r) x round(h r), half to even;
 *   stride > 0 ("auto") reduces each axis' padding modulo stride: the smallest stride-multiple rectangle;
 *   each padding d/2 is split round(d/2 - 0.1) before, round(d/2 + 0.1) after.
 * Fills new_w/new_h/top/left/out_h/out_w of *d; ratio and the (pad_w, pad_h) pair the reference returns (int(d/2),
 * truncated) go to the optional outputs.  Fails with YRE_EINVAL when the resized image is empty. */
int yre_letterbox_geometry_rect(yre_letterbox_desc* d, int32_t new_h, int32_t new_w, int32_t stride, double* ratio,
                                int32_t* pad_w, int32_t* pad_h);
/* yre_letterbox_geometry_rect(d, d->new_shape, d->new_shape, 0, ...): the square letterbox */
int yre_letterbox_geometry(yre_letterbox_desc* d, double* ratio, int32_t* pad_w, int32_t* pad_h);
int yre_letterbox_u8(const yre_letterbox_desc* d, yre_stream_t s);
/* n images sharing the destination extent and out_mode in as few launches as possible (32 images per launch); their
 * resized sizes and offsets inside the destination may differ */
int yre_letterbox_u8_batch(const yre_letterbox_desc* d, int32_t n, yre_stream_t s);
/* K14: K8 on 4:2:0 YUV frames, the output of hardware and software video decoders.  Output is defined as K8 applied to
 * cv2.cvtColor(frame, COLOR_YUV2BGR_<format>), bit for bit: limited range, 20-bit fixed point, nearest chroma (one
 * (U, V) sample per 2 x 2 luma block).  YRE_YUV_BT601 uses cv2's coefficients, YRE_YUV_BT709 the same scheme on
 * the BT.709 ones (HD video).  Each plane has its own pointer and pitch (pitched decoder surfaces, chroma apart from
 * luma); cv2's single (h*3/2) x w array is the case of one allocation. */
enum { YRE_YUV_NV12 = 0, YRE_YUV_NV21 = 1, YRE_YUV_I420 = 2, YRE_YUV_YV12 = 3 };
enum { YRE_YUV_BT601 = 0, YRE_YUV_BT709 = 1 };
typedef struct yre_yuv420_planes {
    const uint8_t* luma;              /* h rows of w bytes, luma_pitch bytes apart */
    int64_t        luma_pitch;
    const uint8_t* chroma[2];         /* NV12 / NV21: [0] = the interleaved UV / VU plane (h/2 rows of w bytes), [1] = NULL;
                                         I420: [0] = U, [1] = V; YV12: [0] = V, [1] = U (h/2 rows of w/2 bytes each) */
    int64_t        chroma_pitch;      /* of every chroma plane */
    int32_t        format;            /* YRE_YUV_NV12 ... */
    int32_t        matrix;            /* YRE_YUV_BT601 / YRE_YUV_BT709 */
} yre_yuv420_planes;
/* n frames, planes[i] the source of d[i]: d[i] gives the luma extent h x w, the geometry, out_mode and dst as for
 * yre_letterbox_u8_batch (geometry from yre_letterbox_geometry_rect on h x w); its src and row_pitch must be 0.
 * YRE_EINVAL before any launch for an odd h or w, a pitch shorter than its plane's row, an unknown format or matrix,
 * or a null plane. */
int yre_letterbox_yuv420_batch(const yre_letterbox_desc* d, const yre_yuv420_planes* planes, int32_t n, yre_stream_t s);
/* K9 replaces scale_boxes                                scripts/detect.py:74-109
 * boxes: n rows of xyxy fp32, `row_stride` floats apart (6 for detection rows), updated in place:
 * x = clamp((x - pad_w) / gain, 0, orig_w), y likewise -- fp32, true division, as torch does on the CPU. */
int yre_scale_boxes(float* boxes, int32_t n, int32_t row_stride, float pad_w, float pad_h, float gain,
                    float orig_w, float orig_h, yre_stream_t s);

/* ---- K11: detection -> ground-truth matching for mAP (SURVEY.md 8f row 3) ------------------------------
 * Replaces the per-prediction loop of compute_map        src/yolo/eval/metrics.py:137-176
 *          box_iou                                        src/yolo/eval/metrics.py:10-31
 * det: fp32 rows [x1,y1,x2,y2,conf,cls], `det_stride` floats apart, the images' rows concatenated; det_off: int32
 * [B+1] row ranges.  Rows of one image must be in matching order = descending score, ties in original order (what
 * yre_nms_batched emits).  gt_boxes fp32 [M][4] xyxy (16-byte aligned), gt_cls int32 [M], gt_off int32 [B+1].
 * thr: n_thr <= 16 IoU thresholds (doubles, compared after a cast to fp32 exactly like torch's `best_iou >= thr`).
 * tp: uint8 [N][n_thr]: 1 = true positive at that threshold.  max_gt_per_image: host-known bound (<= 4096). */
typedef struct yre_match_desc {
    const float*   det;
    int32_t        det_stride;
    const int32_t* det_off;
    const float*   gt_boxes;
    const int32_t* gt_cls;
    const int32_t* gt_off;
    int32_t        B;
    int32_t        n_thr;
    double         thr[16];
    int32_t        max_gt_per_image;
    uint8_t*       tp;
} yre_match_desc;
int yre_match_detections(const yre_match_desc* d, yre_stream_t s);

/* ---- K12/K13: test-time augmentation (YOLOv5/v8/v9 `model(x, augment=True)`) -----------------------------
 * Upstream's _forward_augment runs the batch at three branches (s, flip) = (1, none), (0.83, left-right), (0.67, none)
 * and concatenates their decoded predictions before NMS:
 *   scale_img       flip the width axis (branch 1), F.interpolate(bilinear, align_corners=False) to (int(h s), int(w s)),
 *                   F.pad(value=0.447) right and bottom to (ceil(h s / 32) 32, ceil(w s / 32) 32)
 *   _descale_pred   columns 0..3 / s (fp32), x = w - x for the flipped branch (w: the ORIGINAL width)
 *   _clip_augmented g = 21 (1 + 4 + 16, three levels): branch 0 drops its last A0 / g anchors (P5), branch 2 its first
 *                   16 (A2 / g) (P3); exact for every stride-32 rectangle.
 * oracle/tta_ref.py restates the definition.
 *
 * Host-only: the branch geometry of an h x w input (positive multiples of 32, at most 65536).  YRE_EINVAL otherwise. */
#define YRE_TTA_BRANCHES 3
typedef struct yre_tta_geom {
    int32_t h, w;                        /* the input */
    float   scale[YRE_TTA_BRANCHES];     /* (float)s: 1, 0.83, 0.67 */
    int32_t flip[YRE_TTA_BRANCHES];      /* 0, 1, 0 */
    int32_t rh[YRE_TTA_BRANCHES], rw[YRE_TTA_BRANCHES];         /* resized extent int(h s) x int(w s) */
    int32_t out_h[YRE_TTA_BRANCHES], out_w[YRE_TTA_BRANCHES];   /* padded branch input, multiples of 32 */
    int32_t A[YRE_TTA_BRANCHES];         /* anchors of the branch's y (strides 8, 16, 32) */
    int32_t a_begin[YRE_TTA_BRANCHES], a_end[YRE_TTA_BRANCHES];  /* anchor window kept by _clip_augmented */
    int32_t A_tot;                       /* sum of the windows */
} yre_tta_geom;
int yre_tta_geometry(int32_t h, int32_t w, yre_tta_geom* out);
/* K12: one branch's input.  x: fp32 NCHW RGB [B][3][H][W] (x_nchw) or uint8 BGR frames [B][H][W][3] (x_u8_hwc, the
 * other NULL; the value is (float)v / 255 with channel c read from byte 2 - c, as K8's fp32 mode and the uint8 stem).
 * y: fp32 NCHW [B][3][out_h][out_w]; the first n (1 <= n <= B) images are written.  Pixel (Y, X) with Y < rh, X < rw is
 * the bilinear sample of the (flipped) source, in fp32 without contraction:
 *   scale = (float)in / out;  src = max(scale (d + 0.5) - 0.5, 0);  i0 = (int)src;  i1 = i0 + (i0 < in - 1);
 *   l1 = src - i0;  l0 = 1 - l1;  v = hl0 (wl0 v00 + wl1 v01) + hl1 (wl0 v10 + wl1 v11)
 * every other pixel is 0.447f.  Pointers 4-byte aligned; 1 <= rh <= out_h, 1 <= rw <= out_w. */
typedef struct yre_tta_scale_desc {
    const float*   x_nchw;
    const uint8_t* x_u8_hwc;
    int32_t        B, n, H, W;
    int32_t        flip;             /* 1: mirror the width axis before the resize */
    int32_t        rh, rw;
    int32_t        out_h, out_w;
    float*         y;
} yre_tta_scale_desc;
int yre_tta_scale_img(const yre_tta_scale_desc* d, yre_stream_t s);
/* K13: the merged predictions.  Branch i's y: fp32 [B][A_i][4+nc] (the K6 layout), rows [a_begin, a_end) of each of the
 * first n images are written, in branch order, to out fp32 [B][A_tot][4+nc], A_tot = sum of the windows:
 *   columns 0..3 / scale (fp32 division); then, when flip_w != 0, column 0 = (float)flip_w - column 0; classes copied.
 * y and out 16-byte aligned, 1 <= nc <= 4096, 1 <= n <= B, 0 <= a_begin < a_end <= A_i, scale > 0, flip_w >= 0. */
typedef struct yre_tta_merge_branch {
    const float* y;
    int32_t      A, a_begin, a_end;
    float        scale;
    int32_t      flip_w;
} yre_tta_merge_branch;
typedef struct yre_tta_merge_desc {
    yre_tta_merge_branch br[YRE_TTA_BRANCHES];
    int32_t              B, n, nc;
    float*               out;
} yre_tta_merge_desc;
int yre_tta_merge(const yre_tta_merge_desc* d, yre_stream_t s);

/* ---- K15: instance-segmentation masks of the kept detections ------------------------------------------------------
 * Replaces process_mask / process_mask_native / crop_mask        upstream YOLOv9 utils/segment/general.py
 * One launch for a batch, after yre_nms_batched (or its multi-label form): detection j < counts[b] of image b takes the
 * mask coefficients mc[b][keep_anchor[b][j]] and its box det[b][j][0..3] (xyxy).  With p = 1 / (1 + expf(-x)) of the logit
 * x = sum_k mc[k] proto[y][x][k] (fp32, k = 0..nm-1 in order, no contraction), masks[b][j] is, as uint8 0 / 1:
 *   YRE_MASK_PROTO   process_mask(upsample=False): out_h x out_w = mh x mw.  p cropped to the box scaled to proto pixels
 *                    (x * (float)(mw / in_w), y * (float)(mh / in_h)): pixel (r, c) kept when c >= x1, c < x2, r >= y1,
 *                    r < y2, else 0.  Then > 0.5.
 *   YRE_MASK_INPUT   process_mask(upsample=True): out_h x out_w = in_h x in_w.  The cropped map of YRE_MASK_PROTO, resized
 *                    bilinearly (align_corners=False, K12's arithmetic) to the input, then > 0.5.
 *   YRE_MASK_NATIVE  process_mask_native: p uncropped; gain = min(mh / h0, mw / w0), pad = ((mw - w0 gain) / 2,
 *                    (mh - h0 gain) / 2) in double; rows (int)pad_h .. (int)(mh - pad_h), columns likewise, resized
 *                    bilinearly to h0 x w0; cropped with the box in frame pixels; > 0.5.  (w0, h0) = (int) columns 3 and 4
 *                    of scale[b] (the rows yre_nms_desc.scale takes); image b writes the [0, h0) x [0, w0) window of its
 *                    out_h x out_w planes, clipped to them.
 * Only what can reach the output is computed: the box's proto pixels and their bilinear border.  Rows j >= counts[b]
 * (read on the device: no host sync, CUDA-graph capturable), images >= n and bytes outside a native window are not
 * written.  proto: fp32 NHWC [B][mh][mw][nm], pixels proto_pitch floats apart (a multiple of 4, >= nm), 16-byte aligned;
 * mc: fp32 [B][A][nm], 16-byte aligned; det: fp32 [B][max_det][6]; counts: int32 [B]; keep_anchor: int64 [B][max_det];
 * masks: uint8 [B][max_det][out_h][out_w].  YRE_EINVAL before any launch for a null pointer, nm != 32, an unknown mode,
 * a bad pitch or alignment, non-positive extents, 1 <= n <= B violated, or out_h x out_w other than the mode's. */
enum { YRE_MASK_PROTO = 0, YRE_MASK_INPUT = 1, YRE_MASK_NATIVE = 2 };
typedef struct yre_mask_desc {
    const float*   proto;
    int32_t        B, n, mh, mw, nm;
    int32_t        proto_pitch;
    const float*   mc;
    int32_t        A;
    const float*   det;
    const int32_t* counts;
    const int64_t* keep_anchor;
    int32_t        max_det;
    int32_t        mode;
    int32_t        in_h, in_w;       /* the network input (PROTO and INPUT modes) */
    const float*   scale;            /* NATIVE: fp32 [B][5] = (pad_w, pad_h, gain, orig_w, orig_h) */
    uint8_t*       masks;
    int32_t        out_h, out_w;
} yre_mask_desc;
int yre_seg_masks(const yre_mask_desc* d, yre_stream_t s);

/* ---- flat launch plan -------------------------------------------------------------------------
 * Replaces the named-DAG interpreter loop of YOLO.forward  src/yolo/model/model.py:87-107
 * The host walks the module tree once, records every op (descriptors are copied, TMA tensor
 * maps encoded once) and afterwards replays the whole forward with one call; the replay is
 * CUDA-graph capturable (no allocation, no sync). */
typedef struct yre_plan yre_plan;
int  yre_plan_create(yre_plan** out);
void yre_plan_destroy(yre_plan* p);
int  yre_plan_add_conv(yre_plan* p, const yre_conv_desc* d);
int  yre_plan_add_stem(yre_plan* p, const yre_stem_desc* d);
int  yre_plan_add_adown_prepool(yre_plan* p, const yre_view* x, const yre_view* avg_lo, const yre_view* max_hi);
int  yre_plan_add_spp_maxpool(yre_plan* p, const yre_view* x, const yre_view* y5, const yre_view* y9, const yre_view* y13);
int  yre_plan_add_upsample2x(yre_plan* p, const yre_view* x, const yre_view* y);
int  yre_plan_add_cbfuse_sum(yre_plan* p, const yre_view* srcs, int32_t n_src, const yre_view* target, const yre_view* y);
int  yre_plan_add_nchw_to_view(yre_plan* p, const float* x_nchw, const yre_view* y);
int  yre_plan_add_view_to_nchw(yre_plan* p, const yre_view* x, float* y_nchw);
int  yre_plan_add_decode(yre_plan* p, const yre_decode_desc* d);
int  yre_plan_add_decode_masks(yre_plan* p, const yre_decode_masks_desc* d);
int  yre_plan_add_nms(yre_plan* p, const yre_nms_desc* d);
/* Re-points every recorded pointer field equal to old_ptr (image input, raw-logit / decoded /
 * NCHW outputs, residuals) to new_ptr, so one plan serves fresh input and output tensors on
 * every forward.  Conv inputs and weights are baked into TMA tensor maps: asking to rebind one
 * of those fails with YRE_EUNSUPPORTED.  Returns the number of patched fields (>= 0). */
int  yre_plan_rebind(yre_plan* p, const void* old_ptr, void* new_ptr);
int  yre_plan_run(yre_plan* p, yre_stream_t s);
/* Batch capacity: a plan whose ops were all recorded for the same B images (every plan the Python engine compiles) runs
 * any n <= B of them.  yre_plan_batch_capacity returns that B, or YRE_EINVAL (with a message) for an empty plan or one
 * whose ops disagree on B.
 * yre_plan_run_batch(p, n, s) computes the first n images exactly as yre_plan_run computes them (bit-identical: every
 * kernel keeps the tiling chosen for B images, each output element reads only its own image) and writes no row of an
 * image >= n in any buffer -- so the caller's input and output tensors need only hold n images.  The launches are
 * shorter: grids cover the first n images, the tcgen05 convs walk the first ceil(n / tb) image tiles of their tile
 * schedule (yre_conv_tc_schedule) and store through output tensor maps that end at image n (encoded on the host at the
 * first run of each n, and again when n or a re-bound output pointer changes; the encoding is host work only, so a
 * run_batch is CUDA-graph capturable like yre_plan_run).  n == B launches exactly what yre_plan_run launches.
 * YRE_EINVAL for n < 1, n > B or a plan without a capacity. */
int  yre_plan_run_batch(yre_plan* p, int32_t n, yre_stream_t s);
int  yre_plan_batch_capacity(const yre_plan* p);
/* kernels launched by one yre_plan_run / ops recorded / of which tcgen05 convs */
int  yre_plan_num_launches(const yre_plan* p);
int  yre_plan_num_ops(const yre_plan* p);
int  yre_plan_num_tcgen05(const yre_plan* p);
/* fills flops[i] with the algorithmic FLOPs of op i (0 for non-conv ops); returns n ops */
int  yre_plan_op_flops(const yre_plan* p, double* flops, int32_t cap);
/* launches only op i (per-op timing / profiling) */
int  yre_plan_run_op(yre_plan* p, int32_t i, yre_stream_t s);
/* short static name of op i's kernel family ("conv_tc", "conv_ffma", "stem", ...) */
const char* yre_plan_op_name(const yre_plan* p, int32_t i);
/* which kernel variant runs op i and with which tiling, e.g. "generic-cta2 M=1x8x16 N=256 K=16x64 stages=4 s64 tma thr=384
 * grid=148" (halo-ws = weight-stationary halo kernel, halo-stream[-ybx] = streamed-weight halo kernel, generic[-cta2] =
 * tap-by-tap implicit GEMM [on CTA pairs]); non-conv ops report their family name.  Makes the per-layer kernel selection
 * visible (there is no silent fallback: a conv that tcgen05 declines shows up as "conv_ffma"). */
int  yre_plan_op_variant(const yre_plan* p, int32_t i, char* out, int32_t cap);

#ifdef __cplusplus
}
#endif
#endif /* YRE_H */
