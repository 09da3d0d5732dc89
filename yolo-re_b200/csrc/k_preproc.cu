// K8 / K14 / K9: letterbox pre-processing and box rescaling -- the steps either side of the detection path.
//   letterbox + cv2.resize(INTER_LINEAR, uint8) + BGR->RGB + HWC->CHW + /255     reference scripts/detect.py:40-71, 223-227
//   K14: the same on 4:2:0 YUV frames, each source tap converted as cv2.cvtColor(COLOR_YUV2BGR_*) converts it
//   scale_boxes                                                                  reference scripts/detect.py:74-109
// Byte / integer work, HBM-bound on the fp32 output (4 x 3 bytes written per destination pixel against <= 3 h w read):
// one thread per output pixel, 32 x 8 thread tiles so that the three channel planes are written in full 128-byte
// rows and the source bytes of a tile sit in a handful of adjacent lines.
// The resize restates OpenCV's 8-bit fixed-point bilinear kernel bit for bit (oracle/preproc_ref.py has the
// derivation and is pinned against cv2 and against the reference's own letterbox output).
#include "yre_common.cuh"
#include <math.h>

namespace {

struct LbParams {
    const uint8_t* src;
    int h, w;
    long long pitch;
    int oh, ow;              // destination extent
    int nw, nh, top, left;
    int c0, c1, c2;          // pad colour, source channel order
    int mode;                // 0 bilinear, 1 copy, 2 exact 2x area
    double sx, sy;           // src / dst scale
    void* dst;
};

// coefficient of one axis: (i0, i1, a0, a1) for destination index d.  clamp_w: OpenCV clamps the weight together
// with the index horizontally, but only the indices vertically.
__device__ __forceinline__ void lb_coeff(int d, double scale, int sn, bool clamp_w, int& i0, int& i1, int& a0, int& a1) {
    // (d + 0.5) * scale - 0.5 in double with separate roundings (no FMA contraction), then to float
    float f = (float)__dadd_rn(__dmul_rn((double)d + 0.5, scale), -0.5);
    int s = (int)floorf(f);
    f = __fsub_rn(f, (float)s);
    if (clamp_w) {
        if (s < 0) { s = 0; f = 0.f; }
        if (s >= sn - 1) { s = sn - 1; f = 0.f; }
    }
    i0 = min(max(s, 0), sn - 1);
    i1 = min(max(s + 1, 0), sn - 1);
    a0 = __float2int_rn(__fmul_rn(__fsub_rn(1.f, f), 2048.f));     // saturate_cast<short>: round half to even
    a1 = __float2int_rn(__fmul_rn(f, 2048.f));
}

// Source pixel access: at(p, x, y) is source pixel (x, y), right / below its neighbours, and ch(p, q, c) channel c
// (B, G, R) of pixel q.  The letterbox kernel is written once against this interface: the resize, padding and output
// code is the same for every source layout.
struct BgrSrc {                                        // K8: uint8 [h][w][3], rows `pitch` bytes apart
    using Params = LbParams;
    using Px = const uint8_t*;
    static __device__ __forceinline__ Px at(const Params& p, int x, int y) { return p.src + (long long)y * p.pitch + 3 * x; }
    static __device__ __forceinline__ Px right(const Params&, Px q) { return q + 3; }
    static __device__ __forceinline__ Px below(const Params& p, Px q) { return q + p.pitch; }
    static __device__ __forceinline__ int ch(const Params&, Px q, int c) { return q[c]; }
};

// K14: 4:2:0 YUV, limited range, 20-bit fixed point with nearest chroma (one (U, V) sample per 2 x 2 luma block): the
// arithmetic of cv2.cvtColor(COLOR_YUV2BGR_{NV12,NV21,I420,YV12}).  src / pitch are the luma plane; every format is
// the pair of U and V pointers and the byte step between horizontally adjacent chroma samples (2 interleaved, 1 planar).
struct YuvParams : LbParams {
    const uint8_t* u;
    const uint8_t* v;
    long long cpitch;
    int cstep;
    int matrix;                                      // row of yuv_coeff
};

// 3-decimal limited-range coefficients times 2^20, rounded: BT.601 are cv2's (1.164, 1.596, 0.813, 0.391, 2.018),
// BT.709 the same scheme on (1.164, 1.793, 0.533, 0.213, 2.112)
__constant__ int yuv_coeff[2][5] = {{1220542, 1673527, -852492, -409993, 2116026},      // cy, cvr, cvg, cug, cub
                                    {1220542, 1880097, -558891, -223347, 2214593}};

struct Yuv420Src {
    using Params = YuvParams;
    struct Px { int x, y; };
    static __device__ __forceinline__ Px at(const Params&, int x, int y) { return {x, y}; }
    static __device__ __forceinline__ Px right(const Params&, Px q) { return {q.x + 1, q.y}; }
    static __device__ __forceinline__ Px below(const Params&, Px q) { return {q.x, q.y + 1}; }
    // the three channels of a pixel share their loads and products once inlined
    static __device__ __forceinline__ int ch(const Params& p, Px q, int c) {
        const int lum = p.src[(long long)q.y * p.pitch + q.x];
        const long long o = (long long)(q.y >> 1) * p.cpitch + (long long)(q.x >> 1) * p.cstep;
        const int uu = p.u[o] - 128, vv = p.v[o] - 128;
        const int* k = yuv_coeff[p.matrix];
        const int yy = max(lum - 16, 0) * k[0] + (1 << 19);
        const int t = c == 0 ? yy + k[4] * uu : (c == 1 ? yy + k[2] * vv + k[3] * uu : yy + k[1] * vv);
        return min(max(t >> 20, 0), 255);
    }
};

constexpr int LB_BATCH = 32;                  // images per launch (descriptors travel as kernel parameters, < 4 KB)
template <class P> struct LbBatch { P p[LB_BATCH]; };
static_assert(sizeof(LbBatch<YuvParams>) < 4096, "letterbox descriptors must fit the kernel parameter space");

template <int OUT_U8, class Src>
__global__ void __launch_bounds__(256) letterbox_kernel(const __grid_constant__ LbBatch<typename Src::Params> batch) {
    const typename Src::Params& p = batch.p[blockIdx.z];
    const int X = blockIdx.x * 32 + (threadIdx.x & 31), Y = blockIdx.y * 8 + (threadIdx.x >> 5);
    if (X >= p.ow || Y >= p.oh) return;
    int v0 = p.c0, v1 = p.c1, v2 = p.c2;
    const int dx = X - p.left, dy = Y - p.top;
    if (dx >= 0 && dx < p.nw && dy >= 0 && dy < p.nh) {
        if (p.mode == 1) {
            const typename Src::Px q = Src::at(p, dx, dy);
            v0 = Src::ch(p, q, 0); v1 = Src::ch(p, q, 1); v2 = Src::ch(p, q, 2);
        } else if (p.mode == 2) {
            const typename Src::Px q0 = Src::at(p, 2 * dx, 2 * dy), q1 = Src::below(p, q0);
            const typename Src::Px q0r = Src::right(p, q0), q1r = Src::right(p, q1);
            v0 = (Src::ch(p, q0, 0) + Src::ch(p, q0r, 0) + Src::ch(p, q1, 0) + Src::ch(p, q1r, 0) + 2) >> 2;
            v1 = (Src::ch(p, q0, 1) + Src::ch(p, q0r, 1) + Src::ch(p, q1, 1) + Src::ch(p, q1r, 1) + 2) >> 2;
            v2 = (Src::ch(p, q0, 2) + Src::ch(p, q0r, 2) + Src::ch(p, q1, 2) + Src::ch(p, q1r, 2) + 2) >> 2;
        } else {
            int x0, x1, a0, a1, y0, y1, b0, b1;
            lb_coeff(dx, p.sx, p.w, true, x0, x1, a0, a1);
            lb_coeff(dy, p.sy, p.h, false, y0, y1, b0, b1);
            const typename Src::Px q00 = Src::at(p, x0, y0), q01 = Src::at(p, x1, y0);
            const typename Src::Px q10 = Src::at(p, x0, y1), q11 = Src::at(p, x1, y1);
            int out[3];
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const int h0 = Src::ch(p, q00, c) * a0 + Src::ch(p, q01, c) * a1;       // horizontal pass, 11 fractional bits
                const int h1 = Src::ch(p, q10, c) * a0 + Src::ch(p, q11, c) * a1;
                const int o = (((b0 * (h0 >> 4)) >> 16) + ((b1 * (h1 >> 4)) >> 16) + 2) >> 2;
                out[c] = min(max(o, 0), 255);
            }
            v0 = out[0]; v1 = out[1]; v2 = out[2];
        }
    }
    if (OUT_U8) {
        uint8_t* o = reinterpret_cast<uint8_t*>(p.dst) + ((long long)Y * p.ow + X) * 3;
        o[0] = (uint8_t)v0; o[1] = (uint8_t)v1; o[2] = (uint8_t)v2;
    } else {
        float* o = reinterpret_cast<float*>(p.dst) + (long long)Y * p.ow + X;
        const long long plane = (long long)p.oh * p.ow;
        o[0] = __fdiv_rn((float)v2, 255.f);              // BGR -> RGB: plane 0 is the source's channel 2
        o[plane] = __fdiv_rn((float)v1, 255.f);
        o[2 * plane] = __fdiv_rn((float)v0, 255.f);
    }
}

__global__ void scale_boxes_kernel(float* boxes, int n, int stride, float pad_w, float pad_h, float gain, float ow, float oh) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n * 4) return;
    const int r = i >> 2, c = i & 3;
    float* q = boxes + (long long)r * stride + c;
    const bool is_x = (c & 1) == 0;
    float v = __fsub_rn(*q, is_x ? pad_w : pad_h);
    v = __fdiv_rn(v, gain);
    *q = fminf(fmaxf(v, 0.f), is_x ? ow : oh);
}

}  // namespace

extern "C" int yre_letterbox_geometry_rect(yre_letterbox_desc* d, int32_t new_h, int32_t new_w, int32_t stride,
                                           double* ratio, int32_t* pad_w, int32_t* pad_h) {
    if (!d || d->h <= 0 || d->w <= 0 || new_h <= 0 || new_w <= 0 || stride < 0) YRE_FAIL(YRE_EINVAL, "letterbox: bad size");
    const double r = fmin((double)new_h / d->h, (double)new_w / d->w);
    // Python round() and C nearbyint() under the default rounding mode both round half to even
    const int nw = (int)nearbyint(d->w * r), nh = (int)nearbyint(d->h * r);
    if (nw <= 0 || nh <= 0) YRE_FAIL(YRE_EINVAL, "letterbox: %dx%d resizes to nothing at %dx%d", d->w, d->h, new_w, new_h);
    int pw = new_w - nw, ph = new_h - nh;                  // >= 0: r fits both axes
    if (stride > 0) { pw %= stride; ph %= stride; }        // auto: the smallest stride-multiple rectangle
    const double dw = pw / 2.0, dh = ph / 2.0;
    const int top = (int)nearbyint(dh - 0.1), bottom = (int)nearbyint(dh + 0.1);
    const int left = (int)nearbyint(dw - 0.1), right = (int)nearbyint(dw + 0.1);
    d->new_w = nw; d->new_h = nh; d->top = top; d->left = left;
    d->out_h = nh + top + bottom; d->out_w = nw + left + right;
    if (ratio) *ratio = r;
    if (pad_w) *pad_w = (int32_t)dw;          // int(dw): truncation, scripts/detect.py:71
    if (pad_h) *pad_h = (int32_t)dh;
    return YRE_OK;
}

extern "C" int yre_letterbox_geometry(yre_letterbox_desc* d, double* ratio, int32_t* pad_w, int32_t* pad_h) {
    if (!d) YRE_FAIL(YRE_EINVAL, "letterbox: bad size");
    return yre_letterbox_geometry_rect(d, d->new_shape, d->new_shape, 0, ratio, pad_w, pad_h);
}

static void lb_extent(const yre_letterbox_desc* d, int& oh, int& ow) {
    oh = d->out_h; ow = d->out_w;
    if (oh == 0 && ow == 0) oh = ow = d->new_shape;
}

// destination, geometry, pad colour and resize mode: everything but the source planes
static int lb_fill_common(const yre_letterbox_desc* d, LbParams& p) {
    if (!d || !d->dst) YRE_FAIL(YRE_EINVAL, "letterbox: null pointer");
    if (d->h <= 0 || d->w <= 0) YRE_FAIL(YRE_EINVAL, "letterbox: bad source extent");
    lb_extent(d, p.oh, p.ow);
    if (p.oh <= 0 || p.ow <= 0 || d->new_w <= 0 || d->new_h <= 0 || d->top < 0 || d->left < 0 || d->left + d->new_w > p.ow ||
        d->top + d->new_h > p.oh)
        YRE_FAIL(YRE_EINVAL, "letterbox: geometry does not fit %dx%d", p.oh, p.ow);
    if (d->out_mode != YRE_LB_F32_CHW && d->out_mode != YRE_LB_U8_HWC) YRE_FAIL(YRE_EINVAL, "letterbox: bad out_mode");
    p.h = d->h; p.w = d->w;
    p.nw = d->new_w; p.nh = d->new_h; p.top = d->top; p.left = d->left;
    p.c0 = d->color[0]; p.c1 = d->color[1]; p.c2 = d->color[2];
    p.mode = (d->w == d->new_w && d->h == d->new_h) ? 1 : ((d->w == 2 * d->new_w && d->h == 2 * d->new_h) ? 2 : 0);
    p.sx = (double)d->w / d->new_w; p.sy = (double)d->h / d->new_h;
    p.dst = d->dst;
    return YRE_OK;
}

static int lb_fill(const yre_letterbox_desc* d, LbParams& p) {
    if (!d || !d->src || !d->dst) YRE_FAIL(YRE_EINVAL, "letterbox: null pointer");
    if (d->row_pitch < 3ll * d->w) YRE_FAIL(YRE_EINVAL, "letterbox: bad source extent");
    const int rc = lb_fill_common(d, p);
    if (rc) return rc;
    p.src = d->src; p.pitch = d->row_pitch;
    return YRE_OK;
}

static int lb_fill_yuv(const yre_letterbox_desc* d, const yre_yuv420_planes* q, YuvParams& p) {
    if (!d || !q) YRE_FAIL(YRE_EINVAL, "letterbox_yuv420: null pointer");
    if (d->src || d->row_pitch) YRE_FAIL(YRE_EINVAL, "letterbox_yuv420: src and row_pitch must be 0, the planes describe the source");
    if (d->h <= 0 || d->w <= 0 || (d->h & 1) || (d->w & 1))
        YRE_FAIL(YRE_EINVAL, "letterbox_yuv420: 4:2:0 needs an even, positive luma extent, got %dx%d", d->w, d->h);
    const bool nv = q->format == YRE_YUV_NV12 || q->format == YRE_YUV_NV21;
    if (!nv && q->format != YRE_YUV_I420 && q->format != YRE_YUV_YV12) YRE_FAIL(YRE_EINVAL, "letterbox_yuv420: bad format %d", q->format);
    if (q->matrix != YRE_YUV_BT601 && q->matrix != YRE_YUV_BT709) YRE_FAIL(YRE_EINVAL, "letterbox_yuv420: bad matrix %d", q->matrix);
    if (!q->luma || !q->chroma[0] || (nv ? q->chroma[1] != nullptr : !q->chroma[1]))
        YRE_FAIL(YRE_EINVAL, "letterbox_yuv420: null plane (or a second chroma plane for NV12 / NV21)");
    if (q->luma_pitch < d->w || q->chroma_pitch < (nv ? d->w : d->w / 2))
        YRE_FAIL(YRE_EINVAL, "letterbox_yuv420: a plane's pitch is shorter than its row");
    const int rc = lb_fill_common(d, p);
    if (rc) return rc;
    p.src = q->luma; p.pitch = q->luma_pitch;
    const uint8_t* c0 = q->chroma[0];
    switch (q->format) {
        case YRE_YUV_NV12: p.u = c0; p.v = c0 + 1; break;
        case YRE_YUV_NV21: p.v = c0; p.u = c0 + 1; break;
        case YRE_YUV_I420: p.u = c0; p.v = q->chroma[1]; break;
        default: p.v = c0; p.u = q->chroma[1]; break;         // YV12
    }
    p.cpitch = q->chroma_pitch; p.cstep = nv ? 2 : 1; p.matrix = q->matrix;
    return YRE_OK;
}

// n images with the same destination extent and out_mode, up to LB_BATCH per launch (grid.z = image).  fill(i, params)
// checks and describes image i; every image is checked before the first launch.
template <class Src, class Fill>
static int lb_launch(const yre_letterbox_desc* d, int32_t n, yre_stream_t s, Fill fill) {
    if (n < 0 || (n > 0 && !d)) YRE_FAIL(YRE_EINVAL, "letterbox: bad batch");
    int oh = 0, ow = 0;
    if (n > 0) lb_extent(d, oh, ow);
    for (int i = 0; i < n; ++i) {
        typename Src::Params q;
        const int rc = fill(i, q);
        if (rc) return rc;
        if (q.oh != oh || q.ow != ow || d[i].out_mode != d[0].out_mode)
            YRE_FAIL(YRE_EINVAL, "letterbox: a batch must share the destination extent and out_mode");
    }
    for (int i0 = 0; i0 < n; i0 += LB_BATCH) {
        const int m = n - i0 < LB_BATCH ? n - i0 : LB_BATCH;
        LbBatch<typename Src::Params> b;
        for (int i = 0; i < m; ++i) fill(i0 + i, b.p[i]);
        for (int i = m; i < LB_BATCH; ++i) b.p[i] = b.p[0];
        dim3 grid(yre_cdiv(ow, 32), yre_cdiv(oh, 8), (unsigned)m);
        if (d[0].out_mode == YRE_LB_U8_HWC) letterbox_kernel<1, Src><<<grid, 256, 0, (cudaStream_t)s>>>(b);
        else letterbox_kernel<0, Src><<<grid, 256, 0, (cudaStream_t)s>>>(b);
        YRE_LAUNCH_CHECK("letterbox");
    }
    return YRE_OK;
}

extern "C" int yre_letterbox_u8_batch(const yre_letterbox_desc* d, int32_t n, yre_stream_t s) {
    return lb_launch<BgrSrc>(d, n, s, [d](int i, LbParams& p) { return lb_fill(&d[i], p); });
}

extern "C" int yre_letterbox_yuv420_batch(const yre_letterbox_desc* d, const yre_yuv420_planes* planes, int32_t n, yre_stream_t s) {
    if (n > 0 && !planes) YRE_FAIL(YRE_EINVAL, "letterbox_yuv420: null planes");
    return lb_launch<Yuv420Src>(d, n, s, [d, planes](int i, YuvParams& p) { return lb_fill_yuv(&d[i], &planes[i], p); });
}

extern "C" int yre_letterbox_u8(const yre_letterbox_desc* d, yre_stream_t s) { return yre_letterbox_u8_batch(d, 1, s); }

extern "C" int yre_scale_boxes(float* boxes, int32_t n, int32_t row_stride, float pad_w, float pad_h, float gain,
                               float orig_w, float orig_h, yre_stream_t s) {
    if (n < 0 || row_stride < 4 || (n > 0 && !boxes)) YRE_FAIL(YRE_EINVAL, "scale_boxes: bad arguments");
    if (!(gain > 0.f)) YRE_FAIL(YRE_EINVAL, "scale_boxes: gain must be positive");
    if (n == 0) return YRE_OK;
    scale_boxes_kernel<<<yre_cdiv(4ll * n, 128), 128, 0, (cudaStream_t)s>>>(boxes, n, row_stride, pad_w, pad_h, gain, orig_w, orig_h);
    YRE_LAUNCH_CHECK("scale_boxes");
    return YRE_OK;
}
