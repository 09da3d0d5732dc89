// K12 / K13: test-time augmentation -- the two steps around the branch forwards of upstream's _forward_augment.
//   scale_img (flip + F.interpolate(bilinear, align_corners=False) + F.pad(0.447))   YOLOv5 utils/torch_utils.py
//   _descale_pred + _clip_augmented + torch.cat                                       YOLOv5 models/yolo.py
// Both are HBM-bound copies: K12 writes 12 bytes per branch pixel from <= 4 source pixels per channel, one thread per
// output pixel in 32 x 8 tiles (full 128-byte rows of each channel plane); K13 streams the kept anchor windows of the
// three branches' decoded rows into one buffer, 16 bytes per thread when the row width allows it.
// The arithmetic is fp32 with every rounding explicit (no FMA contraction): the bit-exact contract in include/yre.h.
#include "yre_common.cuh"
#include <math.h>

namespace {

constexpr double kTtaScale[YRE_TTA_BRANCHES] = {1.0, 0.83, 0.67};
constexpr int kTtaFlip[YRE_TTA_BRANCHES] = {0, 1, 0};
constexpr int kTtaGs = 32;                    // max stride: branch inputs are padded to multiples of it
constexpr int kTtaGrid = 1 + 4 + 16;          // anchors per P5 cell over the three levels (_clip_augmented's g)

struct TtaScaleParams {
    const float* xf;
    const uint8_t* xu;
    int H, W, flip, rh, rw, oh, ow;
    float sh, sw;                             // (float)in / out per axis
    float* y;
};

template <int U8>
__device__ __forceinline__ float tta_ld(const TtaScaleParams& p, int b, int c, int y, int x) {
    if (U8) return __fdiv_rn((float)p.xu[(((long long)b * p.H + y) * p.W + x) * 3 + (2 - c)], 255.f);   // BGR -> RGB, /255
    return p.xf[(((long long)b * 3 + c) * p.H + y) * p.W + x];
}

template <int U8>
__global__ void __launch_bounds__(256) tta_scale_kernel(const __grid_constant__ TtaScaleParams p) {
    const int X = blockIdx.x * 32 + (threadIdx.x & 31), Y = blockIdx.y * 8 + (threadIdx.x >> 5), b = blockIdx.z;
    if (X >= p.ow || Y >= p.oh) return;
    const long long plane = (long long)p.oh * p.ow;
    float* o = p.y + (long long)b * 3 * plane + (long long)Y * p.ow + X;
    if (X >= p.rw || Y >= p.rh) {
        o[0] = o[plane] = o[2 * plane] = 0.447f;
        return;
    }
    int y0, y1, x0, x1;
    float h0, h1, w0, w1;
    bilinear_coeff(Y, p.sh, p.H, y0, y1, h0, h1);
    bilinear_coeff(X, p.sw, p.W, x0, x1, w0, w1);
    if (p.flip) { x0 = p.W - 1 - x0; x1 = p.W - 1 - x1; }      // column i of the mirrored image is column W-1-i
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const float v00 = tta_ld<U8>(p, b, c, y0, x0), v01 = tta_ld<U8>(p, b, c, y0, x1);
        const float v10 = tta_ld<U8>(p, b, c, y1, x0), v11 = tta_ld<U8>(p, b, c, y1, x1);
        const float top = __fadd_rn(__fmul_rn(w0, v00), __fmul_rn(w1, v01));
        const float bot = __fadd_rn(__fmul_rn(w0, v10), __fmul_rn(w1, v11));
        o[c * plane] = __fadd_rn(__fmul_rn(h0, top), __fmul_rn(h1, bot));
    }
}

struct TtaMergeParams {
    const float* y[YRE_TTA_BRANCHES];
    int A[YRE_TTA_BRANCHES], a0[YRE_TTA_BRANCHES], len[YRE_TTA_BRANCHES], off[YRE_TTA_BRANCHES];   // len: kept anchors
    float s[YRE_TTA_BRANCHES], fw[YRE_TTA_BRANCHES];
    int flip[YRE_TTA_BRANCHES];
    int no, A_tot;
    float* out;
};

__device__ __forceinline__ float tta_box(float v, int col, const TtaMergeParams& p, int br) {
    v = __fdiv_rn(v, p.s[br]);
    return (col == 0 && p.flip[br]) ? __fsub_rn(p.fw[br], v) : v;
}

// grid: (x tiles, branch, image).  VEC: rows are a multiple of 4 floats, so every float4 lies inside one row and the box
// columns 0..3 are exactly the first float4 of a row
template <int VEC>
__global__ void __launch_bounds__(256) tta_merge_kernel(const __grid_constant__ TtaMergeParams p) {
    const int br = blockIdx.y, b = blockIdx.z;
    const int n = p.len[br] * p.no;                                      // floats of this image's window
    const float* src = p.y[br] + ((long long)b * p.A[br] + p.a0[br]) * p.no;
    float* dst = p.out + ((long long)b * p.A_tot + p.off[br]) * p.no;
    const int step = gridDim.x * blockDim.x;
    if (VEC) {
        const float4* s4 = reinterpret_cast<const float4*>(src);
        float4* d4 = reinterpret_cast<float4*>(dst);
        for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < n / 4; v += step) {
            float4 q = __ldcs(s4 + v);                                   // read once: stream past L2
            if ((4 * v) % p.no == 0) {
                q.x = tta_box(q.x, 0, p, br); q.y = tta_box(q.y, 1, p, br);
                q.z = tta_box(q.z, 2, p, br); q.w = tta_box(q.w, 3, p, br);
            }
            d4[v] = q;
        }
    } else {
        for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += step) {
            const int col = e % p.no;
            const float q = __ldcs(src + e);
            dst[e] = col < 4 ? tta_box(q, col, p, br) : q;
        }
    }
}

bool aligned(const void* ptr, size_t a) { return ((uintptr_t)ptr & (a - 1)) == 0; }

}  // namespace

extern "C" int yre_tta_geometry(int32_t h, int32_t w, yre_tta_geom* g) {
    if (!g) YRE_FAIL(YRE_EINVAL, "tta_geometry: null output");
    if (h <= 0 || w <= 0 || h % kTtaGs || w % kTtaGs || h > 65536 || w > 65536)
        YRE_FAIL(YRE_EINVAL, "tta_geometry: %dx%d is not a positive multiple of %d (at most 65536) on both axes", h, w, kTtaGs);
    g->h = h; g->w = w;
    g->A_tot = 0;
    for (int i = 0; i < YRE_TTA_BRANCHES; ++i) {
        const double s = kTtaScale[i];
        g->scale[i] = (float)s;
        g->flip[i] = kTtaFlip[i];
        if (s == 1.0) {
            g->rh[i] = g->out_h[i] = h;
            g->rw[i] = g->out_w[i] = w;
        } else {   // Python: int(h * s); math.ceil(h * s / gs) * gs -- double arithmetic, one rounding per operation
            const double hs = (double)h * s, ws = (double)w * s;
            g->rh[i] = (int)hs; g->rw[i] = (int)ws;
            g->out_h[i] = (int)ceil(hs / kTtaGs) * kTtaGs;
            g->out_w[i] = (int)ceil(ws / kTtaGs) * kTtaGs;
        }
        const int ch = g->out_h[i] / kTtaGs, cw = g->out_w[i] / kTtaGs;     // P5 cells
        g->A[i] = kTtaGrid * ch * cw;
        g->a_begin[i] = 0;
        g->a_end[i] = g->A[i];
    }
    const int last = YRE_TTA_BRANCHES - 1;
    g->a_end[0] = g->A[0] - g->A[0] / kTtaGrid;                 // branch 0 without its P5 (large objects)
    g->a_begin[last] = 16 * (g->A[last] / kTtaGrid);            // the last branch without its P3 (small objects)
    for (int i = 0; i < YRE_TTA_BRANCHES; ++i) g->A_tot += g->a_end[i] - g->a_begin[i];
    return YRE_OK;
}

extern "C" int yre_tta_scale_img(const yre_tta_scale_desc* d, yre_stream_t s) {
    if (!d || !d->y || (!d->x_nchw) == (!d->x_u8_hwc)) YRE_FAIL(YRE_EINVAL, "tta_scale_img: need y and exactly one input");
    if (d->B < 1 || d->n < 1 || d->n > d->B || d->n > 65535)
        YRE_FAIL(YRE_EINVAL, "tta_scale_img: %d images of a batch of %d", d->n, d->B);
    if (d->H < 1 || d->W < 1 || d->rh < 1 || d->rw < 1 || d->rh > d->out_h || d->rw > d->out_w || d->out_h > 65536 ||
        d->out_w > 65536 || d->H > 65536 || d->W > 65536)
        YRE_FAIL(YRE_EINVAL, "tta_scale_img: bad extents (input %dx%d, resized %dx%d, padded %dx%d)", d->H, d->W, d->rh, d->rw,
                 d->out_h, d->out_w);
    if (d->flip != 0 && d->flip != 1) YRE_FAIL(YRE_EINVAL, "tta_scale_img: flip must be 0 or 1");
    if (!aligned(d->y, 4) || (d->x_nchw && !aligned(d->x_nchw, 4))) YRE_FAIL(YRE_EINVAL, "tta_scale_img: fp32 buffers must be 4-byte aligned");
    TtaScaleParams p;
    p.xf = d->x_nchw; p.xu = d->x_u8_hwc; p.H = d->H; p.W = d->W; p.flip = d->flip;
    p.rh = d->rh; p.rw = d->rw; p.oh = d->out_h; p.ow = d->out_w;
    p.sh = (float)d->H / (float)d->rh; p.sw = (float)d->W / (float)d->rw;      // torch: (float)input_size / output_size
    p.y = d->y;
    const dim3 grid(yre_cdiv(p.ow, 32), yre_cdiv(p.oh, 8), (unsigned)d->n);
    if (p.xu) tta_scale_kernel<1><<<grid, 256, 0, (cudaStream_t)s>>>(p);
    else tta_scale_kernel<0><<<grid, 256, 0, (cudaStream_t)s>>>(p);
    YRE_LAUNCH_CHECK("tta_scale");
    return YRE_OK;
}

extern "C" int yre_tta_merge(const yre_tta_merge_desc* d, yre_stream_t s) {
    if (!d || !d->out) YRE_FAIL(YRE_EINVAL, "tta_merge: null descriptor or output");
    if (d->nc < 1 || d->nc > 4096) YRE_FAIL(YRE_EINVAL, "tta_merge: nc %d (1..4096)", d->nc);
    if (d->B < 1 || d->n < 1 || d->n > d->B || d->n > 65535) YRE_FAIL(YRE_EINVAL, "tta_merge: %d images of a batch of %d", d->n, d->B);
    if (!aligned(d->out, 16)) YRE_FAIL(YRE_EINVAL, "tta_merge: out must be 16-byte aligned");
    TtaMergeParams p;
    p.no = 4 + d->nc;
    long long tot = 0, longest = 0;
    for (int i = 0; i < YRE_TTA_BRANCHES; ++i) {
        const yre_tta_merge_branch& b = d->br[i];
        if (!b.y || !aligned(b.y, 16)) YRE_FAIL(YRE_EINVAL, "tta_merge: branch %d: y must be a 16-byte aligned pointer", i);
        if (b.A < 1 || b.a_begin < 0 || b.a_end <= b.a_begin || b.a_end > b.A)
            YRE_FAIL(YRE_EINVAL, "tta_merge: branch %d: window [%d, %d) of %d anchors", i, b.a_begin, b.a_end, b.A);
        if (!(b.scale > 0.f) || !isfinite(b.scale) || b.flip_w < 0)
            YRE_FAIL(YRE_EINVAL, "tta_merge: branch %d: scale %g, flip width %d", i, b.scale, b.flip_w);
        if ((long long)b.A * p.no > (1ll << 31) - 1) YRE_FAIL(YRE_EINVAL, "tta_merge: branch %d: %d anchors is too many", i, b.A);
        p.y[i] = b.y; p.A[i] = b.A; p.a0[i] = b.a_begin; p.len[i] = b.a_end - b.a_begin; p.off[i] = (int)tot;
        p.s[i] = b.scale; p.fw[i] = (float)b.flip_w; p.flip[i] = b.flip_w != 0;
        tot += p.len[i];
        longest = p.len[i] > longest ? p.len[i] : longest;
    }
    if (tot * p.no > (1ll << 31) - 1)
        YRE_FAIL(YRE_EINVAL, "tta_merge: %lld anchors x %d columns per image is too large", tot, p.no);
    p.A_tot = (int)tot;
    p.out = d->out;
    const int vec = p.no % 4 == 0;
    const long long units = vec ? longest * p.no / 4 : longest * p.no;
    const dim3 grid(yre_cdiv(units, 256 * 4), YRE_TTA_BRANCHES, (unsigned)d->n);    // ~4 units per thread
    if (vec) tta_merge_kernel<1><<<grid, 256, 0, (cudaStream_t)s>>>(p);
    else tta_merge_kernel<0><<<grid, 256, 0, (cudaStream_t)s>>>(p);
    YRE_LAUNCH_CHECK("tta_merge");
    return YRE_OK;
}
