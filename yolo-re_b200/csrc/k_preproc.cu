// K8 / K9: letterbox pre-processing and box rescaling -- the steps either side of the detection path.
//   letterbox + cv2.resize(INTER_LINEAR, uint8) + BGR->RGB + HWC->CHW + /255     reference scripts/detect.py:40-71, 223-227
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

constexpr int LB_BATCH = 32;                  // images per launch (descriptors travel as kernel parameters, < 4 KB)
struct LbBatch { LbParams p[LB_BATCH]; };

template <int OUT_U8>
__global__ void __launch_bounds__(256) letterbox_kernel(const __grid_constant__ LbBatch batch) {
    const LbParams& p = batch.p[blockIdx.z];
    const int X = blockIdx.x * 32 + (threadIdx.x & 31), Y = blockIdx.y * 8 + (threadIdx.x >> 5);
    if (X >= p.ow || Y >= p.oh) return;
    int v0 = p.c0, v1 = p.c1, v2 = p.c2;
    const int dx = X - p.left, dy = Y - p.top;
    if (dx >= 0 && dx < p.nw && dy >= 0 && dy < p.nh) {
        if (p.mode == 1) {
            const uint8_t* q = p.src + (long long)dy * p.pitch + 3 * dx;
            v0 = q[0]; v1 = q[1]; v2 = q[2];
        } else if (p.mode == 2) {
            const uint8_t* q0 = p.src + (long long)(2 * dy) * p.pitch + 6 * dx;
            const uint8_t* q1 = q0 + p.pitch;
            v0 = (q0[0] + q0[3] + q1[0] + q1[3] + 2) >> 2;
            v1 = (q0[1] + q0[4] + q1[1] + q1[4] + 2) >> 2;
            v2 = (q0[2] + q0[5] + q1[2] + q1[5] + 2) >> 2;
        } else {
            int x0, x1, a0, a1, y0, y1, b0, b1;
            lb_coeff(dx, p.sx, p.w, true, x0, x1, a0, a1);
            lb_coeff(dy, p.sy, p.h, false, y0, y1, b0, b1);
            const uint8_t* r0 = p.src + (long long)y0 * p.pitch;
            const uint8_t* r1 = p.src + (long long)y1 * p.pitch;
            int out[3];
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const int h0 = r0[3 * x0 + c] * a0 + r0[3 * x1 + c] * a1;       // horizontal pass, 11 fractional bits
                const int h1 = r1[3 * x0 + c] * a0 + r1[3 * x1 + c] * a1;
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

static int lb_fill(const yre_letterbox_desc* d, LbParams& p) {
    if (!d || !d->src || !d->dst) YRE_FAIL(YRE_EINVAL, "letterbox: null pointer");
    if (d->h <= 0 || d->w <= 0 || d->row_pitch < 3ll * d->w) YRE_FAIL(YRE_EINVAL, "letterbox: bad source extent");
    lb_extent(d, p.oh, p.ow);
    if (p.oh <= 0 || p.ow <= 0 || d->new_w <= 0 || d->new_h <= 0 || d->top < 0 || d->left < 0 || d->left + d->new_w > p.ow ||
        d->top + d->new_h > p.oh)
        YRE_FAIL(YRE_EINVAL, "letterbox: geometry does not fit %dx%d", p.oh, p.ow);
    if (d->out_mode != YRE_LB_F32_CHW && d->out_mode != YRE_LB_U8_HWC) YRE_FAIL(YRE_EINVAL, "letterbox: bad out_mode");
    p.src = d->src; p.h = d->h; p.w = d->w; p.pitch = d->row_pitch;
    p.nw = d->new_w; p.nh = d->new_h; p.top = d->top; p.left = d->left;
    p.c0 = d->color[0]; p.c1 = d->color[1]; p.c2 = d->color[2];
    p.mode = (d->w == d->new_w && d->h == d->new_h) ? 1 : ((d->w == 2 * d->new_w && d->h == 2 * d->new_h) ? 2 : 0);
    p.sx = (double)d->w / d->new_w; p.sy = (double)d->h / d->new_h;
    p.dst = d->dst;
    return YRE_OK;
}

// n images with the same destination extent and out_mode, up to LB_BATCH per launch (grid.z = image)
extern "C" int yre_letterbox_u8_batch(const yre_letterbox_desc* d, int32_t n, yre_stream_t s) {
    if (n < 0 || (n > 0 && !d)) YRE_FAIL(YRE_EINVAL, "letterbox: bad batch");
    int oh = 0, ow = 0;
    if (n > 0) lb_extent(d, oh, ow);
    for (int i0 = 0; i0 < n; i0 += LB_BATCH) {
        const int m = n - i0 < LB_BATCH ? n - i0 : LB_BATCH;
        LbBatch b;
        for (int i = 0; i < m; ++i) {
            const int rc = lb_fill(&d[i0 + i], b.p[i]);
            if (rc) return rc;
            if (b.p[i].oh != oh || b.p[i].ow != ow || d[i0 + i].out_mode != d[0].out_mode)
                YRE_FAIL(YRE_EINVAL, "letterbox: a batch must share the destination extent and out_mode");
        }
        for (int i = m; i < LB_BATCH; ++i) b.p[i] = b.p[0];
        dim3 grid(yre_cdiv(ow, 32), yre_cdiv(oh, 8), (unsigned)m);
        if (d[0].out_mode == YRE_LB_U8_HWC) letterbox_kernel<1><<<grid, 256, 0, (cudaStream_t)s>>>(b);
        else letterbox_kernel<0><<<grid, 256, 0, (cudaStream_t)s>>>(b);
        YRE_LAUNCH_CHECK("letterbox");
    }
    return YRE_OK;
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
