// K15: instance-segmentation masks of the kept detections, after NMS, for a whole batch in one launch.
//   process_mask / process_mask_native / crop_mask      upstream YOLOv9 utils/segment/general.py
// One CTA per (detection row j, image b); rows j >= counts[b] return at once.  The CTA walks its output planes in 16 x 64
// tiles.  A tile that no kept pixel can reach is written as zeros without a logit.  Otherwise the proto pixels its
// outputs sample (only those inside the crop in the proto / input modes) are staged in shared memory as probabilities
// -- each logit once per tile, a 32-term fp32 dot product over the NHWC proto row -- and every thread then writes 4
// neighbouring output bytes from them.  The bilinear arithmetic is K12's (bilinear_coeff, yre_common.cuh); every
// rounding is explicit, so the numpy restatement in oracle/seg_ref.py follows the same operation order.
#include "yre_common.cuh"
#include <math.h>

namespace {

constexpr int NM = 32;
constexpr int THREADS = 256;
constexpr int TY = 16, TX = 64;                      // output tile; one 4-byte group per thread
constexpr int SY = 2 * TY + 4, SX = 2 * TX + 4;      // staged rows / columns of a tile, at most

struct SegParams {
    const float* proto;
    const float* mc;
    const float* det;
    const int32_t* counts;
    const int64_t* keep;
    const float* scale;
    uint8_t* masks;
    int mh, mw, pitch, A, max_det, mode, oh, ow;
    float rx, ry;                                     // box -> proto pixels (proto / input modes)
    float sh, sw;                                     // bilinear scales (proto / input modes)
};

// integers r in [0, n) with r >= lo and r < hi, as [i0, i1); empty for a NaN bound (every comparison is false)
__device__ __forceinline__ void crop_range(float lo, float hi, int n, int& i0, int& i1) {
    if (lo != lo || hi != hi) { i0 = i1 = 0; return; }
    lo = fminf(fmaxf(lo, 0.f), (float)n);
    hi = fminf(fmaxf(hi, 0.f), (float)n);
    i0 = (int)ceilf(lo);
    i1 = max(i0, (int)ceilf(hi));
}

// Per-axis sampling of a tile's active outputs [a0, a1): output i takes staged entries idx[i][0..1] with weights
// w[i][0..1]; src[k] is the source coordinate of staged entry k.  Contiguous sources (upsampling: each one once) when
// they fit, else two entries per output (downsampling: a source is staged at most twice).  Returns the staged count.
__device__ __forceinline__ int axis_setup(int a0, int a1, float scale, int in, int off, int cap, int* src, int (*idx)[2],
                                          float (*w)[2]) {
    int lo, hi, t0, t1;
    float l0, l1;
    bilinear_coeff(a0, scale, in, lo, t1, l0, l1);
    bilinear_coeff(a1 - 1, scale, in, t0, hi, l0, l1);
    const bool contig = hi - lo + 1 <= cap;
    const int n = a1 - a0, cnt = contig ? hi - lo + 1 : 2 * n;
    for (int i = threadIdx.x; i < n; i += THREADS) {
        int i0, i1;
        float w0, w1;
        bilinear_coeff(a0 + i, scale, in, i0, i1, w0, w1);
        w[i][0] = w0; w[i][1] = w1;
        if (contig) {
            idx[i][0] = i0 - lo; idx[i][1] = i1 - lo;
        } else {
            idx[i][0] = 2 * i; idx[i][1] = 2 * i + 1;
            src[2 * i] = i0 + off; src[2 * i + 1] = i1 + off;
        }
    }
    if (contig)
        for (int k = threadIdx.x; k < cnt; k += THREADS) src[k] = lo + k + off;
    return cnt;
}

// n zero bytes from d, block-wide: 16-byte stores between an unaligned head and tail
__device__ __forceinline__ void zero_fill(uint8_t* d, long long n) {
    if (n <= 0) return;
    const long long head = min(n, (long long)((16 - ((uintptr_t)d & 15)) & 15));
    const long long body = (n - head) / 16;
    for (long long i = threadIdx.x; i < head; i += THREADS) d[i] = 0;
    uint4* d16 = reinterpret_cast<uint4*>(d + head);
    for (long long i = threadIdx.x; i < body; i += THREADS) d16[i] = make_uint4(0, 0, 0, 0);
    for (long long i = head + body * 16 + threadIdx.x; i < n; i += THREADS) d[i] = 0;
}

// zeros in rows [r0, r1), columns [c0, c1) of a plane with rows ow bytes apart, block-wide, in groups of 4 columns from
// c0 & ~3: 4-byte stores for whole groups when ow % 4 == 0 (vec), bytes otherwise
__device__ __forceinline__ void zero_cols(uint8_t* plane, int ow, int r0, int r1, int c0, int c1, bool vec) {
    if (r0 >= r1 || c0 >= c1) return;
    const int g0 = c0 & ~3, groups = (c1 - g0 + 3) / 4;
    for (long long k = threadIdx.x; k < (long long)(r1 - r0) * groups; k += THREADS) {
        const int r = r0 + (int)(k / groups), X = g0 + 4 * (int)(k % groups);
        uint8_t* o = plane + (long long)r * ow + X;
        if (vec && X >= c0 && X + 3 < c1) {
            *reinterpret_cast<uint32_t*>(o) = 0u;
        } else {
            for (int e = 0; e < 4; ++e)
                if (X + e >= c0 && X + e < c1) o[e] = 0;
        }
    }
}

__global__ void __launch_bounds__(THREADS) seg_masks_kernel(const __grid_constant__ SegParams p) {
    const int j = blockIdx.x, b = blockIdx.y;
    if (j >= p.counts[b]) return;
    __shared__ float s_mc[NM];
    __shared__ __align__(16) float s_p[SY * SX];
    __shared__ int s_sy[SY], s_sx[SX];
    __shared__ int s_iy[TY][2], s_ix[TX][2];
    __shared__ float s_wy[TY][2], s_wx[TX][2];

    const long long row = (long long)b * p.max_det + j;
    const long long a = p.keep[row];
    const bool has_a = a >= 0 && a < p.A;
    if (threadIdx.x < NM) s_mc[threadIdx.x] = has_a ? p.mc[((long long)b * p.A + a) * NM + threadIdx.x] : 0.f;
    const float x1 = p.det[row * 6], y1 = p.det[row * 6 + 1], x2 = p.det[row * 6 + 2], y2 = p.det[row * 6 + 3];

    const bool native = p.mode == YRE_MASK_NATIVE;
    int hlim = p.oh, wlim = p.ow;                     // the written window of the planes
    int in_h = p.mh, in_w = p.mw, off_y = 0, off_x = 0;   // the sampled proto window
    float sh = p.sh, sw = p.sw;
    int cy0, cy1, cx0, cx1;                           // crop: proto pixels (proto / input), output pixels (native)
    if (native) {
        const int w0 = (int)p.scale[b * 5 + 3], h0 = (int)p.scale[b * 5 + 4];
        if (w0 < 1 || h0 < 1) return;
        const double gain = fmin((double)p.mh / h0, (double)p.mw / w0);
        // Python's (mw - w0 * gain) / 2: the product is rounded before the subtraction (no FMA), or int() may truncate
        // a pad of exactly 8 to 7
        const double pw = __dsub_rn(p.mw, __dmul_rn(w0, gain)) / 2, ph = __dsub_rn(p.mh, __dmul_rn(h0, gain)) / 2;
        off_y = (int)ph; off_x = (int)pw;
        in_h = (int)(p.mh - ph) - off_y; in_w = (int)(p.mw - pw) - off_x;
        sh = (float)in_h / (float)h0; sw = (float)in_w / (float)w0;
        hlim = min(h0, p.oh); wlim = min(w0, p.ow);
        crop_range(y1, y2, hlim, cy0, cy1);
        crop_range(x1, x2, wlim, cx0, cx1);
        if (in_h < 1 || in_w < 1) cy1 = cy0;          // an empty proto window: every pixel is 0
    } else {
        crop_range(__fmul_rn(y1, p.ry), __fmul_rn(y2, p.ry), p.mh, cy0, cy1);
        crop_range(__fmul_rn(x1, p.rx), __fmul_rn(x2, p.rx), p.mw, cx0, cx1);
    }
    if (!has_a) cy1 = cy0;
    // the output band [R0, R1) x [C0, C1) outside which every output is 0: the crop (native), or the outputs whose
    // bilinear taps reach the crop (proto / input; with y1 in {y0, y0 + 1}, a tap is inside when y1 >= cy0 and y0 < cy1)
    __shared__ int s_band[4];
    if (threadIdx.x == 0) { s_band[0] = hlim; s_band[1] = 0; s_band[2] = wlim; s_band[3] = 0; }
    __syncthreads();                                  // s_mc, s_band
    if (native) {
        if (threadIdx.x == 0 && cy0 < cy1 && cx0 < cx1) { s_band[0] = cy0; s_band[1] = cy1; s_band[2] = cx0; s_band[3] = cx1; }
    } else if (cy0 < cy1 && cx0 < cx1) {
        int i0, i1;
        float l0, l1;
        for (int Y = threadIdx.x; Y < hlim; Y += THREADS) {
            bilinear_coeff(Y, sh, p.mh, i0, i1, l0, l1);
            if (i1 >= cy0 && i0 < cy1) { atomicMin(&s_band[0], Y); atomicMax(&s_band[1], Y + 1); }
        }
        for (int X = threadIdx.x; X < wlim; X += THREADS) {
            bilinear_coeff(X, sw, p.mw, i0, i1, l0, l1);
            if (i1 >= cx0 && i0 < cx1) { atomicMin(&s_band[2], X); atomicMax(&s_band[3], X + 1); }
        }
    }
    __syncthreads();
    int R0 = s_band[0], R1 = s_band[1], C0 = s_band[2], C1 = s_band[3];
    if (R0 >= R1 || C0 >= C1) R0 = R1 = C0 = C1 = 0;

    uint8_t* plane = p.masks + row * p.oh * p.ow;
    const bool vec = (p.ow & 3) == 0;
    // zeros outside the band: whole rows (one flat range when the window spans the plane's width), then the band's sides
    if (wlim == p.ow) {
        zero_fill(plane, (long long)R0 * p.ow);
        zero_fill(plane + (long long)R1 * p.ow, (long long)(hlim - R1) * p.ow);
    } else {
        zero_cols(plane, p.ow, 0, R0, 0, wlim, vec);
        zero_cols(plane, p.ow, R1, hlim, 0, wlim, vec);
    }
    const int C0a = C0 & ~3;                          // tiles start on 4-byte groups
    zero_cols(plane, p.ow, R0, R1, 0, C0a, vec);
    zero_cols(plane, p.ow, R0, R1, C1, wlim, vec);

    const int tr = threadIdx.x / (TX / 4), tg = (threadIdx.x % (TX / 4)) * 4;   // this thread's row and first column
    for (int Y0 = R0; Y0 < R1; Y0 += TY) {
        const int Y1 = min(Y0 + TY, R1);
        for (int X0 = C0a; X0 < C1; X0 += TX) {
            const int X1 = min(X0 + TX, C1);
            const int ax0 = max(X0, C0);              // [Y0, Y1) x [ax0, X1): the tile's outputs inside the band
            const int ny = axis_setup(Y0, Y1, sh, in_h, off_y, SY, s_sy, s_iy, s_wy);
            const int nx = axis_setup(ax0, X1, sw, in_w, off_x, SX, s_sx, s_ix, s_wx);
            __syncthreads();
            for (int k = threadIdx.x; k < ny * nx; k += THREADS) {
                const int ry = k / nx, rx = k - ry * nx;
                const int py = s_sy[ry], px = s_sx[rx];
                float v = 0.f;
                if (native || (py >= cy0 && py < cy1 && px >= cx0 && px < cx1)) {
                    const float4* q = reinterpret_cast<const float4*>(p.proto + (((long long)b * p.mh + py) * p.mw + px) * p.pitch);
                    float acc = 0.f;
#pragma unroll
                    for (int c = 0; c < NM / 4; ++c) {
                        const float4 f = q[c];
                        acc = __fadd_rn(acc, __fmul_rn(s_mc[4 * c], f.x));
                        acc = __fadd_rn(acc, __fmul_rn(s_mc[4 * c + 1], f.y));
                        acc = __fadd_rn(acc, __fmul_rn(s_mc[4 * c + 2], f.z));
                        acc = __fadd_rn(acc, __fmul_rn(s_mc[4 * c + 3], f.w));
                    }
                    v = 1.f / (1.f + expf(-acc));
                }
                s_p[ry * SX + rx] = v;
            }
            __syncthreads();
            const int Y = Y0 + tr;
            if (Y < Y1) {
                uint8_t m[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int X = X0 + tg + e;
                    float v = 0.f;
                    if (X >= ax0 && X < X1) {
                        const int iy = Y - Y0, ix = X - ax0;
                        const float h0 = s_wy[iy][0], h1 = s_wy[iy][1], w0 = s_wx[ix][0], w1 = s_wx[ix][1];
                        const float* r0 = s_p + s_iy[iy][0] * SX;
                        const float* r1 = s_p + s_iy[iy][1] * SX;
                        const float top = __fadd_rn(__fmul_rn(w0, r0[s_ix[ix][0]]), __fmul_rn(w1, r0[s_ix[ix][1]]));
                        const float bot = __fadd_rn(__fmul_rn(w0, r1[s_ix[ix][0]]), __fmul_rn(w1, r1[s_ix[ix][1]]));
                        v = __fadd_rn(__fmul_rn(h0, top), __fmul_rn(h1, bot));
                    }
                    m[e] = v > 0.5f;
                }
                uint8_t* o = plane + (long long)Y * p.ow + X0 + tg;
                if (vec && X0 + tg + 3 < X1) {
                    *reinterpret_cast<uint32_t*>(o) = m[0] | m[1] << 8 | m[2] << 16 | (uint32_t)m[3] << 24;
                } else {
                    for (int e = 0; e < 4 && X0 + tg + e < X1; ++e) o[e] = m[e];
                }
            }
            __syncthreads();                          // the staged tile is read until here
        }
    }
}

bool aligned(const void* ptr, size_t a) { return ((uintptr_t)ptr & (a - 1)) == 0; }

}  // namespace

extern "C" int yre_seg_masks(const yre_mask_desc* d, yre_stream_t s) {
    if (!d) YRE_FAIL(YRE_EINVAL, "seg_masks: null descriptor");
    if (!d->proto || !d->mc || !d->det || !d->counts || !d->keep_anchor || !d->masks)
        YRE_FAIL(YRE_EINVAL, "seg_masks: null pointer");
    if (d->mode != YRE_MASK_PROTO && d->mode != YRE_MASK_INPUT && d->mode != YRE_MASK_NATIVE)
        YRE_FAIL(YRE_EINVAL, "seg_masks: unknown mode %d", d->mode);
    if (d->nm != NM) YRE_FAIL(YRE_EINVAL, "seg_masks: nm=%d (32 mask coefficients only)", d->nm);
    if (d->B < 1 || d->n < 1 || d->n > d->B || d->n > 65535) YRE_FAIL(YRE_EINVAL, "seg_masks: %d images of a batch of %d", d->n, d->B);
    if (d->mh < 1 || d->mw < 1 || d->mh > 65536 || d->mw > 65536 || d->A < 1 || d->max_det < 1)
        YRE_FAIL(YRE_EINVAL, "seg_masks: proto %dx%d, %d anchors, max_det %d", d->mh, d->mw, d->A, d->max_det);
    if (d->proto_pitch < d->nm || d->proto_pitch % 4)
        YRE_FAIL(YRE_EINVAL, "seg_masks: proto pixel pitch %d (a multiple of 4, at least nm)", d->proto_pitch);
    if (!aligned(d->proto, 16) || !aligned(d->mc, 16) || !aligned(d->det, 4) || !aligned(d->masks, 4))
        YRE_FAIL(YRE_EINVAL, "seg_masks: proto and mc must be 16-byte aligned, det and masks 4-byte aligned");
    if (d->out_h < 1 || d->out_w < 1 || d->out_h > 65536 || d->out_w > 65536)
        YRE_FAIL(YRE_EINVAL, "seg_masks: output %dx%d", d->out_h, d->out_w);
    if (d->mode == YRE_MASK_NATIVE) {
        if (!d->scale || !aligned(d->scale, 4)) YRE_FAIL(YRE_EINVAL, "seg_masks: native mode needs the [B][5] scale rows");
    } else {
        if (d->in_h < 1 || d->in_w < 1 || d->in_h > 65536 || d->in_w > 65536)
            YRE_FAIL(YRE_EINVAL, "seg_masks: input extent %dx%d", d->in_h, d->in_w);
        const int oh = d->mode == YRE_MASK_PROTO ? d->mh : d->in_h, ow = d->mode == YRE_MASK_PROTO ? d->mw : d->in_w;
        if (d->out_h != oh || d->out_w != ow)
            YRE_FAIL(YRE_EINVAL, "seg_masks: output %dx%d, this mode writes %dx%d", d->out_h, d->out_w, oh, ow);
    }
    SegParams p;
    p.proto = d->proto; p.mc = d->mc; p.det = d->det; p.counts = d->counts; p.keep = d->keep_anchor; p.scale = d->scale;
    p.masks = d->masks;
    p.mh = d->mh; p.mw = d->mw; p.pitch = d->proto_pitch; p.A = d->A; p.max_det = d->max_det; p.mode = d->mode;
    p.oh = d->out_h; p.ow = d->out_w;
    p.rx = p.ry = p.sh = p.sw = 0.f;
    if (d->mode != YRE_MASK_NATIVE) {
        p.rx = (float)((double)d->mw / d->in_w); p.ry = (float)((double)d->mh / d->in_h);   // mw / iw: a Python float
        p.sh = (float)d->mh / (float)d->out_h; p.sw = (float)d->mw / (float)d->out_w;        // torch: (float)in / out
    }
    const dim3 grid((unsigned)d->max_det, (unsigned)d->n);
    seg_masks_kernel<<<grid, THREADS, 0, (cudaStream_t)s>>>(p);
    YRE_LAUNCH_CHECK("seg_masks");
    return YRE_OK;
}
