// K1 (validation / fallback engine): fp32-accurate SIMT implicit-GEMM convolution.
//
//   y = [res +] act(conv(x, w) + bias)        -- reference: src/yolo/blocks/conv.py:88-89 et al.
//
// Products and accumulation are true fp32 FMAs (no TF32), so this engine is the "fp32 validation
// mode" the parity protocol needs; it also takes every shape the tcgen05 engine declines.
// GEMM view: M = B*Ho*Wo output pixels, N = Cout, K = k*k*Cin; 64x64 tile, 16-deep K slices,
// 256 threads x (4 pixels x 4 channels).
#include "yre_common.cuh"
#include <type_traits>

namespace {

struct FfmaParams {
    DView x, y, res, xu;     // xu: optional half-resolution source of the first Cu input channels (2x nearest upsample)
    int Cu;
    const void* w;
    const float* bias;
    int k, stride, pad, act, has_res;
    int Ho, Wo, Cin, Cout;
    long long M;
};

constexpr int TM = 64, TN = 64, TK = 16;

template <typename TIn, typename TOut>
__global__ void __launch_bounds__(256) conv_ffma_kernel(const FfmaParams p) {
    // a 16-bit residual has x's type (fp16 with fp16 operands, bf16 otherwise)
    using TRes16 = std::conditional_t<std::is_same_v<TIn, __half>, __half, __nv_bfloat16>;
    __shared__ __align__(16) float As[TK][TM + 4];
    __shared__ __align__(16) float Bs[TK][TN + 4];

    const int tid = threadIdx.x;
    const long long m0 = (long long)blockIdx.x * TM;
    const int n0 = blockIdx.y * TN;

    // loader role: row = tid/4 (pixel for A, out-channel for B), 4 consecutive k-channels
    const int lrow = tid >> 2, lk = (tid & 3) * 4;
    const long long lm = m0 + lrow;
    int lb = 0, loy = 0, lox = 0;
    const bool lvalid = lm < p.M;
    if (lvalid) {
        lox = (int)(lm % p.Wo);
        long long t = lm / p.Wo;
        loy = (int)(t % p.Ho);
        lb = (int)(t / p.Ho);
    }
    const int ln = n0 + lrow;
    const bool nvalid = ln < p.Cout;

    // compute role
    const int tx = tid & 15, ty = tid >> 4;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

    const int taps = p.k * p.k;
    for (int tap = 0; tap < taps; ++tap) {
        const int dy = tap / p.k, dx = tap % p.k;
        const int iy = loy * p.stride + dy - p.pad, ix = lox * p.stride + dx - p.pad;
        const bool inb = lvalid && iy >= 0 && iy < p.x.H && ix >= 0 && ix < p.x.W;
        const long long xbase = inb ? dview_pix(p.x, lb, iy, ix) : 0;
        const long long ubase = (inb && p.Cu) ? dview_pix(p.xu, lb, iy >> 1, ix >> 1) : 0;   // 1x1 only: nearest source pixel
        const long long wbase = ((long long)ln * taps + tap) * p.Cin;
        for (int c0 = 0; c0 < p.Cin; c0 += TK) {
            float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
            if (inb && c0 + lk < p.Cin)
                a = (c0 + lk < p.Cu) ? ld4<TIn>(p.xu.ptr, ubase + c0 + lk) : ld4<TIn>(p.x.ptr, xbase + c0 + lk - p.Cu);
            if (nvalid && c0 + lk < p.Cin) b = ld4<TIn>(p.w, wbase + c0 + lk);
            __syncthreads();
            As[lk + 0][lrow] = a.x; As[lk + 1][lrow] = a.y; As[lk + 2][lrow] = a.z; As[lk + 3][lrow] = a.w;
            Bs[lk + 0][lrow] = b.x; Bs[lk + 1][lrow] = b.y; Bs[lk + 2][lrow] = b.z; Bs[lk + 3][lrow] = b.w;
            __syncthreads();
#pragma unroll
            for (int kk = 0; kk < TK; ++kk) {
                const float4 av = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
                const float4 bv = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
                const float aa[4] = {av.x, av.y, av.z, av.w};
                const float bb[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(aa[i], bb[j], acc[i][j]);
            }
        }
    }

    const int n = n0 + tx * 4;
    if (n >= p.Cout) return;
    float bias[4] = {0.f, 0.f, 0.f, 0.f};
    if (p.bias) {
#pragma unroll
        for (int j = 0; j < 4; ++j) bias[j] = p.bias[n + j];
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const long long m = m0 + ty * 4 + i;
        if (m >= p.M) continue;
        const int ox = (int)(m % p.Wo);
        const long long t = m / p.Wo;
        const int oy = (int)(t % p.Ho), b = (int)(t / p.Ho);
        float v[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            v[j] = acc[i][j] + bias[j];
            if (p.act == YRE_ACT_SILU) v[j] = silu_f(v[j]);
        }
        if (p.has_res) {
            const float4 r = (p.res.dtype == YRE_F32) ? ld4<float>(p.res.ptr, dview_pix(p.res, b, oy, ox) + n)
                                                      : ld4<TRes16>(p.res.ptr, dview_pix(p.res, b, oy, ox) + n);
            v[0] += r.x; v[1] += r.y; v[2] += r.z; v[3] += r.w;
        }
        st4<TOut>(p.y.ptr, dview_pix(p.y, b, oy, ox) + n, make_float4(v[0], v[1], v[2], v[3]));
    }
}

}  // namespace

double conv_flops(const yre_conv_desc& d) {
    return 2.0 * d.y.B * d.y.H * d.y.W * (double)d.y.C * (d.x.C + (d.xu.ptr ? d.xu.C : 0)) * d.k * d.k;
}

int launch_conv_ffma(const yre_conv_desc& d, int nb, cudaStream_t s) {
    FfmaParams p;
    p.x = make_dview(d.x); p.y = make_dview(d.y);
    p.has_res = d.res.ptr != nullptr;
    p.res = p.has_res ? make_dview(d.res) : p.y;
    p.w = d.w; p.bias = d.bias; p.k = d.k; p.stride = d.stride; p.pad = d.k / 2; p.act = d.act;
    p.Ho = d.y.H; p.Wo = d.y.W; p.Cin = d.x.C; p.Cout = d.y.C;
    p.xu = p.x; p.Cu = 0;
    if (d.xu.ptr) {
        if (d.xu.C % 4 || d.xu.c_off % 4 || d.xu.C_total % 4) YRE_FAIL(YRE_EUNSUPPORTED, "conv_ffma: channel counts/offsets must be multiples of 4");
        p.xu = make_dview(d.xu); p.Cu = d.xu.C; p.Cin += p.Cu;
    }
    p.M = (long long)nb * d.y.H * d.y.W;              // the first nb images: pixels are image-major
    if (p.Cin % 4 || p.Cout % 4 || d.x.c_off % 4 || d.y.c_off % 4 || d.x.C_total % 4 || d.y.C_total % 4 ||
        (p.has_res && (d.res.c_off % 4 || d.res.C_total % 4)))
        YRE_FAIL(YRE_EUNSUPPORTED, "conv_ffma: channel counts/offsets must be multiples of 4");
    dim3 grid(yre_cdiv(p.M, TM), yre_cdiv(p.Cout, TN));
    if (d.x.dtype == YRE_F32 && d.y.dtype == YRE_F32) conv_ffma_kernel<float, float><<<grid, 256, 0, s>>>(p);
    else if (d.x.dtype == YRE_BF16 && d.y.dtype == YRE_BF16) conv_ffma_kernel<__nv_bfloat16, __nv_bfloat16><<<grid, 256, 0, s>>>(p);
    else if (d.x.dtype == YRE_BF16 && d.y.dtype == YRE_F32) conv_ffma_kernel<__nv_bfloat16, float><<<grid, 256, 0, s>>>(p);
    else if (d.x.dtype == YRE_F16 && d.y.dtype == YRE_F16) conv_ffma_kernel<__half, __half><<<grid, 256, 0, s>>>(p);
    else if (d.x.dtype == YRE_F16 && d.y.dtype == YRE_F32) conv_ffma_kernel<__half, float><<<grid, 256, 0, s>>>(p);
    else YRE_FAIL(YRE_EUNSUPPORTED, "conv_ffma: dtype combination x=%d y=%d", d.x.dtype, d.y.dtype);
    YRE_LAUNCH_CHECK("conv_ffma");
    return YRE_OK;
}
