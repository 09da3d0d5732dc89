// Shared host/device helpers for libyre (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <atomic>
#include <mutex>
#include "../../include/yre.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libyre targets sm_100a (B200) only"
#endif

// ---- error plumbing (thread-local message, negative return codes) ---------------------------------
void yre_set_error(const char* fmt, ...);
#define YRE_FAIL(code, ...) do { yre_set_error(__VA_ARGS__); return (code); } while (0)
#define YRE_CUDA(expr) do { cudaError_t _e = (expr); if (_e != cudaSuccess) { \
    yre_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); return YRE_ECUDA; } } while (0)
#define YRE_LAUNCH_CHECK(name) do { cudaError_t _e = cudaGetLastError(); if (_e != cudaSuccess) { \
    yre_set_error("launch of %s failed: %s", name, cudaGetErrorString(_e)); return YRE_ECUDA; } } while (0)

static inline int yre_check_view(const yre_view* v, const char* what) {
    if (!v || !v->ptr) YRE_FAIL(YRE_EINVAL, "%s: null view", what);
    if (v->dtype != YRE_BF16 && v->dtype != YRE_F32 && v->dtype != YRE_F16) YRE_FAIL(YRE_EINVAL, "%s: bad dtype %d", what, v->dtype);
    if (v->layout != YRE_NHWC && v->layout != YRE_PHASE4) YRE_FAIL(YRE_EINVAL, "%s: bad layout %d", what, v->layout);
    if (v->B <= 0 || v->H <= 0 || v->W <= 0 || v->C <= 0 || v->c_off < 0 || v->c_off + v->C > v->C_total)
        YRE_FAIL(YRE_EINVAL, "%s: bad extent B%d H%d W%d C%d off%d tot%d", what, v->B, v->H, v->W, v->C, v->c_off, v->C_total);
    return YRE_OK;
}

static inline int yre_cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

// Function attributes (cudaFuncAttributeMaxDynamicSharedMemorySize) are PER DEVICE: run `f` once for every device
// ordinal a kernel family is launched on (a process may use cuda:0 and then cuda:1), thread-safe.
struct YrePerDeviceOnce {
    std::atomic<unsigned long long> done{0};
    std::mutex mu;
    template <typename F> int run(F&& f) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return f();
        if ((done.load(std::memory_order_acquire) >> dev) & 1ull) return YRE_OK;
        std::lock_guard<std::mutex> g(mu);
        if ((done.load(std::memory_order_relaxed) >> dev) & 1ull) return YRE_OK;
        const int e = f();
        if (e == YRE_OK) done.fetch_or(1ull << dev, std::memory_order_release);
        return e;
    }
};

// ---- device-side view addressing ----------------------------------------------------------------
struct DView {
    void* ptr;
    int dtype, layout, B, H, W, C_total, c_off, C;
    int Hp, Wp;   // parity-plane extent (PHASE4)
};

static inline DView make_dview(const yre_view& v) {
    DView d;
    d.ptr = v.ptr; d.dtype = v.dtype; d.layout = v.layout; d.B = v.B; d.H = v.H; d.W = v.W;
    d.C_total = v.C_total; d.c_off = v.c_off; d.C = v.C; d.Hp = (v.H + 1) / 2; d.Wp = (v.W + 1) / 2;
    return d;
}

// element index (in elements, not bytes) of channel 0 of the window at pixel (b,y,x)
__device__ __forceinline__ long long dview_pix(const DView& v, int b, int y, int x) {
    if (v.layout == YRE_NHWC) return (((long long)b * v.H + y) * v.W + x) * v.C_total + v.c_off;
    const int p = ((y & 1) << 1) | (x & 1);
    return ((((long long)p * v.B + b) * v.Hp + (y >> 1)) * v.Wp + (x >> 1)) * v.C_total + v.c_off;
}

template <typename T> struct Elt;
template <> struct Elt<float> {
    static __device__ __forceinline__ float ld(const void* p, long long i) { return ((const float*)p)[i]; }
    static __device__ __forceinline__ void st(void* p, long long i, float v) { ((float*)p)[i] = v; }
};
template <> struct Elt<__nv_bfloat16> {
    static __device__ __forceinline__ float ld(const void* p, long long i) { return __bfloat162float(((const __nv_bfloat16*)p)[i]); }
    static __device__ __forceinline__ void st(void* p, long long i, float v) { ((__nv_bfloat16*)p)[i] = __float2bfloat16_rn(v); }
};
template <> struct Elt<__half> {
    static __device__ __forceinline__ float ld(const void* p, long long i) { return __half2float(((const __half*)p)[i]); }
    static __device__ __forceinline__ void st(void* p, long long i, float v) { ((__half*)p)[i] = __float2half_rn(v); }
};

// 4 consecutive channels (index i multiple of 4 elements => 8/16-byte aligned)
template <typename T> __device__ __forceinline__ float4 ld4(const void* p, long long i);
template <> __device__ __forceinline__ float4 ld4<float>(const void* p, long long i) {
    return *reinterpret_cast<const float4*>((const float*)p + i);
}
template <> __device__ __forceinline__ float4 ld4<__nv_bfloat16>(const void* p, long long i) {
    const uint2 u = *reinterpret_cast<const uint2*>((const __nv_bfloat16*)p + i);
    float4 r;
    r.x = __uint_as_float(u.x << 16); r.y = __uint_as_float(u.x & 0xffff0000u);
    r.z = __uint_as_float(u.y << 16); r.w = __uint_as_float(u.y & 0xffff0000u);
    return r;
}
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
    __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&h);
}
// fp16 pair, round to nearest even (cvt.rn.f16x2.f32): values beyond +-65504 become +-inf, they are not saturated
__device__ __forceinline__ uint32_t pack_f16x2(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
__device__ __forceinline__ float2 unpack_f16x2(uint32_t u) { return __half22float2(*reinterpret_cast<const __half2*>(&u)); }
// the 16-bit pack of T (bf16 or fp16): lets one kernel body serve both activation types
template <typename T> __device__ __forceinline__ uint32_t pack16x2(float lo, float hi);
template <> __device__ __forceinline__ uint32_t pack16x2<__nv_bfloat16>(float lo, float hi) { return pack_bf16x2(lo, hi); }
template <> __device__ __forceinline__ uint32_t pack16x2<__half>(float lo, float hi) { return pack_f16x2(lo, hi); }
template <> __device__ __forceinline__ float4 ld4<__half>(const void* p, long long i) {
    const uint2 u = *reinterpret_cast<const uint2*>((const __half*)p + i);
    const float2 a = unpack_f16x2(u.x), b = unpack_f16x2(u.y);
    return make_float4(a.x, a.y, b.x, b.y);
}
template <typename T> __device__ __forceinline__ void st4(void* p, long long i, float4 v);
template <> __device__ __forceinline__ void st4<float>(void* p, long long i, float4 v) {
    *reinterpret_cast<float4*>((float*)p + i) = v;
}
template <> __device__ __forceinline__ void st4<__nv_bfloat16>(void* p, long long i, float4 v) {
    uint2 u; u.x = pack_bf16x2(v.x, v.y); u.y = pack_bf16x2(v.z, v.w);
    *reinterpret_cast<uint2*>((__nv_bfloat16*)p + i) = u;
}
template <> __device__ __forceinline__ void st4<__half>(void* p, long long i, float4 v) {
    uint2 u; u.x = pack_f16x2(v.x, v.y); u.y = pack_f16x2(v.z, v.w);
    *reinterpret_cast<uint2*>((__half*)p + i) = u;
}

// 8 consecutive channels as fp32 (index i multiple of 8 elements: one 16-byte access for bf16, two for fp32)
template <typename T> __device__ __forceinline__ void ld8(const void* p, long long i, float* o);
template <> __device__ __forceinline__ void ld8<float>(const void* p, long long i, float* o) {
    const float4 a = *reinterpret_cast<const float4*>((const float*)p + i), b = *reinterpret_cast<const float4*>((const float*)p + i + 4);
    o[0] = a.x; o[1] = a.y; o[2] = a.z; o[3] = a.w; o[4] = b.x; o[5] = b.y; o[6] = b.z; o[7] = b.w;
}
template <> __device__ __forceinline__ void ld8<__nv_bfloat16>(const void* p, long long i, float* o) {
    const uint4 u = *reinterpret_cast<const uint4*>((const __nv_bfloat16*)p + i);
    o[0] = __uint_as_float(u.x << 16); o[1] = __uint_as_float(u.x & 0xffff0000u);
    o[2] = __uint_as_float(u.y << 16); o[3] = __uint_as_float(u.y & 0xffff0000u);
    o[4] = __uint_as_float(u.z << 16); o[5] = __uint_as_float(u.z & 0xffff0000u);
    o[6] = __uint_as_float(u.w << 16); o[7] = __uint_as_float(u.w & 0xffff0000u);
}
template <> __device__ __forceinline__ void ld8<__half>(const void* p, long long i, float* o) {
    const uint4 u = *reinterpret_cast<const uint4*>((const __half*)p + i);
    const float2 a = unpack_f16x2(u.x), b = unpack_f16x2(u.y), c = unpack_f16x2(u.z), d = unpack_f16x2(u.w);
    o[0] = a.x; o[1] = a.y; o[2] = b.x; o[3] = b.y; o[4] = c.x; o[5] = c.y; o[6] = d.x; o[7] = d.y;
}
template <typename T> __device__ __forceinline__ void st8(void* p, long long i, const float* o);
template <> __device__ __forceinline__ void st8<float>(void* p, long long i, const float* o) {
    *reinterpret_cast<float4*>((float*)p + i) = make_float4(o[0], o[1], o[2], o[3]);
    *reinterpret_cast<float4*>((float*)p + i + 4) = make_float4(o[4], o[5], o[6], o[7]);
}
template <> __device__ __forceinline__ void st8<__nv_bfloat16>(void* p, long long i, const float* o) {
    uint4 u;
    u.x = pack_bf16x2(o[0], o[1]); u.y = pack_bf16x2(o[2], o[3]); u.z = pack_bf16x2(o[4], o[5]); u.w = pack_bf16x2(o[6], o[7]);
    *reinterpret_cast<uint4*>((__nv_bfloat16*)p + i) = u;
}
template <> __device__ __forceinline__ void st8<__half>(void* p, long long i, const float* o) {
    uint4 u;
    u.x = pack_f16x2(o[0], o[1]); u.y = pack_f16x2(o[2], o[3]); u.z = pack_f16x2(o[4], o[5]); u.w = pack_f16x2(o[6], o[7]);
    *reinterpret_cast<uint4*>((__half*)p + i) = u;
}

// One axis of torch's bilinear source index (F.interpolate(mode="bilinear", align_corners=False), size given): scale is
// (float)in / out; returns (i0, i1, l0, l1) for destination index d, fp32 with every rounding explicit (no contraction).
// Shared by K12 (TTA resize) and K15 (mask upsampling).
__device__ __forceinline__ void bilinear_coeff(int d, float scale, int in, int& i0, int& i1, float& l0, float& l1) {
    float src = __fsub_rn(__fmul_rn(scale, __fadd_rn((float)d, 0.5f)), 0.5f);
    src = src < 0.f ? 0.f : src;
    i0 = (int)src;
    i1 = i0 + (i0 < in - 1 ? 1 : 0);
    l1 = __fsub_rn(src, (float)i0);
    l0 = __fsub_rn(1.f, l1);
}

__device__ __forceinline__ float silu_f(float v) { return v / (1.0f + __expf(-v)); }
// SiLU with ONE MUFU op: x*sigmoid(x) = 0.5x*(1 + tanh(0.5x)); tanh.approx is good to ~2^-11 relative,
// far inside bf16's 2^-8 -- used wherever the result is rounded to bf16 anyway.
__device__ __forceinline__ float silu_tanh(float x) {
    const float h = 0.5f * x;
    float t;
    asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
    return fmaf(h, t, h);
}

// ---- op launchers implemented in the k_*.cu files (host side, used by the C API and the plan) -----
struct ConvTcPlan;   // pre-encoded tensor maps + tile config of one tcgen05 conv (k_conv_tc.cu)

int check_conv(const yre_conv_desc* d);                                     // descriptor validation shared by every conv entry point
// Every launcher takes nb, the number of images to compute (1 <= nb <= the views' B): the first nb images of the batch the
// views describe.  nb bounds grids and loops only; a view's B stays its layout (the parity-plane stride of YRE_PHASE4).
int launch_conv_ffma(const yre_conv_desc& d, int nb, cudaStream_t s);
int conv_tc_eligible(const yre_conv_desc& d, char* why, size_t why_len);
int conv_tc_prepare(const yre_conv_desc& d, ConvTcPlan** out);
int conv_tc_launch(ConvTcPlan* p, int nb, cudaStream_t s);
void conv_tc_free(ConvTcPlan* p);
void conv_tc_set_reverse(ConvTcPlan* p, int rev);                          // walk the M tiles last-to-first
void conv_tc_describe(const ConvTcPlan* p, char* out, size_t n);          // kernel variant + tile shape, for yre_plan_op_variant
int conv_tc_rebind(ConvTcPlan* p, const void* old_ptr, void* new_ptr);   // patches y/res only
int launch_stem(const yre_stem_desc& d, int nb, cudaStream_t s);
int launch_adown_prepool(const yre_view& x, const yre_view& avg_lo, const yre_view& max_hi, int nb, cudaStream_t s);
int launch_spp_maxpool(const yre_view& x, const yre_view& y5, const yre_view& y9, const yre_view& y13, int nb, cudaStream_t s);
int launch_upsample2x(const yre_view& x, const yre_view& y, int nb, cudaStream_t s);
int launch_cbfuse_sum(const yre_view* srcs, int n, const yre_view& target, const yre_view& y, int nb, cudaStream_t s);
int launch_nchw_to_view(const float* x, const yre_view& y, int nb, cudaStream_t s);
int launch_view_to_nchw(const yre_view& x, float* y, int nb, cudaStream_t s);
int launch_decode(const yre_decode_desc& d, int nb, cudaStream_t s);
int launch_decode_masks(const yre_decode_masks_desc& d, int nb, cudaStream_t s);   // K6 that also gathers mask coefficients
int launch_nms(const yre_nms_desc& d, int nb, cudaStream_t s);   // 3 launches (memset kernel, filter, sort+scan)
int launch_nms_multi_label(const yre_nms_desc& d, int nb, cudaStream_t s);   // same, every class above conf_thres
double conv_flops(const yre_conv_desc& d);
