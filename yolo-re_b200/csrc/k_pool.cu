// K3 (ADown pre-pool), K4 (SPPELAN pyramid), K5 (nearest x2 upsample), K8 (CBFuse sum) and the
// NCHW<->channels-last conversions at the API boundary.  All are HBM-bound: one thread moves
// 8 consecutive channels (16 B of bf16 or fp16 / 32 B of fp32) so that a warp touches whole 128 B lines.
#include "yre_common.cuh"
#include <float.h>

namespace {

// -------------------------------------------------------------------------------------------------
// K3: avg_pool2d(x,2,1,0) then, per channel half, [identity | max_pool2d(3,2,1)]
//     reference: src/yolo/blocks/downsample.py:41-44
// One thread per (output cell of the stride-2 grid, 8-channel group).  For the low channel half
// it emits the four average-map pixels (2oy+py, 2ox+px) -- i.e. one cell of each parity plane;
// for the high half it emits max over average rows/cols 2o-1..2o+1.
template <typename T>
__global__ void __launch_bounds__(256, 2) adown_prepool_kernel(DView x, DView lo, DView hi, int Ho, int Wo, int half) {
    // blockIdx.y selects the channel half, so the (very different) low/high paths never share a warp
    const int hgroups = half / 8;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)x.B * Ho * Wo * hgroups;
    if (idx >= total) return;
    const int g = (int)(idx % hgroups);
    long long t = idx / hgroups;
    const int ox = (int)(t % Wo); t /= Wo;
    const int oy = (int)(t % Ho);
    const int b = (int)(t / Ho);
    const int c = g * 8 + (blockIdx.y ? half : 0);
    const int Ha = x.H - 1, Wa = x.W - 1;          // average-map extent

    if (c < half) {
        // x rows 2oy..2oy+2, cols 2ox..2ox+2, streamed two rows at a time
        float ra[3][8], rb[3][8];
        auto load_row = [&](int iy, float (*r)[8]) {
#pragma unroll
            for (int q = 0; q < 3; ++q) {
                const int ix = 2 * ox + q;
                if (iy < x.H && ix < x.W) ld8<T>(x.ptr, dview_pix(x, b, iy, ix) + c, r[q]);
                else {
#pragma unroll
                    for (int e = 0; e < 8; ++e) r[q][e] = 0.f;
                }
            }
        };
        auto emit = [&](int py, float (*top)[8], float (*bot)[8]) {
#pragma unroll
            for (int px = 0; px < 2; ++px) {
                const int ay = 2 * oy + py, ax = 2 * ox + px;
                float o[8];
                const bool ok = ay < Ha && ax < Wa;
#pragma unroll
                for (int e = 0; e < 8; ++e)
                    o[e] = ok ? (((top[px][e] + top[px + 1][e]) + bot[px][e]) + bot[px + 1][e]) * 0.25f : 0.f;
                if (lo.layout == YRE_PHASE4) {
                    // every cell of every parity plane is written (zeros where no source pixel exists)
                    if ((ay >> 1) < lo.Hp && (ax >> 1) < lo.Wp) st8<T>(lo.ptr, dview_pix(lo, b, ay, ax) + c, o);
                } else if (ok) {
                    st8<T>(lo.ptr, dview_pix(lo, b, ay, ax) + c, o);
                }
            }
        };
        load_row(2 * oy, ra);
        load_row(2 * oy + 1, rb);
        emit(0, ra, rb);
        load_row(2 * oy + 2, ra);
        emit(1, rb, ra);
    } else {
        float m[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) m[e] = -FLT_MAX;
        // average rows 2oy-1..2oy+1 need x rows 2oy-1..2oy+2, x cols 2ox-1..2ox+2
        float prev[4][8];
        bool have_prev = false;
        for (int r = 0; r < 4; ++r) {
            const int iy = 2 * oy - 1 + r;
            const bool rowok = iy >= 0 && iy < x.H;
            float cur[4][8];
            if (rowok) {
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int ix = 2 * ox - 1 + q;
                    if (ix >= 0 && ix < x.W) ld8<T>(x.ptr, dview_pix(x, b, iy, ix) + c, cur[q]);
                    else {
#pragma unroll
                        for (int e = 0; e < 8; ++e) cur[q][e] = 0.f;
                    }
                }
            }
            // average row ay = iy-1 is built from x rows ay (prev) and ay+1 (cur)
            if (have_prev && rowok) {
#pragma unroll
                for (int q = 0; q < 3; ++q) {
                    const int ax = 2 * ox - 1 + q;
                    if (ax >= 0 && ax < Wa) {
#pragma unroll
                        for (int e = 0; e < 8; ++e)
                            m[e] = fmaxf(m[e], (((prev[q][e] + prev[q + 1][e]) + cur[q][e]) + cur[q + 1][e]) * 0.25f);
                    }
                }
            }
            if (rowok) {
#pragma unroll
                for (int q = 0; q < 4; ++q)
#pragma unroll
                    for (int e = 0; e < 8; ++e) prev[q][e] = cur[q][e];
            }
            have_prev = rowok;
        }
        st8<T>(hi.ptr, dview_pix(hi, b, oy, ox) + (c - half), m);
    }
}

// K3, tiled variant: a CTA stages a (2*TY+2) x (2*TX+2) input patch of 128 BYTES per pixel (64 bf16 /
// 32 fp32 channels = whole 128-byte lines, so HBM is read once) in shared memory in its storage type,
// then emits TY x TX cells of the stride-2 grid from it.  Pixel pitch 144 B: consecutive pixels start
// 4 banks apart, which makes the 16-byte shared-memory accesses conflict-free.
constexpr int AD_TY = 4, AD_TX = 16;
constexpr int AD_ROWS = 2 * AD_TY + 2, AD_COLS = 2 * AD_TX + 2;

template <typename T> struct SmemPix;
template <> struct SmemPix<__nv_bfloat16> {
    static constexpr int CHN = 64;
    static __device__ __forceinline__ void ld(const uint4* px, int g, float* o) {      // 8 channels of group g
        const uint4 u = px[g];
        o[0] = __uint_as_float(u.x << 16); o[1] = __uint_as_float(u.x & 0xffff0000u);
        o[2] = __uint_as_float(u.y << 16); o[3] = __uint_as_float(u.y & 0xffff0000u);
        o[4] = __uint_as_float(u.z << 16); o[5] = __uint_as_float(u.z & 0xffff0000u);
        o[6] = __uint_as_float(u.w << 16); o[7] = __uint_as_float(u.w & 0xffff0000u);
    }
};
template <> struct SmemPix<__half> {
    static constexpr int CHN = 64;
    static __device__ __forceinline__ void ld(const uint4* px, int g, float* o) {
        const uint4 u = px[g];
        const float2 a = unpack_f16x2(u.x), b = unpack_f16x2(u.y), c = unpack_f16x2(u.z), d = unpack_f16x2(u.w);
        o[0] = a.x; o[1] = a.y; o[2] = b.x; o[3] = b.y; o[4] = c.x; o[5] = c.y; o[6] = d.x; o[7] = d.y;
    }
};
template <> struct SmemPix<float> {
    static constexpr int CHN = 32;
    static __device__ __forceinline__ void ld(const uint4* px, int g, float* o) {
        const uint4 a = px[2 * g], b = px[2 * g + 1];
        o[0] = __uint_as_float(a.x); o[1] = __uint_as_float(a.y); o[2] = __uint_as_float(a.z); o[3] = __uint_as_float(a.w);
        o[4] = __uint_as_float(b.x); o[5] = __uint_as_float(b.y); o[6] = __uint_as_float(b.z); o[7] = __uint_as_float(b.w);
    }
};

// packed bf16x2 helpers for the bf16 product path of K3: the 2x2 average is formed with three HADD2 (horizontal pair
// sums, then their sum; each rounds to bf16: two roundings more than an fp32 sum, <= 3 * 2^-9 relative) and one exact x0.25;
// the 3x3 max is exact.  This quarters the instruction count of this issue-bound kernel; the fp32
// validation path keeps torch's exact summation order.
__device__ __forceinline__ uint32_t bf2_add(uint32_t a, uint32_t b) {
    __nv_bfloat162 r = __hadd2(*reinterpret_cast<__nv_bfloat162*>(&a), *reinterpret_cast<__nv_bfloat162*>(&b));
    return *reinterpret_cast<uint32_t*>(&r);
}
__device__ __forceinline__ uint32_t bf2_quarter(uint32_t a) {
    const __nv_bfloat162 q = __floats2bfloat162_rn(0.25f, 0.25f);
    __nv_bfloat162 r = __hmul2(*reinterpret_cast<__nv_bfloat162*>(&a), q);
    return *reinterpret_cast<uint32_t*>(&r);
}
__device__ __forceinline__ uint32_t bf2_max(uint32_t a, uint32_t b) {
    __nv_bfloat162 r = __hmax2(*reinterpret_cast<__nv_bfloat162*>(&a), *reinterpret_cast<__nv_bfloat162*>(&b));
    return *reinterpret_cast<uint32_t*>(&r);
}
__device__ __forceinline__ uint4 bf8_add(uint4 a, uint4 b) {
    return make_uint4(bf2_add(a.x, b.x), bf2_add(a.y, b.y), bf2_add(a.z, b.z), bf2_add(a.w, b.w));
}
__device__ __forceinline__ uint4 bf8_quarter(uint4 a) {
    return make_uint4(bf2_quarter(a.x), bf2_quarter(a.y), bf2_quarter(a.z), bf2_quarter(a.w));
}
__device__ __forceinline__ uint4 bf8_max(uint4 a, uint4 b) {
    return make_uint4(bf2_max(a.x, b.x), bf2_max(a.y, b.y), bf2_max(a.z, b.z), bf2_max(a.w, b.w));
}
// the same with packed fp16 (HADD2 / HMUL2 / HMNMX2): each sum rounds to fp16, <= 3 * 2^-12 relative
__device__ __forceinline__ uint32_t h2_add(uint32_t a, uint32_t b) {
    __half2 r = __hadd2(*reinterpret_cast<__half2*>(&a), *reinterpret_cast<__half2*>(&b));
    return *reinterpret_cast<uint32_t*>(&r);
}
__device__ __forceinline__ uint32_t h2_quarter(uint32_t a) {
    __half2 r = __hmul2(*reinterpret_cast<__half2*>(&a), __floats2half2_rn(0.25f, 0.25f));
    return *reinterpret_cast<uint32_t*>(&r);
}
__device__ __forceinline__ uint32_t h2_max(uint32_t a, uint32_t b) {
    __half2 r = __hmax2(*reinterpret_cast<__half2*>(&a), *reinterpret_cast<__half2*>(&b));
    return *reinterpret_cast<uint32_t*>(&r);
}
// eight packed 16-bit channels of type T: add, x0.25, max and the -inf pair
template <typename T> struct Pk8;
template <> struct Pk8<__nv_bfloat16> {
    static constexpr uint32_t NEG_INF2 = 0xff80ff80u;
    static __device__ __forceinline__ uint4 add(uint4 a, uint4 b) { return bf8_add(a, b); }
    static __device__ __forceinline__ uint4 quarter(uint4 a) { return bf8_quarter(a); }
    static __device__ __forceinline__ uint4 max(uint4 a, uint4 b) { return bf8_max(a, b); }
};
template <> struct Pk8<__half> {
    static constexpr uint32_t NEG_INF2 = 0xfc00fc00u;
    static __device__ __forceinline__ uint4 add(uint4 a, uint4 b) {
        return make_uint4(h2_add(a.x, b.x), h2_add(a.y, b.y), h2_add(a.z, b.z), h2_add(a.w, b.w));
    }
    static __device__ __forceinline__ uint4 quarter(uint4 a) { return make_uint4(h2_quarter(a.x), h2_quarter(a.y), h2_quarter(a.z), h2_quarter(a.w)); }
    static __device__ __forceinline__ uint4 max(uint4 a, uint4 b) {
        return make_uint4(h2_max(a.x, b.x), h2_max(a.y, b.y), h2_max(a.z, b.z), h2_max(a.w, b.w));
    }
};

template <typename T>
__global__ void __launch_bounds__(256, sizeof(T) == 2 ? 4 : 3) adown_tiled_kernel(DView x, DView lo, DView hi, int half, int tiles_x, int tiles_y) {
    constexpr int CHN = SmemPix<T>::CHN, G = CHN / 8;
    __shared__ uint4 tile[AD_ROWS][AD_COLS][9];        // 8 x 16 B of data + 16 B pad per pixel
    int t = blockIdx.x;
    const int tx = t % tiles_x; t /= tiles_x;
    const int ty = t % tiles_y;
    const int b = t / tiles_y;
    const int c0 = blockIdx.y * CHN;                   // channel chunk: entirely in the low or the high half
    const int oy0 = ty * AD_TY, ox0 = tx * AD_TX;
    const int iy0 = 2 * oy0 - 1, ix0 = 2 * ox0 - 1;
    const int Ha = x.H - 1, Wa = x.W - 1;
    const int tid = threadIdx.x;
    const T* xp = reinterpret_cast<const T*>(x.ptr);

    // every thread issues ALL of its 16-byte loads into registers first, then stores them to shared memory
    // (a load -> store -> load loop would serialise one HBM round trip per chunk)
    constexpr int NLDS = (AD_ROWS * AD_COLS * 8 + 255) / 256;       // 11
    if (sizeof(T) == 2 && x.layout == YRE_NHWC) {
        // row-linear addressing: thread (cc = tid/8, v = tid%8) copies column cc of all 10 rows (one pointer, a constant
        // row stride), threads 0..159 the two extra columns -- no per-load div/mod or 64-bit index arithmetic.  The copies
        // are cp.async (zero-fill outside the image): no register staging, so four CTAs fit an SM and one CTA's loads
        // overlap the arithmetic of the others (ncu: the shared-memory stores waiting on the loads were 28 % of the samples)
        const int v = tid & 7, cc = tid >> 3;
        const long long rs = (long long)x.W * x.C_total;
        const T* col = xp + (((long long)b * x.H + iy0) * x.W + (ix0 + cc)) * x.C_total + x.c_off + c0 + v * 8;
        const bool xin = (ix0 + cc) >= 0 && (ix0 + cc) < x.W;
        const uint32_t t0 = (uint32_t)__cvta_generic_to_shared(&tile[0][cc][v]);
        constexpr uint32_t ROWB = AD_COLS * 9 * 16;
#pragma unroll
        for (int q = 0; q < AD_ROWS; ++q) {
            const int iy = iy0 + q;
            const bool in = xin && iy >= 0 && iy < x.H;
            const T* src = in ? col + q * rs : xp;
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(t0 + (uint32_t)q * ROWB), "l"(src), "r"(in ? 16 : 0) : "memory");
        }
        if (tid < AD_ROWS * 16) {
            const int er = tid >> 4, ec = AD_COLS - 2 + ((tid >> 3) & 1);
            const int iy = iy0 + er, ix = ix0 + ec;
            const bool in = iy >= 0 && iy < x.H && ix >= 0 && ix < x.W;
            const T* src = in ? xp + (((long long)b * x.H + iy) * x.W + ix) * x.C_total + x.c_off + c0 + v * 8 : xp;
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"((uint32_t)__cvta_generic_to_shared(&tile[er][ec][v])), "l"(src), "r"(in ? 16 : 0) : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        asm volatile("cp.async.wait_group 0;" ::: "memory");
    } else {
        uint4 buf[NLDS];
#pragma unroll
        for (int q = 0; q < NLDS; ++q) {
            const int i = tid + 256 * q;
            const int v = i & 7, pix = i >> 3;
            const int r = pix / AD_COLS, c = pix - r * AD_COLS;
            const int iy = iy0 + r, ix = ix0 + c;
            buf[q] = make_uint4(0u, 0u, 0u, 0u);
            if (i < AD_ROWS * AD_COLS * 8 && iy >= 0 && iy < x.H && ix >= 0 && ix < x.W)
                buf[q] = *reinterpret_cast<const uint4*>(xp + dview_pix(x, b, iy, ix) + c0 + v * (16 / (int)sizeof(T)));
        }
#pragma unroll
        for (int q = 0; q < NLDS; ++q) {
            const int i = tid + 256 * q;
            if (i < AD_ROWS * AD_COLS * 8) {
                const int v = i & 7, pix = i >> 3;
                const int r = pix / AD_COLS, c = pix - r * AD_COLS;
                tile[r][c][v] = buf[q];
            }
        }
    }
    __syncthreads();

    if constexpr (sizeof(T) == 2) {
        using P = Pk8<T>;
        T* lop = reinterpret_cast<T*>(lo.ptr);
        T* hip = reinterpret_cast<T*>(hi.ptr);
        if (c0 < half) {
            // item k of a thread = average pixel (ayl = k, axl = tid / 8), channel group g = tid % 8: the output address is
            // one base per row parity plus a constant row stride
            static_assert(G == 8 && 2 * AD_TX * G == 256, "item decomposition assumes 256 items per average row");
            const int g = tid & 7, axl = tid >> 3;
            const int ax = 2 * ox0 + axl;
            const bool ph4 = lo.layout == YRE_PHASE4;
            long long base[2], rstep;
            if (ph4) {
                for (int pk = 0; pk < 2; ++pk)
                    base[pk] = (((((long long)(pk * 2 + (ax & 1)) * lo.B + b) * lo.Hp + oy0) * lo.Wp + (ax >> 1)) * lo.C_total) + lo.c_off + c0 + g * 8;
                rstep = (long long)lo.Wp * lo.C_total;
            } else {
                base[0] = (((long long)b * lo.H + 2 * oy0) * lo.W + ax) * lo.C_total + lo.c_off + c0 + g * 8;
                base[1] = base[0] + (long long)lo.W * lo.C_total;
                rstep = 2ll * lo.W * lo.C_total;
            }
            const bool xok = ax < Wa, xst = ph4 ? (ax >> 1) < lo.Wp : xok;
            // horizontal pair sums are shared by vertically adjacent averages: avg[k] = (h[k+1] + h[k+2]) / 4
            uint4 hprev = P::add(tile[1][axl + 1][g], tile[1][axl + 2][g]);
#pragma unroll
            for (int k = 0; k < 2 * AD_TY; ++k) {
                const int ay = 2 * oy0 + k;
                const bool ok = xok && ay < Ha;
                const uint4 hcur = P::add(tile[k + 2][axl + 1][g], tile[k + 2][axl + 2][g]);
                uint4 o = make_uint4(0u, 0u, 0u, 0u);
                if (ok) o = P::quarter(P::add(hprev, hcur));
                hprev = hcur;
                const bool st = ph4 ? (xst && (ay >> 1) < lo.Hp) : ok;       // parity planes: cells without a source pixel hold zeros
                if (st) *reinterpret_cast<uint4*>(lop + base[k & 1] + (k >> 1) * rstep) = o;
            }
        } else {
            for (int i = tid; i < AD_TY * AD_TX * G; i += 256) {
                const int g = i % G;
                const int oxl = (i / G) % AD_TX, oyl = i / (G * AD_TX);
                const int oy = oy0 + oyl, ox = ox0 + oxl;
                if (oy >= hi.H || ox >= hi.W) continue;
                // max over the 3x3 window of 2x2 averages: horizontal pair sums h[r][q] are shared by the two average rows
                // that use them, and the exact x0.25 is applied once after the max (monotonic, power of two)
                uint4 m = make_uint4(P::NEG_INF2, P::NEG_INF2, P::NEG_INF2, P::NEG_INF2);      // -inf pairs
                uint4 hp[3], hc[3];
                {
                    const uint4 t0 = tile[2 * oyl][2 * oxl][g], t1 = tile[2 * oyl][2 * oxl + 1][g], t2 = tile[2 * oyl][2 * oxl + 2][g], t3 = tile[2 * oyl][2 * oxl + 3][g];
                    hp[0] = P::add(t0, t1); hp[1] = P::add(t1, t2); hp[2] = P::add(t2, t3);
                }
#pragma unroll
                for (int j = 0; j < 3; ++j) {
                    const uint4 t0 = tile[2 * oyl + j + 1][2 * oxl][g], t1 = tile[2 * oyl + j + 1][2 * oxl + 1][g],
                                t2 = tile[2 * oyl + j + 1][2 * oxl + 2][g], t3 = tile[2 * oyl + j + 1][2 * oxl + 3][g];
                    hc[0] = P::add(t0, t1); hc[1] = P::add(t1, t2); hc[2] = P::add(t2, t3);
                    const int ay = 2 * oy - 1 + j;
                    if (ay >= 0 && ay < Ha) {
#pragma unroll
                        for (int q = 0; q < 3; ++q) {
                            const int ax = 2 * ox - 1 + q;
                            if (ax >= 0 && ax < Wa) m = P::max(m, P::add(hp[q], hc[q]));
                        }
                    }
#pragma unroll
                    for (int q = 0; q < 3; ++q) hp[q] = hc[q];
                }
                m = P::quarter(m);
                *reinterpret_cast<uint4*>(hip + dview_pix(hi, b, oy, ox) + (c0 - half) + g * 8) = m;
            }
        }
        return;
    }
    if (c0 < half) {
        // (2*TY) x (2*TX) average pixels x G channel groups; item -> (ayl, axl, g), g fastest
        for (int i = tid; i < 2 * AD_TY * 2 * AD_TX * G; i += 256) {
            const int g = i % G;
            const int axl = (i / G) % (2 * AD_TX), ayl = i / (G * 2 * AD_TX);
            const int ay = 2 * oy0 + ayl, ax = 2 * ox0 + axl;
            const bool ok = ay < Ha && ax < Wa;
            float o[8];
            if (ok) {
                float a[8], bq[8], cq[8], d[8];
                SmemPix<T>::ld(tile[ayl + 1][axl + 1], g, a);
                SmemPix<T>::ld(tile[ayl + 1][axl + 2], g, bq);
                SmemPix<T>::ld(tile[ayl + 2][axl + 1], g, cq);
                SmemPix<T>::ld(tile[ayl + 2][axl + 2], g, d);
#pragma unroll
                for (int e = 0; e < 8; ++e) o[e] = (((a[e] + bq[e]) + cq[e]) + d[e]) * 0.25f;
            } else {
#pragma unroll
                for (int e = 0; e < 8; ++e) o[e] = 0.f;
            }
            if (lo.layout == YRE_PHASE4) {
                if ((ay >> 1) < lo.Hp && (ax >> 1) < lo.Wp) st8<T>(lo.ptr, dview_pix(lo, b, ay, ax) + c0 + g * 8, o);
            } else if (ok) {
                st8<T>(lo.ptr, dview_pix(lo, b, ay, ax) + c0 + g * 8, o);
            }
        }
    } else {
        // TY x TX cells x G groups: the 4x4 input window is read once, rows stream through registers
        for (int i = tid; i < AD_TY * AD_TX * G; i += 256) {
            const int g = i % G;
            const int oxl = (i / G) % AD_TX, oyl = i / (G * AD_TX);
            const int oy = oy0 + oyl, ox = ox0 + oxl;
            if (oy >= hi.H || ox >= hi.W) continue;
            float m[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) m[e] = -FLT_MAX;
            float prev[4][8], cur[4][8];
#pragma unroll
            for (int q = 0; q < 4; ++q) SmemPix<T>::ld(tile[2 * oyl][2 * oxl + q], g, prev[q]);
#pragma unroll
            for (int j = 0; j < 3; ++j) {                 // average row ay = 2*oy - 1 + j uses tile rows 2*oyl+j, +1
#pragma unroll
                for (int q = 0; q < 4; ++q) SmemPix<T>::ld(tile[2 * oyl + j + 1][2 * oxl + q], g, cur[q]);
                const int ay = 2 * oy - 1 + j;
                if (ay >= 0 && ay < Ha) {
#pragma unroll
                    for (int q = 0; q < 3; ++q) {
                        const int ax = 2 * ox - 1 + q;
                        if (ax >= 0 && ax < Wa) {
#pragma unroll
                            for (int e = 0; e < 8; ++e)
                                m[e] = fmaxf(m[e], (((prev[q][e] + prev[q + 1][e]) + cur[q][e]) + cur[q + 1][e]) * 0.25f);
                        }
                    }
                }
#pragma unroll
                for (int q = 0; q < 4; ++q)
#pragma unroll
                    for (int e = 0; e < 8; ++e) prev[q][e] = cur[q][e];
            }
            st8<T>(hi.ptr, dview_pix(hi, b, oy, ox) + (c0 - half) + g * 8, m);
        }
    }
}

// -------------------------------------------------------------------------------------------------
// K4: windows 5/9/13 max (== three chained MaxPool2d(5,1,2); reference sppelan.py:44-47)
template <typename T>
__global__ void __launch_bounds__(256) spp_kernel(DView x, DView y5, DView y9, DView y13) {
    const int groups = x.C / 8;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)x.B * x.H * x.W * groups;
    if (idx >= total) return;
    const int c = (int)(idx % groups) * 8;
    long long t = idx / groups;
    const int px = (int)(t % x.W); t /= x.W;
    const int py = (int)(t % x.H);
    const int b = (int)(t / x.H);
    float m5[8], m9[8], m13[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) m5[e] = m9[e] = m13[e] = -FLT_MAX;
    for (int dy = -6; dy <= 6; ++dy) {
        const int iy = py + dy;
        if (iy < 0 || iy >= x.H) continue;
        const int ady = dy < 0 ? -dy : dy;
        for (int dx = -6; dx <= 6; ++dx) {
            const int ix = px + dx;
            if (ix < 0 || ix >= x.W) continue;
            const int adx = dx < 0 ? -dx : dx;
            const int r = ady > adx ? ady : adx;
            float v[8];
            ld8<T>(x.ptr, dview_pix(x, b, iy, ix) + c, v);
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                m13[e] = fmaxf(m13[e], v[e]);
                if (r <= 4) m9[e] = fmaxf(m9[e], v[e]);
                if (r <= 2) m5[e] = fmaxf(m5[e], v[e]);
            }
        }
    }
    st8<T>(y5.ptr, dview_pix(y5, b, py, px) + c, m5);
    st8<T>(y9.ptr, dview_pix(y9, b, py, px) + c, m9);
    st8<T>(y13.ptr, dview_pix(y13, b, py, px) + c, m13);
}

// K4, plane-resident variant: one CTA keeps a whole HxW plane of CHK channels in shared memory and runs
// the reference's three chained 5x5 pools literally (each as a row pass + a column pass, ping-ponging
// between two buffers): 30 shared-memory reads per element instead of 169 global loads.  max() is exact,
// so the result is bit-identical to the direct kernel.
template <typename T>
__global__ void __launch_bounds__(256) spp_plane_kernel(DView x, DView y5, DView y9, DView y13, int chk) {
    extern __shared__ __align__(16) float sp[];
    const int H = x.H, W = x.W, g4 = chk / 4;
    const int plane = H * W * chk;
    float* A = sp;
    float* Bf = sp + plane;
    const int b = blockIdx.x, c0 = blockIdx.y * chk;
    const int items8 = H * W * (chk / 8);
    for (int i = threadIdx.x; i < items8; i += blockDim.x) {
        const int g = i % (chk / 8), pix = i / (chk / 8);
        float f[8];
        ld8<T>(x.ptr, dview_pix(x, b, pix / W, pix % W) + c0 + g * 8, f);
        float4* d = reinterpret_cast<float4*>(A + pix * chk + g * 8);
        d[0] = make_float4(f[0], f[1], f[2], f[3]); d[1] = make_float4(f[4], f[5], f[6], f[7]);
    }
    __syncthreads();
    const int items4 = H * W * g4;
    const DView outs[3] = {y5, y9, y13};
    for (int lvl = 0; lvl < 3; ++lvl) {
        // row pass A -> Bf
        for (int i = threadIdx.x; i < items4; i += blockDim.x) {
            const int g = i % g4, pix = i / g4, px = pix % W;
            float4 m = *reinterpret_cast<const float4*>(A + pix * chk + g * 4);
#pragma unroll
            for (int d = -2; d <= 2; ++d) {
                if (d == 0 || px + d < 0 || px + d >= W) continue;
                const float4 v = *reinterpret_cast<const float4*>(A + (pix + d) * chk + g * 4);
                m.x = fmaxf(m.x, v.x); m.y = fmaxf(m.y, v.y); m.z = fmaxf(m.z, v.z); m.w = fmaxf(m.w, v.w);
            }
            *reinterpret_cast<float4*>(Bf + pix * chk + g * 4) = m;
        }
        __syncthreads();
        // column pass Bf -> A
        for (int i = threadIdx.x; i < items4; i += blockDim.x) {
            const int g = i % g4, pix = i / g4, py = pix / W;
            float4 m = *reinterpret_cast<const float4*>(Bf + pix * chk + g * 4);
#pragma unroll
            for (int d = -2; d <= 2; ++d) {
                if (d == 0 || py + d < 0 || py + d >= H) continue;
                const float4 v = *reinterpret_cast<const float4*>(Bf + (pix + d * W) * chk + g * 4);
                m.x = fmaxf(m.x, v.x); m.y = fmaxf(m.y, v.y); m.z = fmaxf(m.z, v.z); m.w = fmaxf(m.w, v.w);
            }
            *reinterpret_cast<float4*>(A + pix * chk + g * 4) = m;
        }
        __syncthreads();
        for (int i = threadIdx.x; i < items8; i += blockDim.x) {
            const int g = i % (chk / 8), pix = i / (chk / 8);
            const float4* sp4 = reinterpret_cast<const float4*>(A + pix * chk + g * 8);
            const float4 u = sp4[0], w = sp4[1];
            const float f[8] = {u.x, u.y, u.z, u.w, w.x, w.y, w.z, w.w};
            st8<T>(outs[lvl].ptr, dview_pix(outs[lvl], b, pix / W, pix % W) + c0 + g * 8, f);
        }
        // the next row pass only reads A, which is complete: no barrier needed before it
    }
}

// bf16 product path of the plane-resident K4: the plane stays in bf16 (eight channels per 16-byte word), max is taken
// with packed HMNMX2 -- max() of bf16 values is exact, so the result equals the fp32-staged kernel's bit for bit -- and the
// column pass stores its result straight to the output slice.  A CTA owns CHK channels of one image; with CHK = 64 a
// pixel is one full 128-byte line on both the load and the three store sides.
// The fp16 instantiation is the same kernel with max.f16x2 (exact as well).
template <typename T> __device__ __forceinline__ uint4 hmax8(const uint4 a, const uint4 b);
template <> __device__ __forceinline__ uint4 hmax8<__nv_bfloat16>(const uint4 a, const uint4 b) {
    uint4 r;
    asm("max.bf16x2 %0, %1, %2;" : "=r"(r.x) : "r"(a.x), "r"(b.x));
    asm("max.bf16x2 %0, %1, %2;" : "=r"(r.y) : "r"(a.y), "r"(b.y));
    asm("max.bf16x2 %0, %1, %2;" : "=r"(r.z) : "r"(a.z), "r"(b.z));
    asm("max.bf16x2 %0, %1, %2;" : "=r"(r.w) : "r"(a.w), "r"(b.w));
    return r;
}
template <> __device__ __forceinline__ uint4 hmax8<__half>(const uint4 a, const uint4 b) {
    uint4 r;
    asm("max.f16x2 %0, %1, %2;" : "=r"(r.x) : "r"(a.x), "r"(b.x));
    asm("max.f16x2 %0, %1, %2;" : "=r"(r.y) : "r"(a.y), "r"(b.y));
    asm("max.f16x2 %0, %1, %2;" : "=r"(r.z) : "r"(a.z), "r"(b.z));
    asm("max.f16x2 %0, %1, %2;" : "=r"(r.w) : "r"(a.w), "r"(b.w));
    return r;
}

template <typename T, int G>      // T: bf16 or fp16; G = CHK / 8 sixteen-byte words per pixel
__global__ void __launch_bounds__(1024) spp_plane16_kernel(DView x, DView y5, DView y9, DView y13) {
    extern __shared__ __align__(16) uint4 sq[];
    const int H = x.H, W = x.W, items = H * W * G;
    uint4* A = sq;
    uint4* Bf = sq + items;
    const int b = blockIdx.x, c0 = blockIdx.y * (G * 8);
    const T* xp = reinterpret_cast<const T*>(x.ptr);
    for (int i = threadIdx.x; i < items; i += blockDim.x) {
        const int g = i % G, pix = i / G;
        A[i] = *reinterpret_cast<const uint4*>(xp + dview_pix(x, b, pix / W, pix % W) + c0 + g * 8);
    }
    __syncthreads();
    const DView outs[3] = {y5, y9, y13};
    for (int lvl = 0; lvl < 3; ++lvl) {
        for (int i = threadIdx.x; i < items; i += blockDim.x) {          // row pass A -> Bf
            const int px = (i / G) % W;
            uint4 m = A[i];
#pragma unroll
            for (int d = -2; d <= 2; ++d) {
                if (d == 0 || px + d < 0 || px + d >= W) continue;
                m = hmax8<T>(m, A[i + d * G]);
            }
            Bf[i] = m;
        }
        __syncthreads();
        T* op = reinterpret_cast<T*>(outs[lvl].ptr);
        for (int i = threadIdx.x; i < items; i += blockDim.x) {          // column pass Bf -> A and the output slice
            const int g = i % G, pix = i / G, py = pix / W;
            uint4 m = Bf[i];
#pragma unroll
            for (int d = -2; d <= 2; ++d) {
                if (d == 0 || py + d < 0 || py + d >= H) continue;
                m = hmax8<T>(m, Bf[i + d * W * G]);
            }
            A[i] = m;
            *reinterpret_cast<uint4*>(op + dview_pix(outs[lvl], b, py, pix % W) + c0 + g * 8) = m;
        }
        __syncthreads();
    }
}

// -------------------------------------------------------------------------------------------------
// K5: nearest x2 (reference: nn.Upsample, parser.py:159-171) written into the consumer's slice
template <typename T>
__global__ void __launch_bounds__(256) upsample2x_kernel(DView x, DView y) {
    // one thread per INPUT (pixel, 8-channel group): one 16-byte load feeds the four output pixels
    const int groups = x.C / 8;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)x.B * x.H * x.W * groups;
    if (idx >= total) return;
    const int c = (int)(idx % groups) * 8;
    long long t = idx / groups;
    const int ix = (int)(t % x.W); t /= x.W;
    const int iy = (int)(t % x.H);
    const int b = (int)(t / x.H);
    float v[8];
    ld8<T>(x.ptr, dview_pix(x, b, iy, ix) + c, v);
    if (y.layout == YRE_NHWC) {
        const long long o = dview_pix(y, b, 2 * iy, 2 * ix) + c;
        const long long rs = (long long)y.W * y.C_total;
        st8<T>(y.ptr, o, v); st8<T>(y.ptr, o + y.C_total, v);
        st8<T>(y.ptr, o + rs, v); st8<T>(y.ptr, o + rs + y.C_total, v);
    } else {
#pragma unroll
        for (int q = 0; q < 4; ++q) st8<T>(y.ptr, dview_pix(y, b, 2 * iy + (q >> 1), 2 * ix + (q & 1)) + c, v);
    }
}

// -------------------------------------------------------------------------------------------------
// K8: CBFuse (reference auxiliary.py:100-110): nearest-resize every source to the target size,
// stack with the target and sum in that order.
struct FuseSrcs { DView v[8]; int n; };
template <typename T>
__global__ void __launch_bounds__(256) cbfuse_kernel(FuseSrcs srcs, DView tgt, DView y) {
    const int groups = y.C / 8;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)y.B * y.H * y.W * groups;
    if (idx >= total) return;
    const int c = (int)(idx % groups) * 8;
    long long t = idx / groups;
    const int ox = (int)(t % y.W); t /= y.W;
    const int oy = (int)(t % y.H);
    const int b = (int)(t / y.H);
    float acc[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) acc[e] = 0.f;
    for (int i = 0; i < srcs.n; ++i) {
        const DView& sv = srcs.v[i];
        // F.interpolate(mode="nearest"): src = floor(dst * in/out)
        const int sy = min((int)floorf(oy * ((float)sv.H / y.H)), sv.H - 1);
        const int sx = min((int)floorf(ox * ((float)sv.W / y.W)), sv.W - 1);
        float v[8];
        ld8<T>(sv.ptr, dview_pix(sv, b, sy, sx) + c, v);
#pragma unroll
        for (int e = 0; e < 8; ++e) acc[e] += v[e];
    }
    float v[8];
    ld8<T>(tgt.ptr, dview_pix(tgt, b, oy, ox) + c, v);
#pragma unroll
    for (int e = 0; e < 8; ++e) acc[e] += v[e];
    st8<T>(y.ptr, dview_pix(y, b, oy, ox) + c, acc);
}

// -------------------------------------------------------------------------------------------------
// NCHW fp32 <-> channels-last view, through a 32x32 shared-memory transpose (channels x pixels)
template <typename T>
__global__ void __launch_bounds__(256) nchw_to_view_kernel(const float* __restrict__ x, DView y) {
    __shared__ float tile[32][33];
    const int b = blockIdx.z;
    const long long HW = (long long)y.H * y.W;
    const long long p0 = (long long)blockIdx.x * 32;
    const int c0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 8 rows per pass
    for (int r = ty; r < 32; r += 8) {
        const int c = c0 + r;
        const long long p = p0 + tx;
        tile[r][tx] = (c < y.C && p < HW) ? x[((long long)b * y.C + c) * HW + p] : 0.f;
    }
    __syncthreads();
    for (int r = ty; r < 32; r += 8) {
        const long long p = p0 + r;
        const int c = c0 + tx;
        if (p < HW && c < y.C) {
            const int py = (int)(p / y.W), px = (int)(p % y.W);
            Elt<T>::st(y.ptr, dview_pix(y, b, py, px) + c, tile[tx][r]);
        }
    }
}

template <typename T>
__global__ void __launch_bounds__(256) view_to_nchw_kernel(DView x, float* __restrict__ y) {
    __shared__ float tile[32][33];
    const int b = blockIdx.z;
    const long long HW = (long long)x.H * x.W;
    const long long p0 = (long long)blockIdx.x * 32;
    const int c0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    for (int r = ty; r < 32; r += 8) {
        const long long p = p0 + r;
        const int c = c0 + tx;
        float v = 0.f;
        if (p < HW && c < x.C) {
            const int py = (int)(p / x.W), px = (int)(p % x.W);
            v = Elt<T>::ld(x.ptr, dview_pix(x, b, py, px) + c);
        }
        tile[r][tx] = v;     // [pixel][channel]
    }
    __syncthreads();
    for (int r = ty; r < 32; r += 8) {
        const int c = c0 + r;
        const long long p = p0 + tx;
        if (c < x.C && p < HW) y[((long long)b * x.C + c) * HW + p] = tile[tx][r];
    }
}

int check8(const yre_view& v, const char* what) {
    if (yre_check_view(&v, what)) return YRE_EINVAL;
    if (v.C % 8 || v.c_off % 8 || v.C_total % 8) YRE_FAIL(YRE_EUNSUPPORTED, "%s: channels must be multiples of 8", what);
    return YRE_OK;
}

}  // namespace

int launch_adown_prepool(const yre_view& x, const yre_view& lo, const yre_view& hi, cudaStream_t s) {
    if (check8(x, "adown.x") || check8(lo, "adown.avg_lo") || check8(hi, "adown.max_hi")) return YRE_EINVAL;
    if (x.layout != YRE_NHWC || hi.layout != YRE_NHWC) YRE_FAIL(YRE_EUNSUPPORTED, "adown: x and max_hi must be NHWC");
    if (x.C % 16) YRE_FAIL(YRE_EUNSUPPORTED, "adown: C must be a multiple of 16");
    const int half = x.C / 2;
    const int Ho = (x.H - 1 + 2 - 3) / 2 + 1, Wo = (x.W - 1 + 2 - 3) / 2 + 1;
    if (lo.C != half || hi.C != half || lo.H != x.H - 1 || lo.W != x.W - 1 || hi.H != Ho || hi.W != Wo ||
        lo.B != x.B || hi.B != x.B || lo.dtype != x.dtype || hi.dtype != x.dtype)
        YRE_FAIL(YRE_EINVAL, "adown: output views do not match the input (want avg %dx%d C%d, max %dx%d)", x.H - 1, x.W - 1, half, Ho, Wo);
    // the thread grid walks ceil((H-1)/2) x ceil((W-1)/2) cells, which covers both outputs
    const int Gy = (x.H - 1 + 1) / 2, Gx = (x.W - 1 + 1) / 2;
    if (Gy < Ho || Gx < Wo) YRE_FAIL(YRE_EINVAL, "adown: grid smaller than the pooled output");
    const long long total = (long long)x.B * Gy * Gx * (half / 8);
    dim3 grid(yre_cdiv(total, 256), 2);
    // NB: kernel indexes its cell grid with (Ho,Wo) = (Gy,Gx); cells beyond hi's extent never
    // occur because Gy==Ho, Gx==Wo for every H,W >= 2.
    if (Gy != Ho || Gx != Wo) YRE_FAIL(YRE_EUNSUPPORTED, "adown: H=%d W=%d", x.H, x.W);
    const int chn = x.dtype == YRE_F32 ? 32 : 64;      // 128 bytes of channels per CTA
    if (half % chn == 0) {
        const int tiles_x = yre_cdiv(Gx, AD_TX), tiles_y = yre_cdiv(Gy, AD_TY);
        dim3 tg((unsigned)(tiles_x * tiles_y * x.B), (unsigned)(x.C / chn));
        if (x.dtype == YRE_F32) adown_tiled_kernel<float><<<tg, 256, 0, s>>>(make_dview(x), make_dview(lo), make_dview(hi), half, tiles_x, tiles_y);
        else if (x.dtype == YRE_F16) adown_tiled_kernel<__half><<<tg, 256, 0, s>>>(make_dview(x), make_dview(lo), make_dview(hi), half, tiles_x, tiles_y);
        else adown_tiled_kernel<__nv_bfloat16><<<tg, 256, 0, s>>>(make_dview(x), make_dview(lo), make_dview(hi), half, tiles_x, tiles_y);
    } else if (x.dtype == YRE_F32) adown_prepool_kernel<float><<<grid, 256, 0, s>>>(make_dview(x), make_dview(lo), make_dview(hi), Gy, Gx, half);
    else if (x.dtype == YRE_F16) adown_prepool_kernel<__half><<<grid, 256, 0, s>>>(make_dview(x), make_dview(lo), make_dview(hi), Gy, Gx, half);
    else adown_prepool_kernel<__nv_bfloat16><<<grid, 256, 0, s>>>(make_dview(x), make_dview(lo), make_dview(hi), Gy, Gx, half);
    YRE_LAUNCH_CHECK("adown_prepool");
    return YRE_OK;
}

int launch_spp_maxpool(const yre_view& x, const yre_view& y5, const yre_view& y9, const yre_view& y13, cudaStream_t s) {
    if (check8(x, "spp.x") || check8(y5, "spp.y5") || check8(y9, "spp.y9") || check8(y13, "spp.y13")) return YRE_EINVAL;
    const yre_view* ys[3] = {&y5, &y9, &y13};
    for (auto* y : ys)
        if (y->B != x.B || y->H != x.H || y->W != x.W || y->C != x.C || y->dtype != x.dtype || y->layout != YRE_NHWC)
            YRE_FAIL(YRE_EINVAL, "spp: output views must match the input");
    if (x.layout != YRE_NHWC) YRE_FAIL(YRE_EUNSUPPORTED, "spp: NHWC only");
    // bf16 / fp16: plane-resident kernel on 16-byte words, 64 (or 32) channels per CTA when the two 16-bit planes fit in
    // shared memory
    if (x.dtype == YRE_BF16 || x.dtype == YRE_F16) {
        int chk = 0;
        for (int c : {64, 32, 16, 8})        // 20x20 planes: 64 channels per CTA; 40x40 (1280x1280 input): 16
            if (x.C % c == 0 && (size_t)2 * x.H * x.W * c * 2 <= 112 * 1024) { chk = c; break; }
        if (chk) {
            const size_t smem = (size_t)2 * x.H * x.W * chk * 2;
            typedef void (*SppFn)(DView, DView, DView, DView);
            static const SppFn fns[2][4] = {
                {spp_plane16_kernel<__nv_bfloat16, 8>, spp_plane16_kernel<__nv_bfloat16, 4>, spp_plane16_kernel<__nv_bfloat16, 2>, spp_plane16_kernel<__nv_bfloat16, 1>},
                {spp_plane16_kernel<__half, 8>, spp_plane16_kernel<__half, 4>, spp_plane16_kernel<__half, 2>, spp_plane16_kernel<__half, 1>}};
            static YrePerDeviceOnce once16;
            if (int e = once16.run([]() -> int {
                    for (const auto& row : fns)
                        for (SppFn f : row) YRE_CUDA(cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, 112 * 1024));
                    return YRE_OK;
                })) return e;
            dim3 pg((unsigned)x.B, (unsigned)(x.C / chk));
            const SppFn f = fns[x.dtype == YRE_F16][chk == 64 ? 0 : chk == 32 ? 1 : chk == 16 ? 2 : 3];
            f<<<pg, 1024, smem, s>>>(make_dview(x), make_dview(y5), make_dview(y9), make_dview(y13));
            YRE_LAUNCH_CHECK("spp_plane16");
            return YRE_OK;
        }
    }
    // plane-resident kernel when a (2 x H x W x CHK) fp32 double buffer fits in shared memory
    int chk = 0;
    for (int c : {32, 16, 8})
        if (x.C % c == 0 && (size_t)2 * x.H * x.W * c * sizeof(float) <= 96 * 1024) { chk = c; break; }
    if (chk) {
        const size_t smem = (size_t)2 * x.H * x.W * chk * sizeof(float);
        static YrePerDeviceOnce once;        // the opt-in is per device
        if (int e = once.run([]() -> int {
                YRE_CUDA(cudaFuncSetAttribute(spp_plane_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
                YRE_CUDA(cudaFuncSetAttribute(spp_plane_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
                YRE_CUDA(cudaFuncSetAttribute(spp_plane_kernel<__half>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
                return YRE_OK;
            })) return e;
        dim3 pg((unsigned)x.B, (unsigned)(x.C / chk));
        if (x.dtype == YRE_F32) spp_plane_kernel<float><<<pg, 256, smem, s>>>(make_dview(x), make_dview(y5), make_dview(y9), make_dview(y13), chk);
        else if (x.dtype == YRE_F16) spp_plane_kernel<__half><<<pg, 256, smem, s>>>(make_dview(x), make_dview(y5), make_dview(y9), make_dview(y13), chk);
        else spp_plane_kernel<__nv_bfloat16><<<pg, 256, smem, s>>>(make_dview(x), make_dview(y5), make_dview(y9), make_dview(y13), chk);
        YRE_LAUNCH_CHECK("spp_plane");
        return YRE_OK;
    }
    const long long total = (long long)x.B * x.H * x.W * (x.C / 8);
    dim3 grid(yre_cdiv(total, 256));
    if (x.dtype == YRE_F32) spp_kernel<float><<<grid, 256, 0, s>>>(make_dview(x), make_dview(y5), make_dview(y9), make_dview(y13));
    else if (x.dtype == YRE_F16) spp_kernel<__half><<<grid, 256, 0, s>>>(make_dview(x), make_dview(y5), make_dview(y9), make_dview(y13));
    else spp_kernel<__nv_bfloat16><<<grid, 256, 0, s>>>(make_dview(x), make_dview(y5), make_dview(y9), make_dview(y13));
    YRE_LAUNCH_CHECK("spp_maxpool");
    return YRE_OK;
}

int launch_upsample2x(const yre_view& x, const yre_view& y, cudaStream_t s) {
    if (check8(x, "upsample.x") || check8(y, "upsample.y")) return YRE_EINVAL;
    if (y.B != x.B || y.H != 2 * x.H || y.W != 2 * x.W || y.C != x.C || y.dtype != x.dtype)
        YRE_FAIL(YRE_EINVAL, "upsample2x: output must be 2x the input");
    const long long total = (long long)x.B * x.H * x.W * (x.C / 8);
    dim3 grid(yre_cdiv(total, 256));
    if (x.dtype == YRE_F32) upsample2x_kernel<float><<<grid, 256, 0, s>>>(make_dview(x), make_dview(y));
    else if (x.dtype == YRE_F16) upsample2x_kernel<__half><<<grid, 256, 0, s>>>(make_dview(x), make_dview(y));
    else upsample2x_kernel<__nv_bfloat16><<<grid, 256, 0, s>>>(make_dview(x), make_dview(y));
    YRE_LAUNCH_CHECK("upsample2x");
    return YRE_OK;
}

int launch_cbfuse_sum(const yre_view* srcs, int n, const yre_view& tgt, const yre_view& y, cudaStream_t s) {
    if (n < 0 || n > 8) YRE_FAIL(YRE_EUNSUPPORTED, "cbfuse: %d sources (max 8)", n);
    if (check8(tgt, "cbfuse.target") || check8(y, "cbfuse.y")) return YRE_EINVAL;
    FuseSrcs fs; fs.n = n;
    for (int i = 0; i < n; ++i) {
        if (check8(srcs[i], "cbfuse.src")) return YRE_EINVAL;
        if (srcs[i].C != y.C || srcs[i].B != y.B || srcs[i].dtype != y.dtype) YRE_FAIL(YRE_EINVAL, "cbfuse: source %d shape/dtype mismatch", i);
        fs.v[i] = make_dview(srcs[i]);
    }
    if (tgt.B != y.B || tgt.H != y.H || tgt.W != y.W || tgt.C != y.C || tgt.dtype != y.dtype) YRE_FAIL(YRE_EINVAL, "cbfuse: target mismatch");
    const long long total = (long long)y.B * y.H * y.W * (y.C / 8);
    dim3 grid(yre_cdiv(total, 256));
    if (y.dtype == YRE_F32) cbfuse_kernel<float><<<grid, 256, 0, s>>>(fs, make_dview(tgt), make_dview(y));
    else if (y.dtype == YRE_F16) cbfuse_kernel<__half><<<grid, 256, 0, s>>>(fs, make_dview(tgt), make_dview(y));
    else cbfuse_kernel<__nv_bfloat16><<<grid, 256, 0, s>>>(fs, make_dview(tgt), make_dview(y));
    YRE_LAUNCH_CHECK("cbfuse_sum");
    return YRE_OK;
}

int launch_nchw_to_view(const float* x, const yre_view& y, cudaStream_t s) {
    if (!x) YRE_FAIL(YRE_EINVAL, "nchw_to_view: null input");
    if (yre_check_view(&y, "nchw_to_view.y")) return YRE_EINVAL;
    dim3 grid(yre_cdiv((long long)y.H * y.W, 32), yre_cdiv(y.C, 32), y.B);
    if (y.dtype == YRE_F32) nchw_to_view_kernel<float><<<grid, 256, 0, s>>>(x, make_dview(y));
    else if (y.dtype == YRE_F16) nchw_to_view_kernel<__half><<<grid, 256, 0, s>>>(x, make_dview(y));
    else nchw_to_view_kernel<__nv_bfloat16><<<grid, 256, 0, s>>>(x, make_dview(y));
    YRE_LAUNCH_CHECK("nchw_to_view");
    return YRE_OK;
}

int launch_view_to_nchw(const yre_view& x, float* y, cudaStream_t s) {
    if (!y) YRE_FAIL(YRE_EINVAL, "view_to_nchw: null output");
    if (yre_check_view(&x, "view_to_nchw.x")) return YRE_EINVAL;
    dim3 grid(yre_cdiv((long long)x.H * x.W, 32), yre_cdiv(x.C, 32), x.B);
    if (x.dtype == YRE_F32) view_to_nchw_kernel<float><<<grid, 256, 0, s>>>(make_dview(x), y);
    else if (x.dtype == YRE_F16) view_to_nchw_kernel<__half><<<grid, 256, 0, s>>>(make_dview(x), y);
    else view_to_nchw_kernel<__nv_bfloat16><<<grid, 256, 0, s>>>(make_dview(x), y);
    YRE_LAUNCH_CHECK("view_to_nchw");
    return YRE_OK;
}
