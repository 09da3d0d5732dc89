// K2: first convolution, straight from the fp32 NCHW image (Cin <= 4, 3x3, pad 1, stride 1|2).
//
//   y = act(conv(x, w) + bias)          -- reference: layers.stem1, src/yolo/blocks/conv.py:88-89
//
// HBM-bound by nature (AI ~ 23 FLOP/B); output is written channels-last, optionally as the 4 parity planes the
// stride-2 tcgen05 conv that follows wants.  Three kernels:
//   stem_kernel           fp32 FMA (validation mode, any Cin <= 4 / Cout): one thread owns 4 consecutive output pixels,
//                         keeps their input patch in registers and walks the output channels 16 at a time with the
//                         folded weights broadcast from shared memory.
//   stem_mma_kernel       16-bit product path (bf16 or fp16 operands, fp32 accumulation), mma.sync m16n8k16 with
//                         K = 9*Cin padded to 32 (too thin for tcgen05), scalar gather; used for stride 1 or W % 4 != 0.
//   stem_mma_s2v_kernel   the stride-2 product kernel: vectorised cp.async gather ring (see its comment).
// The mma.sync kernels take the 16-bit type T16 as a template parameter: the image and the weights are rounded to it,
// the products are exact in fp32 for both types, and the output is written in it.
#include "yre_common.cuh"
#include <algorithm>
#include <cstdlib>

namespace {

struct StemParams {
    const float* x;
    const uint8_t* xu8;  // non-null: uint8 [B][H][W][3] frames in BGR order (cv2 layout); value / 255 and BGR->RGB fused
    DView y;            // y.B is the layout (the parity-plane stride of YRE_PHASE4)
    const float* w;     // [Cout][3][3][Cin]
    const float* bias;
    int B, Cin, H, W, Ho, Wo, Cout, stride, act;     // B: the images computed (the first B of y's y.B)
};

constexpr int PX = 4;   // output pixels per thread (consecutive in x): weights are read once per 4 pixels

template <typename TOut, int CIN, int STRIDE, bool U8 = false>
__global__ void __launch_bounds__(128) stem_kernel(const StemParams p) {
    extern __shared__ __align__(16) float sw[];               // [9*CIN][Cout] + bias[Cout]
    constexpr int K = 9 * CIN;
    constexpr int NCOL = (PX - 1) * STRIDE + 3;
    for (int i = threadIdx.x; i < K * p.Cout; i += blockDim.x) {
        const int co = i / K, kk = i % K;       // global order [co][tap][ci]
        sw[kk * p.Cout + co] = p.w[i];
    }
    float* sb = sw + K * p.Cout;
    for (int i = threadIdx.x; i < p.Cout; i += blockDim.x) sb[i] = p.bias ? p.bias[i] : 0.f;
    __syncthreads();

    const int xg = (p.Wo + PX - 1) / PX;                      // pixel groups per output row
    const long long gidx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)p.B * p.Ho * xg;
    if (gidx >= total) return;
    const int ox0 = (int)(gidx % xg) * PX;
    const long long t = gidx / xg;
    const int oy = (int)(t % p.Ho), b = (int)(t / p.Ho);

    float in[3][NCOL][CIN];
#pragma unroll
    for (int dy = 0; dy < 3; ++dy) {
        const int iy = oy * STRIDE + dy - 1;
        const bool rok = iy >= 0 && iy < p.H;
#pragma unroll
        for (int cx = 0; cx < NCOL; ++cx) {
            const int ix = ox0 * STRIDE + cx - 1;
            const bool ok = rok && ix >= 0 && ix < p.W;
#pragma unroll
            for (int ci = 0; ci < CIN; ++ci) {
                if (U8)      // model channel ci (RGB) is byte 2 - ci of the BGR pixel; float(u8) / 255 as scripts/detect.py:226
                    in[dy][cx][ci] = ok ? __fdiv_rn((float)__ldg(p.xu8 + (((long long)b * p.H + iy) * p.W + ix) * 3 + (2 - ci)), 255.f) : 0.f;
                else
                    in[dy][cx][ci] = ok ? __ldg(p.x + (((long long)b * CIN + ci) * p.H + iy) * p.W + ix) : 0.f;
            }
        }
    }

    long long obase[PX];
#pragma unroll
    for (int q = 0; q < PX; ++q) obase[q] = (ox0 + q < p.Wo) ? dview_pix(p.y, b, oy, ox0 + q) : -1;

    for (int c0 = 0; c0 < p.Cout; c0 += 16) {
        float acc[PX][16];
#pragma unroll
        for (int q = 0; q < PX; ++q)
#pragma unroll
            for (int j = 0; j < 16; ++j) acc[q][j] = sb[c0 + j];
#pragma unroll
        for (int dy = 0; dy < 3; ++dy)
#pragma unroll
            for (int dx = 0; dx < 3; ++dx)
#pragma unroll
                for (int ci = 0; ci < CIN; ++ci) {
                    const float4* wr = reinterpret_cast<const float4*>(sw + ((dy * 3 + dx) * CIN + ci) * p.Cout + c0);
                    float w[16];
#pragma unroll
                    for (int g = 0; g < 4; ++g) {
                        const float4 w4 = wr[g];
                        w[g * 4] = w4.x; w[g * 4 + 1] = w4.y; w[g * 4 + 2] = w4.z; w[g * 4 + 3] = w4.w;
                    }
#pragma unroll
                    for (int q = 0; q < PX; ++q) {
                        const float v = in[dy][q * STRIDE + dx][ci];
#pragma unroll
                        for (int j = 0; j < 16; ++j) acc[q][j] = fmaf(v, w[j], acc[q][j]);
                    }
                }
#pragma unroll
        for (int q = 0; q < PX; ++q) {
            if (obase[q] < 0) continue;
            if (p.act == YRE_ACT_SILU) {
#pragma unroll
                for (int j = 0; j < 16; ++j) acc[q][j] = silu_f(acc[q][j]);
            }
            st8<TOut>(p.y.ptr, obase[q] + c0, acc[q]);
            st8<TOut>(p.y.ptr, obase[q] + c0 + 8, acc[q] + 8);
        }
    }
}

// ---- bf16 product variant: the same conv as a [pixels x 32] x [32 x 64] GEMM on mma.sync ------------
// K = 9*Cin = 27 (zero-padded to 32) is too short for tcgen05 tiles and the layer is HBM-bound, so the
// warp-level HMMA path is the right tool: a CTA stages the 3 input rows of one 64-pixel output row
// segment in shared memory (coalesced fp32 reads), each warp builds the im2col A fragments of 16 pixels
// on the fly, multiplies by the weights held in registers for the whole kernel, applies bias + SiLU and
// writes its 16 x 64 bf16 tile through shared memory as full 16-byte, pixel-contiguous stores.
constexpr int SM_PX = 16;       // output pixels per warp tile (one m16 MMA tile)

template <typename T16> __device__ __forceinline__ void mma_16816(float* c, const uint32_t* a, const uint32_t* b);
template <> __device__ __forceinline__ void mma_16816<__nv_bfloat16>(float* c, const uint32_t* a, const uint32_t* b) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}
template <> __device__ __forceinline__ void mma_16816<__half>(float* c, const uint32_t* a, const uint32_t* b) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

// Warps are independent (no block barrier): each walks its own sequence of 16-pixel row segments,
// and the global loads of segment n+1 are issued into registers before segment n is computed, so
// the HBM latency hides behind the MMA + store work of the current segment.
template <typename T16, int STRIDE>
__global__ void __launch_bounds__(128, 3) stem_mma_kernel(const StemParams p, int segs, long long total_tiles) {
    constexpr int NCOLS = SM_PX * STRIDE + 2;                    // input columns one segment needs
    constexpr int PITCH = NCOLS + 1;
    constexpr int NLD = (9 * NCOLS + 31) / 32;                   // loads per lane (Cin <= 3 -> 9 smem rows)
    __shared__ float sin_all[4][9 * PITCH];                      // per warp: [ci*3+dy][input col]
    __shared__ __align__(16) T16 sout_all[4][16][64 + 8];            // per-warp output tile, 144-byte pitch
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
    float* sin = sin_all[warp];
    T16 (*sout)[72] = sout_all[warp];
    const int K = 9 * p.Cin;                                     // <= 27
    const int nrows = 3 * p.Cin;

    // weights -> B fragments (held in registers for the whole kernel), bias
    uint32_t bfrag[2][8][2];
    float bias[8][2];
#pragma unroll
    for (int ks = 0; ks < 2; ++ks)
#pragma unroll
        for (int j = 0; j < 8; ++j)
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int n = j * 8 + g, k0 = ks * 16 + 2 * t + 8 * h;
                const float w0 = k0 < K ? p.w[n * K + k0] : 0.f, w1 = (k0 + 1) < K ? p.w[n * K + k0 + 1] : 0.f;
                bfrag[ks][j][h] = pack16x2<T16>(w0, w1);
            }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        bias[j][0] = p.bias ? p.bias[j * 8 + 2 * t] : 0.f;
        bias[j][1] = p.bias ? p.bias[j * 8 + 2 * t + 1] : 0.f;
    }
    // smem offsets of the 8 im2col columns this thread contributes (k = tap*Cin + ci)
    int aoff[2][2][2];
#pragma unroll
    for (int ks = 0; ks < 2; ++ks)
#pragma unroll
        for (int h = 0; h < 2; ++h)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int k = ks * 16 + 2 * t + 8 * h + e;
                if (k < K) {
                    const int tap = k / p.Cin, ci = k % p.Cin, dy = tap / 3, dx = tap % 3;
                    aoff[ks][h][e] = (ci * 3 + dy) * PITCH + dx;
                } else aoff[ks][h][e] = -1;
            }

    // segment cursor (seg, oy, b) advanced by the constant warp stride with carries: no div/mod in the loop
    const int wstride = (int)gridDim.x * 4;
    const int d_seg = wstride % segs, d_oy = (wstride / segs) % p.Ho, d_b = (wstride / segs) / p.Ho;
    int tile = (int)blockIdx.x * 4 + warp;
    int seg = tile % segs, oy = (tile / segs) % p.Ho, b = (tile / segs) / p.Ho;
    const int ntiles = (int)total_tiles;
    float pre[NLD];
    // per-lane constants of the gather: (row, col) of load q never change
    int ld_off[NLD];              // ci * H * W + (dy - 1) * W + col - 1
    int ld_dy[NLD], ld_col[NLD];
#pragma unroll
    for (int q = 0; q < NLD; ++q) {
        const int i = lane + 32 * q;
        const int row = i / NCOLS, col = i - row * NCOLS;
        const int ci = row / 3, dy = row - 3 * ci;
        ld_dy[q] = (row < nrows) ? dy - 1 : -100000;
        ld_col[q] = col - 1;
        ld_off[q] = ci * p.H * p.W + (dy - 1) * p.W + col - 1;
    }

    auto fetch = [&](int fb, int foy, int fseg) {                // global -> registers for one segment
        const int iy0 = foy * STRIDE, ix0 = fseg * SM_PX * STRIDE;
        const float* base = p.x + ((long long)fb * p.Cin * p.H + iy0) * p.W + ix0;
#pragma unroll
        for (int q = 0; q < NLD; ++q) {
            const int iy = iy0 + ld_dy[q], ix = ix0 + ld_col[q];
            float v = 0.f;
            if (iy >= 0 && iy < p.H && ix >= 0 && ix < p.W) v = __ldg(base + ld_off[q]);
            pre[q] = v;
        }
    };

    if (tile < ntiles) fetch(b, oy, seg);
    for (; tile < ntiles; tile += wstride) {
        const int ox0 = seg * SM_PX;
        const int cb = b, coy = oy;
        __syncwarp();                                            // previous segment's smem readers are done
#pragma unroll
        for (int q = 0; q < NLD; ++q) {
            const int i = lane + 32 * q;
            const int row = i / NCOLS, col = i - row * NCOLS;
            if (i < 9 * NCOLS) sin[row * PITCH + col] = pre[q];
        }
        __syncwarp();
        // advance the cursor and start the next segment's loads: in flight while this segment is computed
        seg += d_seg; int cy = seg >= segs; seg -= cy ? segs : 0;
        oy += d_oy + cy; cy = oy >= p.Ho; oy -= cy ? p.Ho : 0;
        b += d_b + cy;
        if (tile + wstride < ntiles) fetch(b, oy, seg);

        float acc[8][4];
#pragma unroll
        for (int j = 0; j < 8; ++j) { acc[j][0] = bias[j][0]; acc[j][1] = bias[j][1]; acc[j][2] = bias[j][0]; acc[j][3] = bias[j][1]; }
        const int m0 = g * STRIDE, m1 = m0 + 8 * STRIDE;
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) {
            uint32_t a[4];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int o0 = aoff[ks][h][0], o1 = aoff[ks][h][1];
                const float v00 = o0 >= 0 ? sin[o0 + m0] : 0.f, v01 = o1 >= 0 ? sin[o1 + m0] : 0.f;
                const float v10 = o0 >= 0 ? sin[o0 + m1] : 0.f, v11 = o1 >= 0 ? sin[o1 + m1] : 0.f;
                a[2 * h + 0] = pack16x2<T16>(v00, v01);            // row g
                a[2 * h + 1] = pack16x2<T16>(v10, v11);            // row g + 8
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) mma_16816<T16>(acc[j], a, bfrag[ks][j]);
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            if (p.act == YRE_ACT_SILU) {
#pragma unroll
                for (int q = 0; q < 4; ++q) acc[j][q] = silu_tanh(acc[j][q]);
            }
            *reinterpret_cast<uint32_t*>(&sout[g][j * 8 + 2 * t]) = pack16x2<T16>(acc[j][0], acc[j][1]);
            *reinterpret_cast<uint32_t*>(&sout[g + 8][j * 8 + 2 * t]) = pack16x2<T16>(acc[j][2], acc[j][3]);
        }
        __syncwarp();
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int i = lane + 32 * q, px = i >> 3, c16 = i & 7;
            const int ox = ox0 + px;
            if (ox < p.Wo) {
                const uint4 v = *reinterpret_cast<const uint4*>(&sout[px][c16 * 8]);
                *reinterpret_cast<uint4*>(reinterpret_cast<T16*>(p.y.ptr) + dview_pix(p.y, cb, coy, ox) + c16 * 8) = v;
            }
        }
    }
}

// Stride-2 variant with a vectorised gather (W % 4 == 0): the first version spent ~800 instructions per
// 16-pixel segment, most of them on scalar loads, bounds tests and index arithmetic, and ran at 57 % issue
// utilisation with only 12 resident warps per SM (ncu, profiles/r01_notes.md).  Here a segment's 9 input rows are
// fetched as 90 aligned float4 (columns [32 seg - 4, 32 seg + 36)), stored with 128-bit shared-memory stores, every
// per-lane offset is a kernel-lifetime constant, K padding reads a zero word instead of a predicate, the epilogue
// uses packed fp32x2 math and the output address is one base per segment plus constant per-lane offsets.  The
// copies are cp.async (zero-fill = conv padding) into a per-warp ring of NST stages, NST-1 segments ahead.
template <typename T16, int NST, int MINB>
__global__ void __launch_bounds__(128, MINB) stem_mma_s2v_kernel(const StemParams p, int segs, long long total_tiles) {
    constexpr int NC4 = 10, PITCH = 44, ZERO = 9 * PITCH, STAGE = 9 * PITCH + 4, NLD = 3;
    __shared__ __align__(16) float sin_all[4][NST * STAGE];                // per warp: ring of NST input stages
    __shared__ __align__(16) T16 sout_all[4][16][64 + 8];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
    float* sin = sin_all[warp];
    T16 (*sout)[72] = sout_all[warp];
    const int K = 9 * p.Cin, nrows = 3 * p.Cin;
    for (int i = lane; i < NST * STAGE; i += 32) sin[i] = 0.f;            // rows of absent channels and the zero words

    uint32_t bfrag[2][8][2];
    float2 bias2[8];
#pragma unroll
    for (int ks = 0; ks < 2; ++ks)
#pragma unroll
        for (int j = 0; j < 8; ++j)
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int n = j * 8 + g, k0 = ks * 16 + 2 * t + 8 * h;
                const float w0 = k0 < K ? p.w[n * K + k0] : 0.f, w1 = (k0 + 1) < K ? p.w[n * K + k0 + 1] : 0.f;
                bfrag[ks][j][h] = pack16x2<T16>(w0, w1);
            }
#pragma unroll
    for (int j = 0; j < 8; ++j)
        bias2[j] = make_float2(p.bias ? p.bias[j * 8 + 2 * t] : 0.f, p.bias ? p.bias[j * 8 + 2 * t + 1] : 0.f);
    // word (inside a stage) of im2col element (pixel m, k): row (ci*3 + dy), column 2m + dx + 3; K padding -> zero word
    int ao[2][2][2][2];
#pragma unroll
    for (int ks = 0; ks < 2; ++ks)
#pragma unroll
        for (int h = 0; h < 2; ++h)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int k = ks * 16 + 2 * t + 8 * h + e;
                if (k < K) {
                    const int tap = k / p.Cin, ci = k % p.Cin, dy = tap / 3, dx = tap % 3;
                    const int o = (ci * 3 + dy) * PITCH + dx + 3;
                    ao[ks][h][e][0] = o + 2 * g; ao[ks][h][e][1] = o + 2 * (g + 8);
                } else ao[ks][h][e][0] = ao[ks][h][e][1] = ZERO;
            }
    // gather constants of this lane's three 16-byte copies
    int g_off[NLD], g_c4[NLD], g_dy[NLD];
    uint32_t g_so[NLD];
    bool g_ok[NLD];
    const uint32_t sin_u32 = (uint32_t)__cvta_generic_to_shared(sin);
#pragma unroll
    for (int q = 0; q < NLD; ++q) {
        const int i = lane + 32 * q, row = i / NC4, c4 = i - row * NC4, ci = row / 3, dy = row - 3 * ci;
        g_ok[q] = i < 9 * NC4 && row < nrows;
        g_dy[q] = dy; g_c4[q] = c4;
        g_off[q] = ci * p.H * p.W + (dy - 1) * p.W + 4 * c4 - 4;
        g_so[q] = sin_u32 + 4u * (uint32_t)(row * PITCH + 4 * c4);
    }
    const bool ph4 = p.y.layout == YRE_PHASE4;
    const long long plane = (long long)p.y.B * p.y.Hp * p.y.Wp * p.y.C_total;
    int o_off[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int i = lane + 32 * q, px = i >> 3, c16 = i & 7;
        o_off[q] = (ph4 ? (px >> 1) : px) * p.y.C_total + c16 * 8;      // + plane for odd pixels of the parity layout
    }

    // two cursors over this warp's segments: `f*` runs NST-1 segments ahead and issues the asynchronous copies
    const int wstride = (int)gridDim.x * 4;
    const int d_seg = wstride % segs, d_oy = (wstride / segs) % p.Ho, d_b = (wstride / segs) / p.Ho;
    int tile = (int)blockIdx.x * 4 + warp;
    int seg = tile % segs, oy = (tile / segs) % p.Ho, b = (tile / segs) / p.Ho;
    int ftile = tile, fseg = seg, foy = oy, fb = b, fstage = 0, cstage = 0;
    const int ntiles = (int)total_tiles;

    auto issue = [&]() {           // cp.async the segment under the f-cursor into stage fstage (zero-fill = conv padding), advance
        if (ftile < ntiles) {
            const int iy0 = 2 * foy, ix0 = 32 * fseg;
            const float* base = p.x + ((long long)fb * p.Cin * p.H + iy0) * p.W + ix0;
#pragma unroll
            for (int q = 0; q < NLD; ++q) {
                const int x0 = ix0 - 4 + 4 * g_c4[q], iy = iy0 + g_dy[q] - 1;
                const bool in = iy >= 0 && iy < p.H && x0 >= 0 && x0 < p.W;
                if (g_ok[q]) {
                    const float* src = in ? base + g_off[q] : p.x;
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(g_so[q] + 4u * (uint32_t)(fstage * STAGE)), "l"(src), "r"(in ? 16 : 0) : "memory");
                }
            }
            fseg += d_seg; int cy = fseg >= segs; fseg -= cy ? segs : 0;
            foy += d_oy + cy; cy = foy >= p.Ho; foy -= cy ? p.Ho : 0;
            fb += d_b + cy;
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        ftile += wstride;
        if (++fstage == NST) fstage = 0;
    };

    __syncwarp();
#pragma unroll
    for (int i = 0; i < NST - 1; ++i) issue();
    for (; tile < ntiles; tile += wstride) {
        const int ox0 = seg * SM_PX, cb = b, coy = oy;
        issue();                                                  // refills the stage the previous iteration read
        asm volatile("cp.async.wait_group %0;" ::"n"(NST - 1) : "memory");
        __syncwarp();
        const float* st = sin + cstage * STAGE;
        seg += d_seg; int cy = seg >= segs; seg -= cy ? segs : 0;
        oy += d_oy + cy; cy = oy >= p.Ho; oy -= cy ? p.Ho : 0;
        b += d_b + cy;

        float acc[8][4];
#pragma unroll
        for (int j = 0; j < 8; ++j) { acc[j][0] = bias2[j].x; acc[j][1] = bias2[j].y; acc[j][2] = bias2[j].x; acc[j][3] = bias2[j].y; }
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) {
            uint32_t a[4];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                a[2 * h + 0] = pack16x2<T16>(st[ao[ks][h][0][0]], st[ao[ks][h][1][0]]);     // row g
                a[2 * h + 1] = pack16x2<T16>(st[ao[ks][h][0][1]], st[ao[ks][h][1][1]]);     // row g + 8
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) mma_16816<T16>(acc[j], a, bfrag[ks][j]);
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            float2 lo = make_float2(acc[j][0], acc[j][1]), hi = make_float2(acc[j][2], acc[j][3]);
            if (p.act == YRE_ACT_SILU) {
                const float2 hl = __fmul2_rn(lo, make_float2(0.5f, 0.5f)), hh = __fmul2_rn(hi, make_float2(0.5f, 0.5f));
                float2 tl, th;
                asm("tanh.approx.f32 %0, %1;" : "=f"(tl.x) : "f"(hl.x));
                asm("tanh.approx.f32 %0, %1;" : "=f"(tl.y) : "f"(hl.y));
                asm("tanh.approx.f32 %0, %1;" : "=f"(th.x) : "f"(hh.x));
                asm("tanh.approx.f32 %0, %1;" : "=f"(th.y) : "f"(hh.y));
                lo = __ffma2_rn(hl, tl, hl); hi = __ffma2_rn(hh, th, hh);
            }
            *reinterpret_cast<uint32_t*>(&sout[g][j * 8 + 2 * t]) = pack16x2<T16>(lo.x, lo.y);
            *reinterpret_cast<uint32_t*>(&sout[g + 8][j * 8 + 2 * t]) = pack16x2<T16>(hi.x, hi.y);
        }
        __syncwarp();                                             // sout complete; all lanes are done reading stage cstage
        const long long ybase = ph4
            ? ((((long long)((coy & 1) * 2) * p.y.B + cb) * p.y.Hp + (coy >> 1)) * p.y.Wp + (ox0 >> 1)) * p.y.C_total + p.y.c_off
            : (((long long)cb * p.y.H + coy) * p.y.W + ox0) * p.y.C_total + p.y.c_off;
        T16* yb = reinterpret_cast<T16*>(p.y.ptr) + ybase;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int i = lane + 32 * q, px = i >> 3, c16 = i & 7;
            if (ox0 + px < p.Wo)
                *reinterpret_cast<uint4*>(yb + o_off[q] + ((ph4 && (px & 1)) ? plane : 0ll)) = *reinterpret_cast<const uint4*>(&sout[px][c16 * 8]);
        }
        if (++cstage == NST) cstage = 0;
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
}


// Stride-2 product kernel fed straight from uint8 HWC BGR camera frames (W % 16 == 0, Cin == 3): what
// scripts/detect.py:223-227 does on the host -- BGR->RGB, HWC->CHW, .float() / 255 -- happens in the gather, so the fp32
// image tensor never exists (12 bytes/pixel written by K8 and read back here become 3 bytes/pixel read once).
// A segment's three input rows are three 128-byte windows [96 seg - 16, 96 seg + 112) of the frame rows: 24 aligned
// 16-byte cp.async copies per segment instead of 90 (chunks outside the row are zero-filled = conv padding, the value
// of a padded pixel being 0 after the division as well).  im2col element (pixel m, tap (dy,dx), model channel ci) is
// byte dy*128 + 6m + 3dx + (2 - ci) + 13 of the stage.  bf16(float(v) * (1/255)) equals bf16(float(v) / 255), and
// fp16(float(v) * (1/255)) equals fp16(float(v) / 255), for all 256 byte values (checked exhaustively,
// tests/test_cpu_host.py and tests/test_cpu_fp16.py), so the A fragments are bit-identical to the ones the fp32-tensor
// path builds and so is the output.  float(v) is built as (0x4B000000 | v) - 2^23: no I2F on the MUFU pipe.
template <typename T16, int NST, int MINB>
__global__ void __launch_bounds__(128, MINB) stem_mma_s2u8_kernel(const StemParams p, int segs, long long total_tiles) {
    constexpr int ROWB = 128, ZERO = 3 * ROWB, STAGE = 3 * ROWB + 16;     // bytes; the 16 bytes at ZERO stay 0 (K padding)
    __shared__ __align__(16) uint8_t sin_all[4][NST * STAGE];
    __shared__ __align__(16) T16 sout_all[4][16][64 + 8];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
    uint8_t* sin = sin_all[warp];
    T16 (*sout)[72] = sout_all[warp];
    constexpr int K = 27;
    for (int i = lane; i < NST * STAGE / 4; i += 32) reinterpret_cast<uint32_t*>(sin)[i] = 0u;

    uint32_t bfrag[2][8][2];
    float2 bias2[8];
#pragma unroll
    for (int ks = 0; ks < 2; ++ks)
#pragma unroll
        for (int j = 0; j < 8; ++j)
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int n = j * 8 + g, k0 = ks * 16 + 2 * t + 8 * h;
                const float w0 = k0 < K ? p.w[n * K + k0] : 0.f, w1 = (k0 + 1) < K ? p.w[n * K + k0 + 1] : 0.f;
                bfrag[ks][j][h] = pack16x2<T16>(w0, w1);
            }
#pragma unroll
    for (int j = 0; j < 8; ++j)
        bias2[j] = make_float2(p.bias ? p.bias[j * 8 + 2 * t] : 0.f, p.bias ? p.bias[j * 8 + 2 * t + 1] : 0.f);
    // byte (inside a stage) of im2col element (pixel m, k = tap * 3 + ci); K padding -> a zero byte
    int ao[2][2][2][2];
#pragma unroll
    for (int ks = 0; ks < 2; ++ks)
#pragma unroll
        for (int h = 0; h < 2; ++h)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int k = ks * 16 + 2 * t + 8 * h + e;
                if (k < K) {
                    const int tap = k / 3, ci = k % 3, dy = tap / 3, dx = tap % 3;
                    const int o = dy * ROWB + 3 * dx + (2 - ci) + 13;
                    ao[ks][h][e][0] = o + 6 * g; ao[ks][h][e][1] = o + 6 * (g + 8);
                } else ao[ks][h][e][0] = ao[ks][h][e][1] = ZERO;
            }
    // this lane's 16-byte copy of a segment: row dy = lane / 8, chunk lane % 8 (lanes 24..31 copy nothing)
    const bool g_ok = lane < 24;
    const int g_dy = lane >> 3, g_c16 = lane & 7;
    const long long rowb = (long long)p.W * 3;
    const uint32_t g_so = (uint32_t)__cvta_generic_to_shared(sin) + (uint32_t)(g_dy * ROWB + 16 * g_c16);
    const bool ph4 = p.y.layout == YRE_PHASE4;
    const long long plane = (long long)p.y.B * p.y.Hp * p.y.Wp * p.y.C_total;
    int o_off[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int i = lane + 32 * q, px = i >> 3, c16 = i & 7;
        o_off[q] = (ph4 ? (px >> 1) : px) * p.y.C_total + c16 * 8;
    }

    const int wstride = (int)gridDim.x * 4;
    const int d_seg = wstride % segs, d_oy = (wstride / segs) % p.Ho, d_b = (wstride / segs) / p.Ho;
    int tile = (int)blockIdx.x * 4 + warp;
    int seg = tile % segs, oy = (tile / segs) % p.Ho, b = (tile / segs) / p.Ho;
    int ftile = tile, fseg = seg, foy = oy, fb = b, fstage = 0, cstage = 0;
    const int ntiles = (int)total_tiles;

    auto issue = [&]() {
        if (ftile < ntiles) {
            const int iy = 2 * foy + g_dy - 1;
            const long long xb = 96ll * fseg - 16 + 16 * g_c16;             // first byte of the chunk inside its frame row
            const bool in = iy >= 0 && iy < p.H && xb >= 0 && xb < rowb;     // rowb % 16 == 0: a chunk is inside or outside
            if (g_ok) {
                const uint8_t* src = in ? p.xu8 + ((long long)fb * p.H + iy) * rowb + xb : p.xu8;
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(g_so + (uint32_t)(fstage * STAGE)), "l"(src), "r"(in ? 16 : 0) : "memory");
            }
            fseg += d_seg; int cy = fseg >= segs; fseg -= cy ? segs : 0;
            foy += d_oy + cy; cy = foy >= p.Ho; foy -= cy ? p.Ho : 0;
            fb += d_b + cy;
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        ftile += wstride;
        if (++fstage == NST) fstage = 0;
    };
    // float(byte) * (1/255): (0x4B000000 | v) is the float 2^23 + v, the subtraction is exact, one rounding in the product
    auto cvt = [](uint8_t v) { return __fmul_rn(__fsub_rn(__uint_as_float(0x4B000000u | (uint32_t)v), 8388608.f), 1.0f / 255.0f); };

    __syncwarp();
#pragma unroll
    for (int i = 0; i < NST - 1; ++i) issue();
    for (; tile < ntiles; tile += wstride) {
        const int ox0 = seg * SM_PX, cb = b, coy = oy;
        issue();
        asm volatile("cp.async.wait_group %0;" ::"n"(NST - 1) : "memory");
        __syncwarp();
        const uint8_t* st = sin + cstage * STAGE;
        seg += d_seg; int cy = seg >= segs; seg -= cy ? segs : 0;
        oy += d_oy + cy; cy = oy >= p.Ho; oy -= cy ? p.Ho : 0;
        b += d_b + cy;

        float acc[8][4];
#pragma unroll
        for (int j = 0; j < 8; ++j) { acc[j][0] = bias2[j].x; acc[j][1] = bias2[j].y; acc[j][2] = bias2[j].x; acc[j][3] = bias2[j].y; }
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) {
            uint32_t a[4];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                a[2 * h + 0] = pack16x2<T16>(cvt(st[ao[ks][h][0][0]]), cvt(st[ao[ks][h][1][0]]));     // row g
                a[2 * h + 1] = pack16x2<T16>(cvt(st[ao[ks][h][0][1]]), cvt(st[ao[ks][h][1][1]]));     // row g + 8
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) mma_16816<T16>(acc[j], a, bfrag[ks][j]);
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            float2 lo = make_float2(acc[j][0], acc[j][1]), hi = make_float2(acc[j][2], acc[j][3]);
            if (p.act == YRE_ACT_SILU) {
                const float2 hl = __fmul2_rn(lo, make_float2(0.5f, 0.5f)), hh = __fmul2_rn(hi, make_float2(0.5f, 0.5f));
                float2 tl, th;
                asm("tanh.approx.f32 %0, %1;" : "=f"(tl.x) : "f"(hl.x));
                asm("tanh.approx.f32 %0, %1;" : "=f"(tl.y) : "f"(hl.y));
                asm("tanh.approx.f32 %0, %1;" : "=f"(th.x) : "f"(hh.x));
                asm("tanh.approx.f32 %0, %1;" : "=f"(th.y) : "f"(hh.y));
                lo = __ffma2_rn(hl, tl, hl); hi = __ffma2_rn(hh, th, hh);
            }
            *reinterpret_cast<uint32_t*>(&sout[g][j * 8 + 2 * t]) = pack16x2<T16>(lo.x, lo.y);
            *reinterpret_cast<uint32_t*>(&sout[g + 8][j * 8 + 2 * t]) = pack16x2<T16>(hi.x, hi.y);
        }
        __syncwarp();
        const long long ybase = ph4
            ? ((((long long)((coy & 1) * 2) * p.y.B + cb) * p.y.Hp + (coy >> 1)) * p.y.Wp + (ox0 >> 1)) * p.y.C_total + p.y.c_off
            : (((long long)cb * p.y.H + coy) * p.y.W + ox0) * p.y.C_total + p.y.c_off;
        T16* yb = reinterpret_cast<T16*>(p.y.ptr) + ybase;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int i = lane + 32 * q, px = i >> 3, c16 = i & 7;
            if (ox0 + px < p.Wo)
                *reinterpret_cast<uint4*>(yb + o_off[q] + ((ph4 && (px & 1)) ? plane : 0ll)) = *reinterpret_cast<const uint4*>(&sout[px][c16 * 8]);
        }
        if (++cstage == NST) cstage = 0;
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
}

// The stem kernels write output pixels only.  A parity-plane output of an odd extent also has cells without a source
// pixel (the last row of the planes of odd rows when Ho is odd, the last column of the planes of odd columns when Wo is
// odd), which a stride-2 conv reads at its last output row and column: they must hold zeros (include/yre.h).  One thread
// per 8 channels of a cell on the last row or column of a plane, for the first nb images (planes p * y.B + b, b < nb).
template <typename T>
__global__ void __launch_bounds__(256) phase4_zero_edges_kernel(const DView y, int nb) {
    const int groups = y.C / 8, cells = y.Hp + y.Wp;
    const long long total = 4LL * nb * cells * groups;
    const float z[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int g = (int)(i % groups);
        long long r = i / groups;
        const int cell = (int)(r % cells); r /= cells;
        const int b = (int)(r % nb), p = (int)(r / nb);
        const int py = 2 * (cell < y.Wp ? y.Hp - 1 : cell - y.Wp) + (p >> 1), px = 2 * (cell < y.Wp ? cell : y.Wp - 1) + (p & 1);
        if (py >= y.H || px >= y.W) st8<T>(y.ptr, dview_pix(y, b, py, px) + g * 8, z);
    }
}

}  // namespace

static int launch_stem_pixels(const yre_stem_desc& d, int nb, cudaStream_t s);

int launch_stem(const yre_stem_desc& d, int nb, cudaStream_t s) {
    if (int e = launch_stem_pixels(d, nb, s)) return e;
    if (d.y.layout == YRE_PHASE4 && ((d.y.H | d.y.W) & 1)) {
        const DView y = make_dview(d.y);
        const long long total = 4LL * nb * (y.Hp + y.Wp) * (y.C / 8);
        const unsigned grid = (unsigned)std::min<long long>(yre_cdiv(total, 256), 1024);
        if (d.y.dtype == YRE_F32) phase4_zero_edges_kernel<float><<<grid, 256, 0, s>>>(y, nb);
        else if (d.y.dtype == YRE_F16) phase4_zero_edges_kernel<__half><<<grid, 256, 0, s>>>(y, nb);
        else phase4_zero_edges_kernel<__nv_bfloat16><<<grid, 256, 0, s>>>(y, nb);
        YRE_LAUNCH_CHECK("stem_phase4_edges");
    }
    return YRE_OK;
}

static int launch_stem_pixels(const yre_stem_desc& d, int nb, cudaStream_t s) {
    const bool u8 = d.x_u8_hwc != nullptr;
    if ((!d.x_nchw && !u8) || !d.w) YRE_FAIL(YRE_EINVAL, "stem: null pointer");
    if (u8 && d.Cin != 3) YRE_FAIL(YRE_EUNSUPPORTED, "stem: uint8 HWC frames need Cin == 3 (got %d)", d.Cin);
    if (yre_check_view(&d.y, "stem.y")) return YRE_EINVAL;
    if (d.Cin < 1 || d.Cin > 4) YRE_FAIL(YRE_EUNSUPPORTED, "stem: Cin=%d (supported 1..4)", d.Cin);
    if (d.stride != 1 && d.stride != 2) YRE_FAIL(YRE_EUNSUPPORTED, "stem: stride %d", d.stride);
    if (d.y.C % 16 || d.y.c_off % 8 || d.y.C_total % 8) YRE_FAIL(YRE_EUNSUPPORTED, "stem: Cout must be a multiple of 16");
    const int Ho = (d.H + 2 - 3) / d.stride + 1, Wo = (d.W + 2 - 3) / d.stride + 1;
    if (Ho != d.y.H || Wo != d.y.W || d.B != d.y.B) YRE_FAIL(YRE_EINVAL, "stem: output extent mismatch");
    if (nb < 1 || nb > d.B) YRE_FAIL(YRE_EINVAL, "stem: %d images outside 1..%d", nb, d.B);
    StemParams p;
    p.x = d.x_nchw; p.xu8 = d.x_u8_hwc; p.y = make_dview(d.y); p.w = d.w; p.bias = d.bias;
    p.B = nb; p.Cin = d.Cin; p.H = d.H; p.W = d.W; p.Ho = Ho; p.Wo = Wo; p.Cout = d.y.C; p.stride = d.stride; p.act = d.act;
    const bool f16 = d.y.dtype == YRE_F16;
    if (u8 && d.y.dtype != YRE_F32 && d.y.C == 64 && d.stride == 2 && d.W % 16 == 0 &&
        (reinterpret_cast<uintptr_t>(d.y.ptr) & 15) == 0 && (reinterpret_cast<uintptr_t>(d.x_u8_hwc) & 15) == 0) {
        const int segs = yre_cdiv(Wo, SM_PX);
        const long long tiles = (long long)nb * Ho * segs;
        int dev = 0, sms = 148;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        const long long want = (tiles + 3) / 4;
        const unsigned grid = (unsigned)(want < (long long)sms * 4 ? want : (long long)sms * 4);
        if (f16) stem_mma_s2u8_kernel<__half, 3, 3><<<grid, 128, 0, s>>>(p, segs, tiles);
        else stem_mma_s2u8_kernel<__nv_bfloat16, 3, 3><<<grid, 128, 0, s>>>(p, segs, tiles);
        YRE_LAUNCH_CHECK("stem_mma_u8");
        return YRE_OK;
    }
    if (!u8 && d.y.dtype != YRE_F32 && d.Cin <= 3 && d.y.C == 64 && (reinterpret_cast<uintptr_t>(d.y.ptr) & 15) == 0) {
        const int segs = yre_cdiv(Wo, SM_PX);
        const long long tiles = (long long)nb * Ho * segs;
        int dev = 0, sms = 148;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        const long long want = (tiles + 3) / 4;
        const unsigned grid = (unsigned)(want < (long long)sms * 4 ? want : (long long)sms * 4);
        bool vec = d.stride == 2 && d.W % 4 == 0 && (reinterpret_cast<uintptr_t>(d.x_nchw) & 15) == 0;
#ifdef YRE_TUNING
        if (getenv("YRE_STEM_VEC") && atoi(getenv("YRE_STEM_VEC")) == 0) vec = false;
#endif
        // vec: 4 stages or 4 CTAs/SM (128 regs, spills) measured no better
        if (vec && f16) stem_mma_s2v_kernel<__half, 3, 3><<<grid, 128, 0, s>>>(p, segs, tiles);
        else if (vec) stem_mma_s2v_kernel<__nv_bfloat16, 3, 3><<<grid, 128, 0, s>>>(p, segs, tiles);
        else if (d.stride == 2 && f16) stem_mma_kernel<__half, 2><<<grid, 128, 0, s>>>(p, segs, tiles);
        else if (d.stride == 2) stem_mma_kernel<__nv_bfloat16, 2><<<grid, 128, 0, s>>>(p, segs, tiles);
        else if (f16) stem_mma_kernel<__half, 1><<<grid, 128, 0, s>>>(p, segs, tiles);
        else stem_mma_kernel<__nv_bfloat16, 1><<<grid, 128, 0, s>>>(p, segs, tiles);
        YRE_LAUNCH_CHECK("stem_mma");
        return YRE_OK;
    }
    const long long total = (long long)nb * Ho * ((Wo + PX - 1) / PX);
    const size_t smem = (size_t)(9 * d.Cin + 1) * d.y.C * sizeof(float);
    if (smem > 48 * 1024) YRE_FAIL(YRE_EUNSUPPORTED, "stem: Cout too large for the weight cache");
    dim3 grid(yre_cdiv(total, 128));
#define STEM_GO(T, C) do { if (d.stride == 2) stem_kernel<T, C, 2><<<grid, 128, smem, s>>>(p); else stem_kernel<T, C, 1><<<grid, 128, smem, s>>>(p); } while (0)
#define STEM_T(T) switch (d.Cin) { case 1: STEM_GO(T, 1); break; case 2: STEM_GO(T, 2); break; case 3: STEM_GO(T, 3); break; default: STEM_GO(T, 4); }
#define STEM_U8(T) do { if (d.stride == 2) stem_kernel<T, 3, 2, true><<<grid, 128, smem, s>>>(p); else stem_kernel<T, 3, 1, true><<<grid, 128, smem, s>>>(p); } while (0)
    if (u8) { if (d.y.dtype == YRE_F32) STEM_U8(float); else if (f16) STEM_U8(__half); else STEM_U8(__nv_bfloat16); }
    else if (d.y.dtype == YRE_F32) { STEM_T(float) } else if (f16) { STEM_T(__half) } else { STEM_T(__nv_bfloat16) }
#undef STEM_U8
#undef STEM_T
#undef STEM_GO
    YRE_LAUNCH_CHECK("stem");
    return YRE_OK;
}
