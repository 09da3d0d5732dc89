// K1 (product engine): convolutions on the 5th-gen tensor cores (tcgen05 / TMEM), operands staged by TMA, fused epilogue.
//
//   y = [res +] act(conv(x, w) + bias)      reference: src/yolo/blocks/conv.py:88-89 (+ conv.py:140-141,
//                                           bottleneck.py:49-51, heads/detect.py:52,61, auxiliary.py:61-62)
//
// GEMM view      D[M x N] = A[M x K] * W[N x K]^T,  M = output pixels, N = Cout, K = taps * Cin.
// Three kernels share the PTX wrappers, the epilogue and the host-side plan (ConvTcPlan):
//   conv_tc_kernel            generic implicit GEMM: for filter tap (dy,dx) and channel chunk kc ONE TMA box
//                             {BLOCK_K ch, tw, th, tb} shifted by the tap offset is loaded straight from the NHWC
//                             activation -- out-of-bounds coordinates are zero-filled by the TMA unit, which *is* the
//                             conv padding (no im2col buffer).  Stride-2 convs read a parity-plane (YRE_PHASE4) input,
//                             so each tap is again a unit-stride box (5-D tensor map, plane index = tap parity).
//   conv3_halo_kernel         3x3 stride-1, Cin <= 64, Cout 32/64: weights resident in shared memory, one 10x18-pixel
//                             halo box per 8x16 patch, the nine taps are descriptor shifts of that one tile.
//   conv3_halo_stream_kernel  3x3 stride-1, Cin a multiple of 64: same halo tile per 64-channel chunk, weight boxes
//                             streamed through a second ring, optionally two patches per weight box; on maps that 8x16
//                             patches do not tile, 8x8 patches of two images (TcParams::ybx).
// conv_tc_kernel<.., CTA2>: clusters of two CTAs feed one 256-row cta_group::2 MMA (each stages half of the weight tile).
// Which kernel / tile shape a layer gets is decided by conv_tc_select, a host-only function of the shapes and the SM count,
// from rules measured per layer (profiles/r02_notes.md); yre_conv_tc_describe reports its choice without a device.
// Operands land in 128B- (BLOCK_K=64) or 64B- (BLOCK_K=32) swizzled shared memory that the UMMA smem descriptors read
// directly.  Accumulators live in a ring of TMEM buffers (6x64, 4x128, 3x160 or 2x256 columns), so the epilogue of
// one tile overlaps the MMAs of the next ones.  All kernels are persistent (grid = min(work units, SMs)).
//
// Warp roles of the generic kernel (384 or 512 threads, 1 CTA / SM):
//   warps 0 / 2 : TMA producers, warps 1 / 3 : tcgen05.mma issuers (two producer-issuer pairs ping-pong over the CTA's
//   tiles when the stage ring is deep enough), warp 2 also allocates TMEM;
//   warps 4..   : epilogue, two or three groups of four warps (warp w owns TMEM lane quarter w % 4 = 32 pixels); groups
//   take tiles round-robin and/or split the 32-column chunks of a tile, each warp has its own double-buffered staging
//   tile and issues its own TMA stores -- no CTA-wide barrier in the steady state.
// Epilogue: tcgen05.ld -> +bias -> SiLU -> (+residual) -> bf16 -> 64B-swizzled shared-memory staging tile -> TMA store
// (cp.async.bulk.tensor) into the consumer's channel window (concat-slice write, ragged tile edges clipped by the TMA
// unit).  fp32 outputs (the raw head logits) take the same route through a fp32 staging tile on the one-CTA generic kernel
// (direct 16-byte stores elsewhere and for a 16-column tail).  All role loops are warp-uniform (elect.sync
// picks the issuing lane), which keeps the descriptors in uniform registers -- a lane-0 branch made ptxas wrap every
// UTCHMMA/UTMALDG in a serialising ELECT loop.  Measurements behind the design choices: profiles/r01_notes.md.
#include "yre_common.cuh"
#include <cuda.h>
#include <algorithm>
#include <cstring>
#include <cstdlib>
#include <memory>

struct ConvTcPlan;

namespace {

// threads per CTA: 4 role warps (2 x (TMA, MMA)) + 2 or 3 epilogue warpgroups (4 TMEM lane quarters each).
// 384 threads leave 168 registers per thread, 512 only 128: the third warpgroup pays off for small-N tiles only.
constexpr int NT_2WG = 384, NT_3WG = 512;
constexpr int BLOCK_M = 128;
constexpr int TMEM_COLS = 512;

struct TcParams {
    int tw, th, tb;                 // tile patch; tw*th*tb == 128
    int tiles_x, tiles_y, tiles_b, tiles_n, num_tiles;
    int Ho, Wo, B;
    int taps, kchunks, block_k, block_n, stages;
    int phase4;                     // stride-2 conv reading parity planes
    int x_coff, Cin, Cout;
    uint32_t a_bytes, b_bytes;
    uint32_t sbo16;                 // stride-byte-offset >> 4 of the smem descriptors
    uint32_t layout_type;           // 2 = SWIZZLE_128B, 4 = SWIZZLE_64B
    uint32_t idesc;                 // tcgen05 instruction descriptor
    const float* bias;
    int act;
    void* y; int y_f32; int y_ctot, y_coff;
    const void* res; int res_f32; int res_ctot, res_coff;
    int* dbg;                       // optional watchdog record (may be null)
    int tma_store;                  // 1: 16-bit (or fp32) output through the smem-staged TMA store
    int npipes;                     // 1 or 2 (producer, MMA) warp pairs
    int nthreads;                   // NT_2WG or NT_3WG
    int nacc, acc_stride;           // TMEM accumulator ring (2..6 buffers), columns per buffer
    int ngroups, tgroups, csplit;   // epilogue warpgroups = tgroups (tiles round-robin) x csplit (32-col chunks round-robin)
    int stw, sth, stb;              // the 32 pixels of one TMEM lane quarter as a (stb x sth x stw) sub-patch
    uint32_t stage_out_bytes;       // bytes of one per-warp staging buffer (32 rows x 32 ch x 2 = 2048; 4096 with stage64)
    int stage64;                    // 1: the epilogue stages and stores 64-column units (128B-swizzled tile, one TMA store per unit)
    // weight-stationary halo variant (conv3_halo_kernel)
    int halo;                       // 1: weight-stationary halo kernel, 2: halo kernel with streamed weights
    int stages_b, tps;              // halo == 2: slots of the weight ring, filter taps per slot (1 or 3)
    // halo == 2 schedules UNITS: unit P -> N tile P / upn, patches npair * (P % upn) + {0 .. npair-1} (M index, x fastest).
    // npair == 2: two patches share every weight box (two accumulators fed per box, half the weight traffic per pixel).
    int npair, upn, num_units, mtiles;
    uint32_t halo_tx;               // bytes one halo box delivers (10 x 18 pixels x BLOCK_K channels)
    // CTA-pair variant of the generic kernel (cta_group::2): a cluster of two CTAs takes UNIT u -> N tile u % tiles_n,
    // M tiles 2 * (u / tiles_n) + {0, 1} (cluster rank); each CTA stages its own 128-pixel A tile and block_n / 2 rows of
    // the weight tile, the leader issues 256 x block_n MMAs.  num_units = tiles_n * ceil(mtiles / 2).
    int cta2;
    // virtual cat([upsample2x(xu), x]) input of a 1x1 conv (yre_conv_desc::xu): the first ku_chunks K chunks come from the
    // half-resolution tensor through tmAu -- dims {C, 2, W/2, 2, (H/2) * B} with the two "2" dimensions at global stride 0,
    // so one box {block_k, 2, tw/2, 2, th/2} delivers the tw x th patch of the UPSAMPLED map in the usual row order
    int ku_chunks, xu_coff, xu_rows;      // xu_rows = H/2 (rows of one image in the merged row dimension)
    // rev: walk the M tiles from the last to the first.  The plan alternates the direction from one conv launch to the next, so a
    // layer starts with the part of its input that the previous layer wrote LAST -- the part that is still in the 126 MB L2
    int rev;
    // ybx (halo == 2 only): a tile is an 8 (x) by 8 (y) patch of TWO images (tb = 2) and its rows run (y, image, x) instead of
    // (image, y, x): the halo box {C, 10, 2, 10} of a tensor map with the batch dimension ahead of H lands as 20 pixel rows per
    // image row pair, so the sixteen 8-pixel row groups of the MMA are again one halo row (10 pixels) apart.  Tiles 40x40 maps
    // exactly (8x16 patches waste a sixth of them); tap (ky, kx) is a shift of ky * 20 + kx pixel rows.
    int ybx;
};

// ---- PTX wrappers --------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}
__device__ __forceinline__ unsigned long long gtimer() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
// Waits on an mbarrier phase.  A pipeline bug must never hang the GPU: after ~2 s the wait records
// where it was stuck and traps (the launch then fails with an error instead of spinning forever).
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, int* dbg, int code) {
    if (mbar_try(bar, parity)) return;
    unsigned long long t0 = 0;
    int spins = 0;
    while (!mbar_try(bar, parity)) {
        if (++spins == 4096) {
            spins = 0;
            const unsigned long long now = gtimer();
            if (t0 == 0) t0 = now;
            else if (now - t0 > 2000000000ull) {
                if (dbg) { dbg[0] = code; dbg[1] = (int)blockIdx.x; dbg[2] = (int)parity; }
                __threadfence_system();
                __trap();
            }
        }
    }
}

__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
                 ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void tma_load_5d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1, int c2, int c3, int c4) {
    asm volatile("cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
                 ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4) : "memory");
}
// ---- CTA pair (cta_group::2) variants: the two CTAs of a cluster feed ONE 256-row MMA.  The data lands in the issuing
// CTA's own shared memory, the transaction bytes are counted on the LEADER's (cluster rank 0) mbarrier: clearing bit 24
// of a shared-window address selects the even CTA of the pair.
constexpr uint32_t PEER_MASK = 0xFEFFFFFFu;
__device__ __forceinline__ void tma_load_2d_cg2(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar & PEER_MASK), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_load_4d_cg2(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
                 ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar & PEER_MASK), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void tma_load_5d_cg2(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1, int c2, int c3, int c4) {
    asm volatile("cp.async.bulk.tensor.5d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
                 ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar & PEER_MASK), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4) : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive on the LEADER CTA's copy of a barrier (from either CTA of the pair)
__device__ __forceinline__ void mbar_arrive_leader(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(bar & PEER_MASK) : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* tm) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tm)) : "memory");
}

__device__ __forceinline__ uint32_t elect_one() {
    uint32_t pred = 0;
    asm volatile("{\n\t.reg .b32 rx;\n\t.reg .pred px;\n\telect.sync rx|px, %1;\n\t@px mov.s32 %0, 1;\n\t}"
                 : "+r"(pred) : "r"(0xFFFFFFFFu));
    return pred;
}
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* tm, uint32_t src, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
                 ::"l"(reinterpret_cast<uint64_t>(tm)), "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// Programmatic dependent launch: `pdl_launch_dependents` lets the next kernel of the stream start its prologue
// (barrier init, TMEM alloc, tensor-map prefetch, bias copy) while this grid drains; `pdl_wait` blocks until the
// previous grid has completed and its writes are visible.  Both are no-ops for a normally launched kernel.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// descriptors are passed as (low word, shared high word): only the 14-bit start address in the low word
// changes per stage / K step, which keeps the issue loop on 32-bit arithmetic
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint32_t a_lo, uint32_t b_lo, uint32_t desc_hi, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\tsetp.ne.b32 p, %5, 0;\n\t"
        "mov.b64 da, {%1, %3};\n\tmov.b64 db, {%2, %3};\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %4, p;\n\t}"
        ::"r"(tmem_d), "r"(a_lo), "r"(b_lo), "r"(desc_hi), "r"(idesc), "r"(accumulate) : "memory");
}
// same with separate high words for A and B (different stride-byte-offsets)
__device__ __forceinline__ void umma_bf16_ab(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\tsetp.ne.b32 p, %6, 0;\n\t"
        "mov.b64 da, {%1, %2};\n\tmov.b64 db, {%3, %4};\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t}"
        ::"r"(tmem_d), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// CTA pair: one 256 x N x 16 MMA across both SMs (each supplies its 128 rows of A and its N/2 rows of B, read through the
// same shared-memory offsets in both CTAs); issued by the leader CTA only.
__device__ __forceinline__ void umma_bf16_cg2(uint32_t tmem_d, uint32_t a_lo, uint32_t b_lo, uint32_t desc_hi, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\tsetp.ne.b32 p, %5, 0;\n\t"
        "mov.b64 da, {%1, %3};\n\tmov.b64 db, {%2, %3};\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %4, p;\n\t}"
        ::"r"(tmem_d), "r"(a_lo), "r"(b_lo), "r"(desc_hi), "r"(idesc), "r"(accumulate) : "memory");
}
// completion of the pair's MMAs is signalled on the barrier at the same offset in BOTH CTAs
__device__ __forceinline__ void umma_commit_cg2(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(bar), "h"((uint16_t)3) : "memory");
}

#define TMEM_LD32(addr, v)                                                                                        \
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "                                                        \
                 "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "                        \
                 "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"        \
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), \
                   "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]),        \
                   "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]),      \
                   "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]),      \
                   "=r"(v[29]), "=r"(v[30]), "=r"(v[31])                                                           \
                 : "r"(addr) : "memory")
#define TMEM_LD16(addr, v)                                                                                        \
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 "                                                        \
                 "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"                 \
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), \
                   "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]),        \
                   "=r"(v[15])                                                                                     \
                 : "r"(addr) : "memory")
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Tile cursor: (nt, xt, yt, bt) of tile index t, advanced by a constant stride without div/mod.
struct TileCur {
    int nt, xt, yt, bt;
    int dn, dx, dy, db;      // digits of the stride
    __device__ __forceinline__ void init(const TcParams& p, int t, int stride) {
        nt = t % p.tiles_n; int m = t / p.tiles_n; xt = m % p.tiles_x; m /= p.tiles_x; yt = m % p.tiles_y; bt = m / p.tiles_y;
        dn = stride % p.tiles_n; m = stride / p.tiles_n; dx = m % p.tiles_x; m /= p.tiles_x; dy = m % p.tiles_y; db = m / p.tiles_y;
    }
    __device__ __forceinline__ void step(const TcParams& p) {
        nt += dn; int c = nt >= p.tiles_n; nt -= c ? p.tiles_n : 0;
        xt += dx + c; c = xt >= p.tiles_x; xt -= c ? p.tiles_x : 0;
        yt += dy + c; c = yt >= p.tiles_y; yt -= c ? p.tiles_y : 0;
        bt += db + c;
    }
};

// optional timeline trace (YRE_TC_TRACE=1): CTA 0 records (role, event, clock) triples
__device__ __forceinline__ void trace(int* dbg, int role, int& n, int ev) {
    if (dbg && blockIdx.x == 0 && n < 96) {
        long long c = clock64();
        int* slot = dbg + 16 + ((role * 96 + n) * 4);
        slot[0] = ev; slot[1] = (int)(c & 0xffffffffll); slot[2] = (int)(c >> 32); slot[3] = 1;
        ++n;
    }
}

// K-major shared-memory matrix descriptor (sm_100 "version 1"), start address advanced by the caller
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t sbo16, uint32_t layout_type) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFFu);        // start address
    d |= (uint64_t)1 << 16;                          // leading byte offset (unused for swizzled K-major)
    d |= (uint64_t)(sbo16 & 0x3FFFu) << 32;          // stride byte offset: 8 rows * swizzle width
    d |= (uint64_t)1 << 46;                          // descriptor version (Blackwell)
    d |= (uint64_t)(layout_type & 7u) << 61;
    return d;
}

// f[0..8) += the eight 16-bit residual values in u (bf16: a shift or a mask per value; fp16: a conversion per pair)
template <typename T16> __device__ __forceinline__ void add_res8(const uint4& u, float* f);
template <> __device__ __forceinline__ void add_res8<__nv_bfloat16>(const uint4& u, float* f) {
    f[0] += __uint_as_float(u.x << 16); f[1] += __uint_as_float(u.x & 0xffff0000u);
    f[2] += __uint_as_float(u.y << 16); f[3] += __uint_as_float(u.y & 0xffff0000u);
    f[4] += __uint_as_float(u.z << 16); f[5] += __uint_as_float(u.z & 0xffff0000u);
    f[6] += __uint_as_float(u.w << 16); f[7] += __uint_as_float(u.w & 0xffff0000u);
}
template <> __device__ __forceinline__ void add_res8<__half>(const uint4& u, float* f) {
    const float2 a = unpack_f16x2(u.x), b = unpack_f16x2(u.y), c = unpack_f16x2(u.z), d = unpack_f16x2(u.w);
    f[0] += a.x; f[1] += a.y; f[2] += b.x; f[3] += b.y; f[4] += c.x; f[5] += c.y; f[6] += d.x; f[7] += d.y;
}

// epilogue math for NC accumulator columns [n, n+NC): +bias -> SiLU -> (+residual), result in f[].
// `sbias` = shared-memory copy of the bias vector (whole Cout); packed fp32x2 ops (FADD2/FMUL2/FFMA2) halve
// the FP issue slots, SiLU costs one MUFU.TANH per element.  T16: the 16-bit activation type (bf16 or fp16) of a
// 16-bit residual.
template <int NC, typename T16>
__device__ __forceinline__ void epilogue_math(const TcParams& p, const float* sbias, const uint32_t* v, float* f, bool valid, long long pix, int n,
                                              const uint4* rpre = nullptr) {
    float2 x2[NC / 2];
#pragma unroll
    for (int i = 0; i < NC; i += 4) {
        const float4 b4 = *reinterpret_cast<const float4*>(sbias + n + i);
        x2[i / 2] = __fadd2_rn(make_float2(__uint_as_float(v[i]), __uint_as_float(v[i + 1])), make_float2(b4.x, b4.y));
        x2[i / 2 + 1] = __fadd2_rn(make_float2(__uint_as_float(v[i + 2]), __uint_as_float(v[i + 3])), make_float2(b4.z, b4.w));
    }
    if (p.act == YRE_ACT_SILU) {
#pragma unroll
        for (int i = 0; i < NC / 2; ++i) {
            const float2 h = __fmul2_rn(x2[i], make_float2(0.5f, 0.5f));
            float2 t;
            asm("tanh.approx.f32 %0, %1;" : "=f"(t.x) : "f"(h.x));
            asm("tanh.approx.f32 %0, %1;" : "=f"(t.y) : "f"(h.y));
            x2[i] = __ffma2_rn(h, t, h);
        }
    }
#pragma unroll
    for (int i = 0; i < NC / 2; ++i) { f[2 * i] = x2[i].x; f[2 * i + 1] = x2[i].y; }
    if (p.res && valid) {
        if (p.res_f32) {
            const float* r = reinterpret_cast<const float*>(p.res) + pix * p.res_ctot + p.res_coff + n;
#pragma unroll
            for (int i = 0; i < NC; i += 4) {
                const float4 r4 = *reinterpret_cast<const float4*>(r + i);
                f[i] += r4.x; f[i + 1] += r4.y; f[i + 2] += r4.z; f[i + 3] += r4.w;
            }
        } else {
            const T16* r = reinterpret_cast<const T16*>(p.res) + pix * p.res_ctot + p.res_coff + n;
#pragma unroll
            for (int i = 0; i < NC; i += 8) {
                const uint4 u = rpre ? rpre[i / 8] : *reinterpret_cast<const uint4*>(r + i);     // rpre: loaded a chunk ahead
                add_res8<T16>(u, f + i);
            }
        }
    }
}

// direct global store of NC columns (fp32 or 16-bit output)
template <int NC, typename T16>
__device__ __forceinline__ void store_direct(const TcParams& p, const float* f, long long pix, int n) {
    if (p.y_f32) {
        float* o = reinterpret_cast<float*>(p.y) + pix * p.y_ctot + p.y_coff + n;
#pragma unroll
        for (int i = 0; i < NC; i += 4) *reinterpret_cast<float4*>(o + i) = make_float4(f[i], f[i + 1], f[i + 2], f[i + 3]);
    } else {
        T16* o = reinterpret_cast<T16*>(p.y) + pix * p.y_ctot + p.y_coff + n;
#pragma unroll
        for (int i = 0; i < NC; i += 8) {
            uint4 u;
            u.x = pack16x2<T16>(f[i], f[i + 1]); u.y = pack16x2<T16>(f[i + 2], f[i + 3]);
            u.z = pack16x2<T16>(f[i + 4], f[i + 5]); u.w = pack16x2<T16>(f[i + 6], f[i + 7]);
            *reinterpret_cast<uint4*>(o + i) = u;
        }
    }
}

// 32 16-bit (T16) columns of one row into the swizzled staging tile.  `row_base` = smem address of the row,
// `c16` = first 16-byte chunk inside the row, `sw` = XOR pattern of the row (matches the TMA swizzle).
template <typename T16>
__device__ __forceinline__ void store_staged32(const float* f, uint32_t row_base, uint32_t c16, uint32_t sw) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const uint32_t a = row_base + (((c16 + q) ^ sw) << 4);
        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a),
                     "r"(pack16x2<T16>(f[q * 8 + 0], f[q * 8 + 1])), "r"(pack16x2<T16>(f[q * 8 + 2], f[q * 8 + 3])),
                     "r"(pack16x2<T16>(f[q * 8 + 4], f[q * 8 + 5])), "r"(pack16x2<T16>(f[q * 8 + 6], f[q * 8 + 7])) : "memory");
    }
}

// 32 fp32 columns of one row (128 bytes) into a SWIZZLE_128B staging tile: 16-byte chunk q lands at chunk (q ^ sw7)
__device__ __forceinline__ void store_staged32_f32(const float* f, uint32_t row_base, uint32_t sw7) {
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        const uint32_t a = row_base + ((((uint32_t)q) ^ sw7) << 4);
        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a),
                     "r"(__float_as_uint(f[q * 4 + 0])), "r"(__float_as_uint(f[q * 4 + 1])),
                     "r"(__float_as_uint(f[q * 4 + 2])), "r"(__float_as_uint(f[q * 4 + 3])) : "memory");
    }
}

// Epilogue role of one warp (warps 4..): tcgen05.ld -> +bias -> SiLU -> (+residual) -> bf16 staging -> TMA store.
// warpgroup grp = (tg, cs): tile-group tg takes local tiles tg, tg+GT, ...; inside a tile the csplit warpgroups of
// a tile-group share the 32-column chunks round-robin.  tfull0 / tempty0 = addresses of the first accumulator
// full / empty mbarrier (8 bytes apart per buffer).
// PF: prefetch the next chunk's tcgen05.ld into a second 32-register buffer (the 168-register / 384-thread kernels); the
// 512-thread kernels have 128 registers per thread and at most two chunks per tile, so they load each chunk in place.
// S64: 64-column staging units (TcParams::stage64) -- a template parameter because with both store paths in one kernel
// ptxas spilled ~350 bytes in the chunk loop (16 with one path)
// F32T: fp32 outputs (the raw head logits) leave through a 128B-swizzled fp32 staging tile + TMA store as well (generic
// one-CTA kernel only); a template parameter for the same reason as S64
// T16: the 16-bit activation type (bf16 or fp16) of 16-bit outputs and residuals; a template parameter for the same reason
template <typename T16, bool PF, bool CTA2 = false, bool S64 = false, bool F32T = false>
__device__ __forceinline__ void epilogue_role(const TcParams& p, const CUtensorMap* tmY, const float* sbias, int warp, int lane,
                                              uint32_t tmem_base, uint32_t out_base, uint32_t tfull0, uint32_t tempty0) {
        // ================= epilogue (warp-local, no CTA barrier) =================
        // warpgroup grp = (tg, cs): tile-group tg takes local tiles tg, tg+GT, ...; inside a tile the csplit
        // warpgroups of a tile-group share the 32-column chunks round-robin (cs, cs+CS, ...).
        const int q = warp & 3;                 // TMEM lane quarter -> rows 32q .. 32q+31 of the tile
        const int grp = (warp - 4) >> 2;
        const uint32_t G = (uint32_t)p.tgroups, NACC = (uint32_t)p.nacc;
        const int tg = grp % p.tgroups, cs = grp / p.tgroups, CS = p.csplit;
        const int row = q * 32 + lane;
        const int patch = p.tw * p.th;
        const int rem = row % patch;
        const int bi = p.ybx ? (row / p.tw) % p.tb : row / patch, yy = p.ybx ? row / (p.tw * p.tb) : rem / p.tw, xx = p.ybx ? row % p.tw : rem % p.tw;
        // origin of this warp's 32-pixel sub-patch inside the tile (row 32q)
        const int r0 = q * 32;
        const int sb0 = p.ybx ? (r0 / p.tw) % p.tb : r0 / patch, sy0 = p.ybx ? r0 / (p.tw * p.tb) : (r0 % patch) / p.tw, sx0 = p.ybx ? r0 % p.tw : (r0 % patch) % p.tw;
        const uint32_t stg = out_base + (uint32_t)(warp - 4) * 2u * p.stage_out_bytes;
        const uint32_t sw = (uint32_t)((lane >> 1) & 3);         // SWIZZLE_64B pattern of this row
        const int nchunks = (p.block_n + 31) >> 5;
        const bool tracer = (warp == 4 && lane == 0);
        const bool tma_store = p.tma_store != 0;
        const uint32_t stage_out = p.stage_out_bytes;
        const int block_n = p.block_n, y_coff = p.y_coff;
        uint32_t acc = (uint32_t)tg % NACC, acc_phase = ((uint32_t)tg / NACC) & 1u, obuf = 0;
        int tn = 0;
        TileCur tc;
        tc.init(p, blockIdx.x + tg * (int)gridDim.x, (int)(G * gridDim.x));
        const bool units = p.halo == 2;          // unit schedule of conv3_halo_stream_kernel (see TcParams)
        const int pair_rank = CTA2 ? (int)cluster_ctarank() : 0;
        for (int t = blockIdx.x + tg * (int)gridDim.x, j = tg; ; t += (int)(G * gridDim.x), j += (int)G, tc.step(p)) {
            int x0, y0, b0, n0;
            if (CTA2) {                           // CTA-pair schedule: cluster c takes units c, c + #clusters, ...
                const int u = (int)(blockIdx.x >> 1) + j * (int)(gridDim.x >> 1);
                if (u >= p.num_units) break;
                int m = 2 * (u / p.tiles_n) + pair_rank;             // m >= mtiles (odd tile out): loads zero-fill, stores clip
                if (p.rev) m = ((p.mtiles + 1) & ~1) - 1 - m;
                const int r = m / p.tiles_x;
                x0 = (m % p.tiles_x) * p.tw; y0 = (r % p.tiles_y) * p.th; b0 = (r / p.tiles_y) * p.tb; n0 = (u % p.tiles_n) * p.block_n;
            } else if (units) {
                const int P = (int)blockIdx.x + (j / p.npair) * (int)gridDim.x;
                if (P >= p.num_units) break;
                int m = p.npair * (P % p.upn) + (j % p.npair);
                if (p.rev) m = p.npair * p.upn - 1 - m;
                const int r = m / p.tiles_x;
                x0 = (m % p.tiles_x) * p.tw; y0 = (r % p.tiles_y) * p.th; b0 = (r / p.tiles_y) * p.tb; n0 = (P / p.upn) * p.block_n;
            } else {
                if (t >= p.num_tiles) break;
                const int xt = p.rev ? p.tiles_x - 1 - tc.xt : tc.xt, yt = p.rev ? p.tiles_y - 1 - tc.yt : tc.yt, bt = p.rev ? p.tiles_b - 1 - tc.bt : tc.bt;
                x0 = xt * p.tw; y0 = yt * p.th; b0 = bt * p.tb; n0 = tc.nt * p.block_n;
            }
            const int x = x0 + xx, y = y0 + yy, b = b0 + bi;
            const bool valid = (x < p.Wo) && (y < p.Ho) && (b < p.B);
            // TMA-store coordinates of this warp's 32-pixel box: {c, x, y, image}, or {c, x, image, y} for a ybx tile
            const int tc1 = x0 + sx0, tc2 = p.ybx ? b0 + sb0 : y0 + sy0, tc3 = p.ybx ? y0 + sy0 : b0 + sb0;
            const long long pix = ((long long)b * p.Ho + y) * p.Wo + x;
            const uint32_t tfull = tfull0 + 8u * acc, tempty = tempty0 + 8u * acc;
            // 16-bit residual of the chunk about to be processed: fetched before the accumulator wait / one chunk ahead,
            // so its global-memory latency hides behind the MMAs and the previous chunk's staging (it was the top stall)
            const bool res16 = p.res && !p.res_f32 && valid;
            const T16* rrow = reinterpret_cast<const T16*>(p.res) + pix * p.res_ctot + p.res_coff + n0;
            uint4 rr[4];
            const int first_col = S64 ? cs * 64 : cs * 32;         // this warpgroup's first chunk of the tile
            if (res16 && first_col + 32 <= p.block_n) {
#pragma unroll
                for (int i = 0; i < 4; ++i) rr[i] = *reinterpret_cast<const uint4*>(rrow + first_col + 8 * i);
            }
            if (tracer) trace(p.dbg, 2, tn, 20);
            mbar_wait(tfull, acc_phase, p.dbg, 4);
            tc_fence_after();
            if (tracer) trace(p.dbg, 2, tn, 21);
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * (uint32_t)p.acc_stride;
            // One full 32-column chunk: math -> (next residual) -> staging -> TMA store.  Everything the elected lane passes
            // to the TMA unit is warp-uniform, so the issue stays on the uniform datapath (no per-lane serialising loop).
            auto process32 = [&](const uint32_t* w, int col, bool more) {
                float f[32];
#ifdef YRE_TUNING
                if (tracer) trace(p.dbg, 2, tn, 23);
#endif
                epilogue_math<32, T16>(p, sbias, w, f, valid, pix, n0 + col, res16 ? rr : nullptr);
#ifdef YRE_TUNING
                if (tracer) trace(p.dbg, 2, tn, 24);
#endif
                if (res16 && more) {                      // this group's next full chunk of the tile
#pragma unroll
                    for (int i = 0; i < 4; ++i) rr[i] = *reinterpret_cast<const uint4*>(rrow + col + 32 * CS + 8 * i);
                }
                if (tma_store) {
                    if (elect_one()) bulk_wait_read<1>();       // the store that used this buffer two chunks ago has read it
                    __syncwarp();
#ifdef YRE_TUNING
                    if (tracer) trace(p.dbg, 2, tn, 25);
#endif
                    const uint32_t buf = stg + obuf * stage_out;
                    if (F32T) store_staged32_f32(f, buf + (uint32_t)lane * 128u, (uint32_t)(lane & 7));
                    else store_staged32<T16>(f, buf + (uint32_t)lane * 64u, 0u, sw);
                    fence_async_smem();
                    __syncwarp();
                    if (elect_one()) {
                        tma_store_4d(tmY, buf, y_coff + n0 + col, tc1, tc2, tc3);
                        bulk_commit();
                    }
#ifdef YRE_TUNING
                    if (tracer) trace(p.dbg, 2, tn, 26);
#endif
                    obuf ^= 1u;
                } else if (valid) {
                    store_direct<32, T16>(p, f, pix, n0 + col);
                }
            };
            auto tail16 = [&](int col) {                  // 16-column tail (block_n % 32 == 16, direct-store outputs only)
                uint32_t w16[16];
                float f[16];
                TMEM_LD16(taddr + (uint32_t)col, w16);
                tmem_ld_wait();
                epilogue_math<16, T16>(p, sbias, w16, f, valid, pix, n0 + col);
                if (valid) store_direct<16, T16>(p, f, pix, n0 + col);
            };
            auto full_at = [&](int c) { return c < nchunks && c * 32 + 32 <= block_n; };
            if (S64) {
                // 64-column units: the two 32-column chunks of a unit are staged side by side in one 128B-swizzled tile and leave
                // with ONE TMA store.  The per-store fixed costs (bulk-group wait, proxy fence, two warp syncs, store issue:
                // ~500 of the ~1100 cycles a chunk takes in the timeline traces, profiles/r02_notes.md) are paid per 64 columns.
                uint32_t va[32], vb[32];
                const int nunits = block_n >> 6;
                const uint32_t sw7 = (uint32_t)(lane & 7);                  // SWIZZLE_128B pattern of this row
                int u = cs;
                if (u < nunits) TMEM_LD32(taddr + (uint32_t)(u * 64), va);
                while (u < nunits) {
                    const int col = u * 64;
                    const bool more = u + CS < nunits;
                    float f[32];
                    tmem_ld_wait();
                    TMEM_LD32(taddr + (uint32_t)(col + 32), vb);
                    epilogue_math<32, T16>(p, sbias, va, f, valid, pix, n0 + col, res16 ? rr : nullptr);
                    if (res16) {
#pragma unroll
                        for (int i = 0; i < 4; ++i) rr[i] = *reinterpret_cast<const uint4*>(rrow + col + 32 + 8 * i);
                    }
                    if (elect_one()) bulk_wait_read<1>();                   // the store that used this buffer two units ago has read it
                    __syncwarp();
                    const uint32_t buf = stg + obuf * stage_out;
                    const uint32_t rowb = buf + (uint32_t)lane * 128u;
                    store_staged32<T16>(f, rowb, 0u, sw7);
                    tmem_ld_wait();
                    if (more) TMEM_LD32(taddr + (uint32_t)((u + CS) * 64), va);
                    epilogue_math<32, T16>(p, sbias, vb, f, valid, pix, n0 + col + 32, res16 ? rr : nullptr);
                    if (res16 && more) {
#pragma unroll
                        for (int i = 0; i < 4; ++i) rr[i] = *reinterpret_cast<const uint4*>(rrow + (u + CS) * 64 + 8 * i);
                    }
                    store_staged32<T16>(f, rowb, 4u, sw7);
                    fence_async_smem();
                    __syncwarp();
                    if (elect_one()) {
                        tma_store_4d(tmY, buf, y_coff + n0 + col, tc1, tc2, tc3);
                        bulk_commit();
                    }
                    obuf ^= 1u;
                    u += CS;
                }
            } else if (PF) {
                // two register buffers, alternately consumed and refilled: the loop is unrolled by two chunks so that no
                // buffer is ever copied (a rotating single pair cost 64 register moves per chunk)
                uint32_t va[32], vb[32];
                int c = cs;
                bool ha = full_at(c), hb = false;
                if (ha) TMEM_LD32(taddr + (uint32_t)(c * 32), va);
                while (c < nchunks) {
                    if (ha) {
                        tmem_ld_wait();
                        hb = full_at(c + CS);
                        if (hb) TMEM_LD32(taddr + (uint32_t)((c + CS) * 32), vb);
                        process32(va, c * 32, hb);
                    } else { tail16(c * 32); hb = false; }
                    c += CS;
                    if (c >= nchunks) break;
                    if (hb) {
                        tmem_ld_wait();
                        ha = full_at(c + CS);
                        if (ha) TMEM_LD32(taddr + (uint32_t)((c + CS) * 32), va);
                        process32(vb, c * 32, ha);
                    } else { tail16(c * 32); ha = false; }
                    c += CS;
                }
            } else {
                for (int c = cs; c < nchunks; c += CS) {
                    if (full_at(c)) {
                        uint32_t w[32];
                        TMEM_LD32(taddr + (uint32_t)(c * 32), w);
                        tmem_ld_wait();
                        process32(w, c * 32, full_at(c + CS));
                    } else tail16(c * 32);
                }
            }
            // every tcgen05.ld of this accumulator has completed: hand the TMEM buffer back
            tc_fence_before();
            __syncwarp();
            if (lane == 0) { if (CTA2) mbar_arrive_leader(tempty); else mbar_arrive(tempty); }    // the issuer lives in the leader CTA
            if (tracer) trace(p.dbg, 2, tn, 22);
            acc += G;
            while (acc >= NACC) { acc -= NACC; acc_phase ^= 1u; }
        }
        if (tma_store && elect_one()) bulk_wait_all();            // stores must land before the CTA retires
    }

// KSTEPS = BLOCK_K / 16: 4 (128-byte swizzle) or 2 (64-byte swizzle); NT = threads per CTA;
// CTA2: launched as clusters of two CTAs that feed one cta_group::2 MMA (see TcParams::cta2).  Per 256 x N x 16 MMA each
// SM then reads 4 KB of A + 16 N bytes of B from its shared memory instead of 4 KB + 32 N, and the TMA writes shrink
// alike -- the shared-memory port was what bounded the one-CTA kernel at N >= 128 (profiles/r01_notes.md).
template <typename T16, int KSTEPS, int NT, bool CTA2, bool S64, bool F32T>
__global__ void __launch_bounds__(NT, 1)
conv_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmY, const __grid_constant__ CUtensorMap tmAu, const TcParams p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    pdl_launch_dependents();
    if (p.dbg && threadIdx.x == 0) {       // trace mode: per-CTA entry stamp (globaltimer ns, SM clock)
        const unsigned long long g = gtimer(); const long long c = clock64();
        int* e = p.dbg + 2048 + blockIdx.x * 8;
        e[0] = (int)(g & 0xffffffffull); e[1] = (int)(g >> 32); e[2] = (int)(c & 0xffffffffll); e[3] = (int)(c >> 32);
    }
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t sbase = (raw + 1023u) & ~1023u;          // swizzle atoms need 1024-byte alignment
    // the CTA-pair variant is sized without alignment slack (it buys the sixth stage at Cout = 512): the declared
    // alignment of smem_raw must hold, otherwise fail loudly instead of running past the allocation
    if (CTA2 && (raw & 1023u)) { if (p.dbg) p.dbg[0] = 99; __trap(); }
    const uint32_t stage_bytes = p.a_bytes + p.b_bytes;
    const uint32_t S = (uint32_t)p.stages;
    const uint32_t out_base = sbase + S * stage_bytes;       // 8 warps x 2 staging buffers for the TMA-store epilogue
    const uint32_t bar_base = out_base + 8u * (uint32_t)p.ngroups * p.stage_out_bytes;   // staging: 4 warps x 2 buffers per group
    // barrier i at bar_base + 8*i : full[0..S), empty[S..2S), tmem_full[2S..2S+8), tmem_empty[2S+8..2S+16)
    const uint32_t tmem_slot = bar_base + 8u * (2u * S + 16u);
    volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - raw));
    float* sbias = reinterpret_cast<float*>(smem_raw + (tmem_slot + 16u - raw));     // [Cout] bias copy (zeros if none)
    for (int i = threadIdx.x; i < p.Cout; i += NT) sbias[i] = p.bias ? p.bias[i] : 0.f;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = CTA2 ? cluster_ctarank() : 0u;                 // 0 = leader (issues the pair's MMAs)
    // work items of this CTA (tiles) or of its cluster (units): first index and stride
    const int w0 = CTA2 ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
    const int wstride = CTA2 ? (int)(gridDim.x >> 1) : (int)gridDim.x;
    const int wtotal = CTA2 ? p.num_units : p.num_tiles;

    if (warp == 0 && lane == 0) { tma_prefetch_desc(&tmA); tma_prefetch_desc(&tmB); if (p.tma_store) tma_prefetch_desc(&tmY); if (p.ku_chunks) tma_prefetch_desc(&tmAu); }
    if (warp == 1 && lane == 0) {
        // the leader's tmem_empty barriers collect the epilogue warps of BOTH CTAs of a pair
        const uint32_t n_epi = 4u * (uint32_t)p.csplit * (CTA2 ? 2u : 1u);
        for (uint32_t i = 0; i < S; ++i) { mbar_init(bar_base + 8u * i, 1); mbar_init(bar_base + 8u * (S + i), 1); }
        for (uint32_t i = 0; i < 8; ++i) { mbar_init(bar_base + 8u * (2u * S + i), 1); mbar_init(bar_base + 8u * (2u * S + 8u + i), n_epi); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        if (CTA2) {
            asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"((uint32_t)TMEM_COLS) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
        } else {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"((uint32_t)TMEM_COLS) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        }
    }
    tc_fence_before();
    __syncthreads();
    if (CTA2) cluster_sync_all();    // the peer's barriers are initialised before anything signals them
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_ptr;
    pdl_wait();      // everything above overlapped the previous kernel's tail; activations are read below

    const int kiters = p.taps * p.kchunks;

    // Two independent (producer, MMA-issuer) warp pairs ping-pong over the CTA's tiles: pair `pipe` takes the
    // local tiles j with (j & 1) == pipe, owns half of the shared-memory stage ring and accumulator buffer
    // `pipe`.  One issuing thread needs ~600 cycles per k-iteration (mbarrier wait + descriptor math on the
    // uniform datapath + commit); two of them keep the tensor pipe and the TMA unit fed.
    const uint32_t NP = (uint32_t)p.npipes;
    const uint32_t S2 = S / NP;
    if ((warp == 0 || warp == 2) && (uint32_t)(warp >> 1) < NP) {
        // ================= TMA producer (whole warp runs the loop, one elected lane issues) =================
        const uint32_t pipe = (uint32_t)warp >> 1;
        uint32_t stage = 0, phase = 0;
        int tn = 0;
        TileCur tc;
        tc.init(p, w0 + (int)pipe * wstride, (int)NP * wstride);
        for (int t = w0 + (int)pipe * wstride; t < wtotal; t += (int)NP * wstride, tc.step(p)) {
            int x0, y0, b0, n0;
            if (CTA2) {
                int m = 2 * (t / p.tiles_n) + (int)rank;
                if (p.rev) m = ((p.mtiles + 1) & ~1) - 1 - m;
                const int r = m / p.tiles_x;
                x0 = (m % p.tiles_x) * p.tw; y0 = (r % p.tiles_y) * p.th; b0 = (r / p.tiles_y) * p.tb;
                n0 = (t % p.tiles_n) * p.block_n + (int)rank * (p.block_n >> 1);     // this CTA's half of the weight tile
            } else {
                const int xt = p.rev ? p.tiles_x - 1 - tc.xt : tc.xt, yt = p.rev ? p.tiles_y - 1 - tc.yt : tc.yt, bt = p.rev ? p.tiles_b - 1 - tc.bt : tc.bt;
                x0 = xt * p.tw; y0 = yt * p.th; b0 = bt * p.tb; n0 = tc.nt * p.block_n;
            }
            for (int tap = 0; tap < p.taps; ++tap) {
                int dx = 0, dy = 0, plane = 0;
                if (p.taps == 9) {
                    const int ky = tap / 3, kx = tap - 3 * ky;
                    if (p.phase4) {   // input row 2*oy + ky - 1  ->  parity (ky != 1), plane row oy - (ky == 0)
                        plane = ((ky != 1) << 1) | (kx != 1);
                        dy = (ky == 0) ? -1 : 0; dx = (kx == 0) ? -1 : 0;
                    } else { dy = ky - 1; dx = kx - 1; }
                }
                for (int kc = 0; kc < p.kchunks; ++kc) {
                    const uint32_t gs = pipe * S2 + stage;
                    const uint32_t full = bar_base + 8u * gs, empty = bar_base + 8u * (S + gs);
                    mbar_wait(empty, phase ^ 1u, p.dbg, 1);
                    if (pipe == 0 && lane == 0) trace(p.dbg, 0, tn, 1);
                    if (elect_one()) {
                        const uint32_t sa = sbase + gs * stage_bytes, sb = sa + p.a_bytes;
                        const bool up = kc < p.ku_chunks;          // this K chunk comes from the upsampled half-resolution source
                        const int c = up ? p.xu_coff + kc * p.block_k : p.x_coff + (kc - p.ku_chunks) * p.block_k;
                        const uint32_t img_bytes = p.a_bytes / (uint32_t)p.tb;      // one image's tw x th rows of the A tile
                        if (CTA2) {
                            // both CTAs' boxes complete on the leader's barrier, which expects the pair's bytes
                            if (rank == 0) mbar_expect_tx(full, 2u * stage_bytes);
                            if (up) {
                                for (int i = 0; i < p.tb; ++i)
                                    tma_load_5d_cg2(sa + (uint32_t)i * img_bytes, &tmAu, full, c, 0, x0 >> 1, 0, (b0 + i) * p.xu_rows + (y0 >> 1));
                            }
                            else if (p.phase4) tma_load_5d_cg2(sa, &tmA, full, c, x0 + dx, y0 + dy, b0, plane);
                            else tma_load_4d_cg2(sa, &tmA, full, c, x0 + dx, y0 + dy, b0);
                            tma_load_2d_cg2(sb, &tmB, full, tap * p.Cin + kc * p.block_k, n0);
                        } else {
                            mbar_expect_tx(full, stage_bytes);
                            if (up) {
                                for (int i = 0; i < p.tb; ++i)
                                    tma_load_5d(sa + (uint32_t)i * img_bytes, &tmAu, full, c, 0, x0 >> 1, 0, (b0 + i) * p.xu_rows + (y0 >> 1));
                            }
                            else if (p.phase4) tma_load_5d(sa, &tmA, full, c, x0 + dx, y0 + dy, b0, plane);
                            else tma_load_4d(sa, &tmA, full, c, x0 + dx, y0 + dy, b0);
                            tma_load_2d(sb, &tmB, full, tap * p.Cin + kc * p.block_k, n0);
                        }
                    }
                    __syncwarp();
                    if (pipe == 0 && lane == 0) trace(p.dbg, 0, tn, 2);
                    if (++stage == S2) { stage = 0; phase ^= 1u; }
                }
            }
        }
    } else if ((warp == 1 || warp == 3) && (uint32_t)(warp >> 1) < NP && rank == 0) {
        // ================= MMA issuer (warp-uniform loop, elected lane issues; leader CTA only) =================
        const uint32_t pipe = (uint32_t)warp >> 1;
        uint32_t stage = 0, phase = 0;
        const uint64_t desc0 = make_smem_desc(0, p.sbo16, p.layout_type);
        const uint32_t desc_hi = (uint32_t)(desc0 >> 32), desc_lo0 = (uint32_t)desc0;
        const uint32_t stage16 = stage_bytes >> 4, a16 = p.a_bytes >> 4;
        const uint32_t ring_lo = desc_lo0 + (((sbase + pipe * S2 * stage_bytes) >> 4) & 0x3FFFu);   // 14-bit start-address field (smem < 256 KB)
        int tn = 0;
        // local tile j of this CTA uses accumulator j % nacc, in phase (j / nacc) & 1
        const uint32_t NACC = (uint32_t)p.nacc;
        uint32_t acc = pipe % NACC, acc_phase = (pipe / NACC) & 1u;
        for (int t = w0 + (int)pipe * wstride; t < wtotal; t += (int)NP * wstride) {
            const uint32_t tfull = bar_base + 8u * (2u * S + acc), tempty = bar_base + 8u * (2u * S + 8u + acc);
            const uint32_t d_tmem = tmem_base + acc * (uint32_t)p.acc_stride;
            mbar_wait(tempty, acc_phase ^ 1u, p.dbg, 2);
            tc_fence_after();
            if (pipe == 0 && lane == 0) trace(p.dbg, 1, tn, 10);
            for (int it = 0; it < kiters; ++it) {
                const uint32_t gs = pipe * S2 + stage;
                const uint32_t full = bar_base + 8u * gs, empty = bar_base + 8u * (S + gs);
                mbar_wait(full, phase, p.dbg, 3);
                tc_fence_after();
                if (pipe == 0 && lane == 0) trace(p.dbg, 1, tn, 11);
                if (elect_one()) {
                    const uint32_t a_lo = ring_lo + stage * stage16, b_lo = a_lo + a16;
                    if (CTA2) {
                        umma_bf16_cg2(d_tmem, a_lo, b_lo, desc_hi, p.idesc, it > 0 ? 1u : 0u);
#pragma unroll
                        for (int k = 1; k < KSTEPS; ++k)
                            umma_bf16_cg2(d_tmem, a_lo + 2u * k, b_lo + 2u * k, desc_hi, p.idesc, 1u);
                        umma_commit_cg2(empty);                       // frees the stage in both CTAs
                        if (it == kiters - 1) umma_commit_cg2(tfull); // both CTAs' accumulator halves complete -> their epilogues
                    } else {
                        umma_bf16(d_tmem, a_lo, b_lo, desc_hi, p.idesc, it > 0 ? 1u : 0u);
#pragma unroll
                        for (int k = 1; k < KSTEPS; ++k)   // +32 bytes along K inside the swizzle atom = +2 in the >>4 address field
                            umma_bf16(d_tmem, a_lo + 2u * k, b_lo + 2u * k, desc_hi, p.idesc, 1u);
                        umma_commit(empty);                       // frees the smem stage when these MMAs retire
                        if (it == kiters - 1) umma_commit(tfull); // accumulator complete -> epilogue
                    }
                }
                __syncwarp();
                if (pipe == 0 && lane == 0) trace(p.dbg, 1, tn, 12);
                if (++stage == S2) { stage = 0; phase ^= 1u; }
            }
            acc += NP;
            while (acc >= NACC) { acc -= NACC; acc_phase ^= 1u; }
        }
    } else if (warp >= 4 && ((warp - 4) >> 2) < p.ngroups) {
        epilogue_role<T16, NT == NT_2WG, CTA2, S64, F32T>(p, &tmY, sbias, warp, lane, tmem_base, out_base, bar_base + 8u * (2u * S), bar_base + 8u * (2u * S + 8u));
    }

    tc_fence_before();
    __syncthreads();
    if (CTA2) cluster_sync_all();    // neither CTA retires (or frees TMEM) while its peer may still signal it
    if (warp == 2) {
        tc_fence_after();
        if (CTA2) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)TMEM_COLS) : "memory");
        else      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)TMEM_COLS) : "memory");
    }
    if (p.dbg && threadIdx.x == 0) {
        const unsigned long long g = gtimer(); const long long c = clock64();
        int* e = p.dbg + 2048 + blockIdx.x * 8;
        e[4] = (int)(g & 0xffffffffull); e[5] = (int)(g >> 32); e[6] = (int)(c & 0xffffffffll); e[7] = (int)(c >> 32);
    }
}


// ---- weight-stationary halo variant for small-channel 3x3 stride-1 convs -----------------------------------
// The generic kernel re-reads every input pixel nine times (one shifted box per filter tap) and synchronises
// once per tap; with Cin = Cout <= 64 a tap is only 32-128 tensor-pipe cycles of work, so those layers were
// bound by the per-k-iteration handshake and by L2->SM traffic.  Here
//   * the whole weight matrix (9 taps x Cout x Cin, <= 72 KB) is loaded ONCE per CTA and stays in shared memory;
//   * a tile is an 8 (x) by 16 (y) pixel patch of one image, and ONE TMA box of 10 x 18 pixels (the patch plus
//     its halo; out-of-bounds rows/columns zero-filled = the conv padding) is loaded per tile;
//   * tap (ky,kx) is the same shared-memory tile read through a UMMA descriptor whose start address is moved by
//     (ky*10 + kx) pixel rows and whose stride between 8-row groups is one halo row (10 pixels): the 8 rows of
//     a group are the 8 consecutive pixels of one patch row, so no data is moved or duplicated.  The swizzle
//     XOR is a function of the absolute shared-memory address on both the TMA write and the UMMA read side,
//     so a start address that is not aligned to the 1024-byte swizzle repeat needs no descriptor base offset
//     (measured: base_offset = 0 is bit-correct, a non-zero one is not);
//   * the 9 x KSTEPS MMAs of a tile are issued back to back behind a single mbarrier wait.
//   * one thread needs ~50 cycles per tcgen05.mma (descriptor moves on the uniform datapath), more than the
//     16-32 cycles such a small MMA occupies the tensor pipe, so TWO warps issue, each taking every other
//     tile; Cout is a template parameter so that every descriptor offset is an immediate.
// Warp roles: warp 0 TMA producer, warps 1 and 3 MMA issuers, warp 2 TMEM alloc, warps 4.. epilogue.
template <typename T16, int KSTEPS, int COUT>
__global__ void __launch_bounds__(NT_3WG, 1)
conv3_halo_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                  const __grid_constant__ CUtensorMap tmY, const __grid_constant__ CUtensorMap /*tmAu: generic kernel only*/, const TcParams p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    pdl_launch_dependents();
    if (p.dbg && threadIdx.x == 0) {       // trace mode: per-CTA entry stamp (globaltimer ns, SM clock)
        const unsigned long long g = gtimer(); const long long c = clock64();
        int* e = p.dbg + 2048 + blockIdx.x * 8;
        e[0] = (int)(g & 0xffffffffull); e[1] = (int)(g >> 32); e[2] = (int)(c & 0xffffffffll); e[3] = (int)(c >> 32);
    }
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t sbase = (raw + 1023u) & ~1023u;
    constexpr uint32_t ROW_BYTES = KSTEPS * 32;               // one pixel row: BLOCK_K bf16
    constexpr uint32_t A_BYTES = (180u * ROW_BYTES + 1023u) & ~1023u;    // 10 x 18 halo pixels, 1024-aligned slot
    constexpr uint32_t B_BYTES = (uint32_t)COUT * ROW_BYTES;  // one tap of the weight matrix
    const uint32_t S = (uint32_t)p.stages;                    // halo ring slots (even)
    const uint32_t sB = sbase;                                // 9 resident weight sub-tiles
    const uint32_t sA = sB + 9u * B_BYTES;                    // S halo slots
    const uint32_t out_base = sA + S * A_BYTES;
    const uint32_t bar_base = out_base + 8u * (uint32_t)p.ngroups * p.stage_out_bytes;
    // barriers: full[0..S), empty[S..2S), tmem_full[2S..2S+8), tmem_empty[2S+8..2S+16), weights at 2S+16
    const uint32_t bfull = bar_base + 8u * (2u * S + 16u);
    const uint32_t tmem_slot = bar_base + 8u * (2u * S + 18u);
    volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - raw));
    float* sbias = reinterpret_cast<float*>(smem_raw + (tmem_slot + 16u - raw));
    for (int i = threadIdx.x; i < COUT; i += NT_3WG) sbias[i] = p.bias ? p.bias[i] : 0.f;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == 0 && lane == 0) { tma_prefetch_desc(&tmA); tma_prefetch_desc(&tmB); if (p.tma_store) tma_prefetch_desc(&tmY); }
    if (warp == 1 && lane == 0) {
        for (uint32_t i = 0; i < S; ++i) { mbar_init(bar_base + 8u * i, 1); mbar_init(bar_base + 8u * (S + i), 1); }
        for (uint32_t i = 0; i < 8; ++i) { mbar_init(bar_base + 8u * (2u * S + i), 1); mbar_init(bar_base + 8u * (2u * S + 8u + i), 4u * (uint32_t)p.csplit); }
        mbar_init(bfull, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"((uint32_t)TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_ptr;
    pdl_wait();      // everything above overlapped the previous kernel's tail; activations are read below

    if (warp == 0) {
        // ================= TMA producer =================
        if (elect_one()) {
            mbar_expect_tx(bfull, 9u * B_BYTES);
            for (int tap = 0; tap < 9; ++tap) tma_load_2d(sB + (uint32_t)tap * B_BYTES, &tmB, bfull, tap * p.Cin, 0);
        }
        __syncwarp();
        uint32_t stage = 0, phase = 0;
        int tn = 0;
        TileCur tc;
        tc.init(p, blockIdx.x, (int)gridDim.x);
        for (int t = blockIdx.x; t < p.num_tiles; t += (int)gridDim.x, tc.step(p)) {
            const int x0 = (p.rev ? p.tiles_x - 1 - tc.xt : tc.xt) * p.tw, y0 = (p.rev ? p.tiles_y - 1 - tc.yt : tc.yt) * p.th;
            const int b0 = p.rev ? p.tiles_b - 1 - tc.bt : tc.bt;
            const uint32_t full = bar_base + 8u * stage, empty = bar_base + 8u * (S + stage);
            mbar_wait(empty, phase ^ 1u, p.dbg, 1);
            if (lane == 0) trace(p.dbg, 0, tn, 1);
            if (elect_one()) {
                mbar_expect_tx(full, p.halo_tx);
                tma_load_4d(sA + stage * A_BYTES, &tmA, full, p.x_coff, x0 - 1, y0 - 1, b0);
            }
            __syncwarp();
            if (lane == 0) trace(p.dbg, 0, tn, 2);
            if (++stage == S) { stage = 0; phase ^= 1u; }
        }
    } else if (warp == 1 || warp == 3) {
        // ================= MMA issuers: warp 1 takes the even local tiles, warp 3 the odd ones =================
        constexpr uint32_t ROW16 = ROW_BYTES >> 4, A16 = A_BYTES >> 4, B16 = B_BYTES >> 4;
        const uint32_t pipe = (uint32_t)warp >> 1;
        const uint64_t dA = make_smem_desc(0, 10u * ROW16, p.layout_type);      // 8-row groups one halo row apart
        const uint64_t dB = make_smem_desc(0, p.sbo16, p.layout_type);
        const uint32_t a_hi = (uint32_t)(dA >> 32), b_hi = (uint32_t)(dB >> 32);
        const uint32_t a_lo0 = (uint32_t)dA + (sA >> 4), b_lo0 = (uint32_t)dB + (sB >> 4);
        const uint32_t NACC = (uint32_t)p.nacc;
        uint32_t stage = pipe, phase = 0, acc = pipe, acc_phase = 0;          // S and NACC are even and >= 2
        int tn = 0;
        mbar_wait(bfull, 0, p.dbg, 5);
        for (int t = blockIdx.x + (int)pipe * gridDim.x; t < p.num_tiles; t += 2 * (int)gridDim.x) {
            const uint32_t tfull = bar_base + 8u * (2u * S + acc), tempty = bar_base + 8u * (2u * S + 8u + acc);
            const uint32_t full = bar_base + 8u * stage, empty = bar_base + 8u * (S + stage);
            const uint32_t d_tmem = tmem_base + acc * (uint32_t)p.acc_stride;
            mbar_wait(tempty, acc_phase ^ 1u, p.dbg, 2);
            if (pipe == 0 && lane == 0) trace(p.dbg, 1, tn, 10);
            mbar_wait(full, phase, p.dbg, 3);
            tc_fence_after();
            if (pipe == 0 && lane == 0) trace(p.dbg, 1, tn, 11);
            if (elect_one()) {
                const uint32_t a_slot = a_lo0 + stage * A16;
#pragma unroll
                for (int tap = 0; tap < 9; ++tap) {
                    const uint32_t a_lo = a_slot + (uint32_t)((tap / 3) * 10 + (tap % 3)) * ROW16;   // tap shift in pixel rows
                    const uint32_t b_lo = b_lo0 + (uint32_t)tap * B16;
#pragma unroll
                    for (int k = 0; k < KSTEPS; ++k)
                        umma_bf16_ab(d_tmem, a_lo + 2u * k, a_hi, b_lo + 2u * k, b_hi, p.idesc, (tap | k) ? 1u : 0u);
                }
                umma_commit(empty);
                umma_commit(tfull);
            }
            __syncwarp();
            if (pipe == 0 && lane == 0) trace(p.dbg, 1, tn, 12);
            stage += 2; if (stage >= S) { stage -= S; phase ^= 1u; }
            acc += 2;   if (acc >= NACC) { acc -= NACC; acc_phase ^= 1u; }
        }
    } else if (warp >= 4 && ((warp - 4) >> 2) < p.ngroups) {
        epilogue_role<T16, false>(p, &tmY, sbias, warp, lane, tmem_base, out_base, bar_base + 8u * (2u * S), bar_base + 8u * (2u * S + 8u));
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)TMEM_COLS) : "memory");
    }
    if (p.dbg && threadIdx.x == 0) {
        const unsigned long long g = gtimer(); const long long c = clock64();
        int* e = p.dbg + 2048 + blockIdx.x * 8;
        e[4] = (int)(g & 0xffffffffull); e[5] = (int)(g >> 32); e[6] = (int)(c & 0xffffffffll); e[7] = (int)(c >> 32);
    }
}

// ---- halo variant with streamed weights (3x3 stride-1, Cin a multiple of 64, any Cout tile) -------------------
// Same 8x16 patch + halo tile as above, but the weight matrix does not fit shared memory, so one {64, block_n}
// weight box per (channel chunk, tap) streams through its own ring.  Per tile and channel chunk ONE halo box
// replaces nine shifted activation boxes: the TMA write traffic into shared memory -- which shares the 128 B/clk
// port with the UMMA operand reads and bounded the generic kernel at N = 128 (8 KB read + 8 KB written per
// 64-cycle MMA) -- drops by the 4 KB of A per MMA.
// Warp roles: warp 0 halo producer, warp 2 TMEM alloc + weight producer, warp 1 MMA issuer, warps 4.. epilogue.
template <typename T16, int NT, bool S64>
__global__ void __launch_bounds__(NT, 1)
conv3_halo_stream_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                         const __grid_constant__ CUtensorMap tmY, const __grid_constant__ CUtensorMap /*tmAu: generic kernel only*/, const TcParams p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    pdl_launch_dependents();
    if (p.dbg && threadIdx.x == 0) {
        const unsigned long long g = gtimer(); const long long c = clock64();
        int* e = p.dbg + 2048 + blockIdx.x * 8;
        e[0] = (int)(g & 0xffffffffull); e[1] = (int)(g >> 32); e[2] = (int)(c & 0xffffffffll); e[3] = (int)(c >> 32);
    }
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t sbase = (raw + 1023u) & ~1023u;
    constexpr uint32_t ROW_BYTES = 128, KSTEPS = 4;
    const uint32_t A_BYTES = p.a_bytes;                       // 10 x 18 (or 10 x 2 x 10) halo pixels, 1024-aligned slot
    const uint32_t SA = (uint32_t)p.stages, SB = (uint32_t)p.stages_b;
    const uint32_t sA = sbase;
    const uint32_t NPAIR = (uint32_t)p.npair;
    const uint32_t sB = sA + SA * NPAIR * A_BYTES;
    const uint32_t out_base = sB + SB * (uint32_t)p.tps * p.b_bytes;
    const uint32_t bar_base = out_base + 8u * (uint32_t)p.ngroups * p.stage_out_bytes;
    // barriers: fullA[SA] emptyA[SA] fullB[SB] emptyB[SB] tmem_full[8] tmem_empty[8]
    const uint32_t barB = bar_base + 8u * (2u * SA);
    const uint32_t bar_t = barB + 8u * (2u * SB);
    const uint32_t tmem_slot = bar_t + 8u * 16u;
    volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - raw));
    float* sbias = reinterpret_cast<float*>(smem_raw + (tmem_slot + 16u - raw));
    for (int i = threadIdx.x; i < p.Cout; i += NT) sbias[i] = p.bias ? p.bias[i] : 0.f;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == 0 && lane == 0) { tma_prefetch_desc(&tmA); tma_prefetch_desc(&tmB); if (p.tma_store) tma_prefetch_desc(&tmY); }
    if (warp == 1 && lane == 0) {
        for (uint32_t i = 0; i < 2u * SA; ++i) mbar_init(bar_base + 8u * i, 1);
        for (uint32_t i = 0; i < 2u * SB; ++i) mbar_init(barB + 8u * i, 1);
        for (uint32_t i = 0; i < 8; ++i) { mbar_init(bar_t + 8u * i, 1); mbar_init(bar_t + 8u * (8u + i), 4u * (uint32_t)p.csplit); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"((uint32_t)TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_ptr;
    pdl_wait();      // everything above overlapped the previous kernel's tail; activations are read below

    if (warp == 0) {
        // ================= halo producer: npair boxes per (unit, channel chunk), runs ahead by SA slots =================
        uint32_t stage = 0, phase = 0;
        int tn = 0;
        for (int P = blockIdx.x; P < p.num_units; P += (int)gridDim.x) {
            const int mp = P % p.upn;
            for (int kc = 0; kc < p.kchunks; ++kc) {
                const uint32_t full = bar_base + 8u * stage, empty = bar_base + 8u * (SA + stage);
                mbar_wait(empty, phase ^ 1u, p.dbg, 1);
                if (lane == 0) trace(p.dbg, 0, tn, 1);
                if (elect_one()) {
                    mbar_expect_tx(full, NPAIR * p.halo_tx);
                    for (uint32_t h = 0; h < NPAIR; ++h) {
                        // patch h of the unit (coordinates re-derived per box: a few integer ops, no per-thread arrays)
                        int m = (int)NPAIR * mp + (int)h;
                        if (p.rev) m = (int)NPAIR * p.upn - 1 - m;
                        const int r = m / p.tiles_x;
                        const int x0 = (m % p.tiles_x) * p.tw - 1, y0 = (r % p.tiles_y) * p.th - 1;
                        const int b0 = (r / p.tiles_y) * p.tb;            // b0 >= B for the odd patch out: zero-filled
                        const uint32_t dst = sA + (stage * NPAIR + h) * A_BYTES;
                        if (p.ybx) tma_load_4d(dst, &tmA, full, p.x_coff + kc * 64, x0, b0, y0);
                        else tma_load_4d(dst, &tmA, full, p.x_coff + kc * 64, x0, y0, b0);
                    }
                }
                __syncwarp();
                if (lane == 0) trace(p.dbg, 0, tn, 2);
                if (++stage == SA) { stage = 0; phase ^= 1u; }
            }
        }
    } else if (warp == 2) {
        // ================= weight producer: tps {64, block_n} boxes (filter taps) per ring slot =================
        uint32_t stage = 0, phase = 0;
        const uint32_t slot_bytes = (uint32_t)p.tps * p.b_bytes;
        for (int P = blockIdx.x; P < p.num_units; P += (int)gridDim.x) {
            const int n0 = (P / p.upn) * p.block_n;
            for (int kc = 0; kc < p.kchunks; ++kc) {
                for (int tap = 0; tap < 9; tap += p.tps) {
                    const uint32_t full = barB + 8u * stage, empty = barB + 8u * (SB + stage);
                    mbar_wait(empty, phase ^ 1u, p.dbg, 6);
                    if (elect_one()) {
                        mbar_expect_tx(full, slot_bytes);
                        for (int i = 0; i < p.tps; ++i)
                            tma_load_2d(sB + stage * slot_bytes + (uint32_t)i * p.b_bytes, &tmB, full, (tap + i) * p.Cin + kc * 64, n0);
                    }
                    __syncwarp();
                    if (++stage == SB) { stage = 0; phase ^= 1u; }
                }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer =================
        constexpr uint32_t ROW16 = ROW_BYTES >> 4;
        const uint32_t A16 = A_BYTES >> 4;
        const uint64_t dA = make_smem_desc(0, 10u * ROW16, p.layout_type);      // 8-row groups one halo row apart
        const uint64_t dB = make_smem_desc(0, p.sbo16, p.layout_type);
        const uint32_t a_hi = (uint32_t)(dA >> 32), b_hi = (uint32_t)(dB >> 32);
        const uint32_t a_lo0 = (uint32_t)dA + (sA >> 4), b_lo0 = (uint32_t)dB + (sB >> 4);
        const uint32_t b16 = p.b_bytes >> 4;
        const uint32_t yrows = p.ybx ? 20u : 10u;                 // pixel rows between two image rows of the halo tile
        const uint32_t NACC = (uint32_t)p.nacc, TPS = (uint32_t)p.tps, astr = (uint32_t)p.acc_stride;
        uint32_t sa = 0, pha = 0, sb = 0, phb = 0, acc = 0, acc_phase = 0;
        int tn = 0;
        for (int P = blockIdx.x; P < p.num_units; P += (int)gridDim.x) {
            const uint32_t d_tmem = tmem_base + acc * astr;
            for (uint32_t h = 0; h < NPAIR; ++h) mbar_wait(bar_t + 8u * (8u + acc + h), acc_phase ^ 1u, p.dbg, 2);
            if (lane == 0) trace(p.dbg, 1, tn, 10);
            for (int kc = 0; kc < p.kchunks; ++kc) {
                mbar_wait(bar_base + 8u * sa, pha, p.dbg, 3);
                const uint32_t a_slot = a_lo0 + sa * NPAIR * A16;
                for (uint32_t tap0 = 0; tap0 < 9; tap0 += TPS) {
                    mbar_wait(barB + 8u * sb, phb, p.dbg, 7);
                    tc_fence_after();
                    if (lane == 0) trace(p.dbg, 1, tn, 11);
                    if (elect_one()) {
                        for (uint32_t i = 0; i < TPS; ++i) {
                            const uint32_t tap = tap0 + i;
                            const uint32_t shift = ((tap / 3u) * yrows + (tap % 3u)) * ROW16;    // tap shift in pixel rows
                            const uint32_t b_lo = b_lo0 + (sb * TPS + i) * b16;
                            for (uint32_t h = 0; h < NPAIR; ++h) {
                                const uint32_t a_lo = a_slot + h * A16 + shift;
#pragma unroll
                                for (uint32_t k = 0; k < KSTEPS; ++k)
                                    umma_bf16_ab(d_tmem + h * astr, a_lo + 2u * k, a_hi, b_lo + 2u * k, b_hi, p.idesc, ((uint32_t)kc | tap | k) ? 1u : 0u);
                            }
                        }
                        umma_commit(barB + 8u * (SB + sb));                      // weight slot free when these MMAs retire
                        if (tap0 + TPS == 9) {
                            umma_commit(bar_base + 8u * (SA + sa));              // halo slot free
                            if (kc == p.kchunks - 1)                             // accumulators complete -> epilogue
                                for (uint32_t h = 0; h < NPAIR; ++h) umma_commit(bar_t + 8u * (acc + h));
                        }
                    }
                    __syncwarp();
                    if (lane == 0) trace(p.dbg, 1, tn, 12);
                    if (++sb == SB) { sb = 0; phb ^= 1u; }
                }
                if (++sa == SA) { sa = 0; pha ^= 1u; }
            }
            acc += NPAIR; if (acc >= NACC) { acc -= NACC; acc_phase ^= 1u; }
        }
    } else if (warp >= 4 && ((warp - 4) >> 2) < p.ngroups) {
        epilogue_role<T16, NT == NT_2WG, false, S64>(p, &tmY, sbias, warp, lane, tmem_base, out_base, bar_t, bar_t + 64u);
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)TMEM_COLS) : "memory");
    }
    if (p.dbg && threadIdx.x == 0) {
        const unsigned long long g = gtimer(); const long long c = clock64();
        int* e = p.dbg + 2048 + blockIdx.x * 8;
        e[4] = (int)(g & 0xffffffffull); e[5] = (int)(g >> 32); e[6] = (int)(c & 0xffffffffll); e[7] = (int)(c >> 32);
    }
}

// ---- host side ---------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode() {
    static const EncodeTiledFn fn = [] {          // looked up once, thread-safe
        void* sym = nullptr;
        cudaDriverEntryPointQueryResult qres;
        const bool ok = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) == cudaSuccess &&
                        qres == cudaDriverEntryPointSuccess;
        return ok ? reinterpret_cast<EncodeTiledFn>(sym) : nullptr;
    }();
    return fn;
}

int* g_trace_buf = nullptr;

// ---- knobs ----
int env_int(const char* name, int dflt) {
#ifdef YRE_TUNING
    const char* v = getenv(name);
    return (v && *v) ? atoi(v) : dflt;
#else
    (void)name;
    return dflt;
#endif
}

struct TcKnobs {
    int pdl, sms, halo, halo_slack, halo_wide, halo_ybx, halo_pair, halo_pair64, halo_tps, prefer128, block_n, cta2, threads,
        tgroups, split, stages, pipes, stage64, direct_store, f32_tma, l2promo_a, trace;
};

// Tuning knobs (YRE_TC_*) are read only in builds made with -DYRE_TUNING (YRE_TUNING=1 python yolo-re_b200/build.py); the
// product build reads no environment variables and runs with the defaults below.  A "forced" knob left at its default
// leaves the rule in charge.  (YRE_TC_REV, the tile-walk order of a plan, is read in yre_capi.cu.)
TcKnobs tc_knobs() {
    TcKnobs k;
    k.pdl          = env_int("YRE_TC_PDL", 1);            // programmatic dependent launch
    k.sms          = env_int("YRE_TC_SMS", 0);            // > 0: persistent grids sized for that many SMs, not the device's
    k.halo         = env_int("YRE_TC_HALO", 2);           // 0: no halo kernels, 1: the weight-stationary one only, 2: both
    k.halo_slack   = env_int("YRE_TC_HALO_SLACK", 100);   // streamed halo while its tiles are <= this % of the generic tiles
    k.halo_wide    = env_int("YRE_TC_HALO_WIDE", 0);      // 1: streamed halo also where Cout tiles into 256-wide N
    k.halo_ybx     = env_int("YRE_TC_HALO_YBX", 1);       // 0: no two-image 8x8 halo tiles, 2: also for Cout % 128 == 0
    k.halo_pair    = env_int("YRE_TC_HALO_PAIR", 1);      // 0: no patch pairs on the streamed halo kernel
    k.halo_pair64  = env_int("YRE_TC_HALO_PAIR64", 1);    // 0: no patch pairs for a single 64-wide N tile
    k.halo_tps     = env_int("YRE_TC_HALO_TPS", 0);       // 1 or 3: forced filter taps per weight slot (streamed halo)
    k.prefer128    = env_int("YRE_TC_PREFER128", 1);      // 128-wide N tiles instead of the widths between 128 and 256
    k.block_n      = env_int("YRE_TC_BLOCK_N", 0);        // forced N tile width
    k.cta2         = env_int("YRE_TC_CTA2", -1);          // 0: no CTA pairs, 1: CTA pairs wherever legal
    k.threads      = env_int("YRE_TC_THREADS", 0);        // forced threads per CTA (384 or 512)
    k.tgroups      = env_int("YRE_TC_TGROUPS", 0);        // forced epilogue tile groups
    k.split        = env_int("YRE_TC_SPLIT", 0);          // forced epilogue column split
    k.stages       = env_int("YRE_TC_STAGES", 0);         // forced (shallower) operand ring
    k.pipes        = env_int("YRE_TC_PIPES", 0);          // forced (producer, MMA) pair count
    k.stage64      = env_int("YRE_TC_STAGE64", -1);       // 0: no 64-column output staging, 1: wherever legal
    k.direct_store = env_int("YRE_TC_DIRECT_STORE", 0);   // 1: bf16 outputs without the staged TMA store
    k.f32_tma      = env_int("YRE_TC_F32_TMA", 1);        // 0: fp32 outputs without the staged TMA store
    k.l2promo_a    = env_int("YRE_TC_L2PROMO_A", (int)CU_TENSOR_MAP_L2_PROMOTION_L2_128B);   // L2 promotion of activation loads
    k.trace        = env_int("YRE_TC_TRACE", 0);          // 1: per-role pipeline trace (yre_debug_read_trace)
    return k;
}

// ---- select ----
#define NOPE(msg) do { if (why && n) snprintf(why, n, "%s", msg); return 0; } while (0)
// what the kernels need of the dtypes, layouts, kernel size and channel windows -- all that conv_tc_select relies on
int tc_shape_rules(const yre_conv_desc& d, char* why, size_t n) {
    if (d.x.dtype != YRE_BF16 && d.x.dtype != YRE_F16) NOPE("input must be bf16 or fp16");
    if (d.y.layout != YRE_NHWC) NOPE("output must be NHWC");
    if (d.k != 1 && d.k != 3) NOPE("kernel must be 1x1 or 3x3");
    if (d.stride == 2 && !(d.k == 3 && d.x.layout == YRE_PHASE4)) NOPE("stride-2 needs a 3x3 kernel on a PHASE4 input");
    if (d.stride == 1 && d.x.layout != YRE_NHWC) NOPE("stride-1 needs an NHWC input");
    if (d.x.C % 32 || d.x.c_off % 8 || d.x.C_total % 8) NOPE("Cin must be a multiple of 32 (window 16-byte aligned)");
    if (d.xu.ptr) {
        if (d.k != 1 || d.stride != 1) NOPE("an upsampled source needs a 1x1 stride-1 conv");
        if (d.xu.dtype != d.x.dtype || d.xu.layout != YRE_NHWC) NOPE("upsampled source must be NHWC of x's dtype");
        if (d.xu.C % 32 || d.xu.c_off % 8 || d.xu.C_total % 8) NOPE("upsampled source: channels must be a multiple of 32 (window 16-byte aligned)");
        const int bk = ((d.x.C + d.xu.C) % 64 == 0) ? 64 : 32;
        if (d.xu.C % bk || d.x.C % bk) NOPE("upsampled source: both sources must be whole K chunks");
        if ((d.x.H & 1) || (d.x.W & 1)) NOPE("upsampled source: the map must have even extents");
    }
    if (d.y.C % 16) NOPE("Cout must be a multiple of 16");
    const int yal = d.y.dtype == YRE_F32 ? 4 : 8;
    if (d.y.c_off % yal || d.y.C_total % yal) NOPE("output window must be 16-byte aligned");
    if (d.res.ptr) {
        const int ral = d.res.dtype == YRE_F32 ? 4 : 8;
        if (d.res.layout != YRE_NHWC || d.res.c_off % ral || d.res.C_total % ral) NOPE("residual must be an aligned NHWC window");
    }
    return 1;
}

// Kernel, tiling, pipeline depth, shared memory and grid of a conv that passes tc_shape_rules on a device with `sms` SMs.
// A pure function: no CUDA call, no global state; pointers are copied into the parameters, never read.  The rules were
// measured per layer (profiles/r02_notes.md).  Fails with YRE_EUNSUPPORTED when the tile does not fit shared memory.
int conv_tc_select(const yre_conv_desc& d, int sms, const TcKnobs& kn, TcParams* out, int* grid, size_t* smem) {
    if (kn.sms > 0) sms = kn.sms;              // tuning builds: persistent grids sized for a share of the machine
    TcParams& p = *out;
    p = TcParams{};
    const int Cu = d.xu.ptr ? d.xu.C : 0;
    const int Cin = d.x.C + Cu, Cout = d.y.C, Ho = d.y.H, Wo = d.y.W, B = d.y.B;
    p.Ho = Ho; p.Wo = Wo; p.B = B; p.Cin = Cin; p.Cout = Cout; p.x_coff = d.x.c_off;
    p.taps = d.k * d.k;
    p.phase4 = d.stride == 2;
    p.block_k = (Cin % 64 == 0) ? 64 : 32;
    p.kchunks = Cin / p.block_k;
    p.ku_chunks = Cu / p.block_k; p.xu_coff = d.xu.ptr ? d.xu.c_off : 0; p.xu_rows = d.xu.ptr ? d.xu.H : 0;
    p.layout_type = p.block_k == 64 ? 2u : 4u;
    p.sbo16 = (uint32_t)(8 * p.block_k * 2) >> 4;

    // ---- M tiling: (tw, th, tb) powers of two with product 128 minimising the tile count ----
    long long best = -1; int btw = 128, bth = 1, btb = 1;
    for (int tw = 128; tw >= 1; tw >>= 1)
        for (int th = 128 / tw; th >= 1; th >>= 1) {
            const int tb = 128 / (tw * th);
            // upsampled source: a patch is a box of whole 2x2 blocks, one box per image, each a whole number of swizzle atoms
            if (Cu && (tw < 2 || th < 2 || tw * th < 8)) continue;
            const long long tiles = (long long)yre_cdiv(Wo, tw) * yre_cdiv(Ho, th) * yre_cdiv(B, tb);
            if (best < 0 || tiles < best) { best = tiles; btw = tw; bth = th; btb = tb; }
        }
    // weight-stationary halo kernel: small-channel 3x3 stride-1 convs whose 8x16 patches tile the map well
    {
        const long long htiles = (long long)yre_cdiv(Wo, 8) * yre_cdiv(Ho, 16) * B;
        p.halo = d.k == 3 && d.stride == 1 && p.kchunks == 1 && (Cout == 64 || Cout == 32) &&
                 htiles * 3 <= best * 4 && kn.halo != 0;
        // larger layers: streamed weights; worth it while the 8x16 patches waste less than the halo saves.  Not for Cout that
        // tiles into 256-wide N: there the CTA-pair generic kernel (256 x 256 MMAs, half of the weight tile per SM) is
        // 11 % faster (3x3 256->256 @80x80 B64: 370 -> 327 us, 3x3 512->512 @80x80 B16: 332 -> 296 us)
        // (measured at batch 64: +5..8% on the 80x80 maps that tile exactly, a loss on 40x40 where a sixth of the
        //  patch rows is padding -- so by default only maps without patch waste take this path)
        if (!p.halo && d.k == 3 && d.stride == 1 && p.block_k == 64 && htiles * 100 <= best * kn.halo_slack &&
            kn.halo >= 2 && (Cout % 256 != 0 || kn.halo_wide)) p.halo = 2;
        if (p.halo) { btw = 8; bth = 16; btb = 1; best = htiles; }
        // maps that 8x16 patches do not tile but 8x8 ones do (40x40): the same kernel on 8 x 8 patches of TWO images (ybx)
        const long long htiles2 = (long long)yre_cdiv(Wo, 8) * yre_cdiv(Ho, 8) * yre_cdiv(B, 2);
        // (only where two patches can share every weight box -- the unpaired halo stream loses to the CTA-pair generic kernel)
        // Measured at batch 64 on 40x40 maps: the single 64-wide N tile with a long K gains (3x3 512->64: 104 -> 81 us, the weight
        // matrix is re-streamed per patch PAIR instead of per tile), 128-wide tiles lose to the CTA-pair generic kernel
        // (3x3 128->128: 33.5 -> 40 us: 400 units are 2.7 rounds of long units) -- those need YRE_TC_HALO_YBX=2 (tuning builds)
        const bool pairable = (Cout % 128 == 0 && ((htiles2 + 1) / 2) * (Cout / 128) >= sms && kn.halo_ybx >= 2) ||
                              (Cout == 64 && p.kchunks >= 2 && (htiles2 + 1) / 2 >= sms);
        if (!p.halo && d.k == 3 && d.stride == 1 && p.block_k == 64 && B % 2 == 0 && htiles2 <= best && Cout % 256 != 0 && pairable &&
            kn.halo >= 2 && kn.halo_ybx) {
            p.halo = 2; p.ybx = 1; btw = 8; bth = 8; btb = 2; best = htiles2;
        }
    }
    p.tw = btw; p.th = bth; p.tb = btb;
    p.tiles_x = yre_cdiv(Wo, btw); p.tiles_y = yre_cdiv(Ho, bth); p.tiles_b = yre_cdiv(B, btb);
    const long long mtiles = best;

    // ---- N tiling ----
    int bn = 0;
    for (int c = 256; c >= 16; c -= 16) if (Cout % c == 0) { bn = c; break; }
    // 128-wide tiles beat the odd widths between 128 and 256 (3x3 512->640 @40x40: 5 x 128 runs in 118 us, 4 x 160 in 165 us:
    // four 128-column accumulators and CTA pairs against three unpaired 160-column ones)
    if (bn > 128 && bn < 256 && Cout % 128 == 0 && kn.prefer128) bn = 128;
    // keep the machine busy: halve N tiles while there are fewer tiles than SMs
    while (bn >= 64 && bn % 32 == 0 && mtiles * (Cout / bn) < sms) bn /= 2;
    if (kn.block_n >= 16 && kn.block_n <= 256 && kn.block_n % 16 == 0 && Cout % kn.block_n == 0) bn = kn.block_n;
    if (p.halo == 1) bn = Cout;
    p.npair = 1;
    if (p.halo == 2) {
        // two patches per weight box when a 128-wide N tile exists and there are enough pairs to fill the machine
        if (kn.halo_pair && Cout % 128 == 0 && ((mtiles + 1) / 2) * (Cout / 128) >= sms) { p.npair = 2; bn = 128; }
        // a single 64-wide N tile with a long K (head box tower, 3x3 256->64 @80x80): every patch re-streams the whole weight
        // matrix (295 KB against 92 KB of halo), so pairing halves what bounds it (L2 -> SM traffic)
        else if (kn.halo_pair >= 1 && kn.halo_pair64 && Cout == 64 && p.kchunks >= 2 && (mtiles + 1) / 2 >= sms) { p.npair = 2; bn = 64; }
    }
    p.block_n = bn;
    p.tiles_n = Cout / bn;
    p.num_tiles = (int)(mtiles * p.tiles_n);
    p.mtiles = (int)mtiles;
    p.upn = (int)((mtiles + p.npair - 1) / p.npair);
    p.num_units = p.upn * p.tiles_n;
    // CTA pairs for the wide N tiles of the generic kernel.  What they buy is operand traffic: per 128 x N x 64 k-iteration a
    // CTA pulls 16 KB of A + N * 128 B of B from L2 (and the MMAs read as much from shared memory); a pair halves the B half.
    // Rule from the per-layer sweep at batch 64 (scripts/gpu_sweep.sh, profiles/r02_notes.md): pairs win wherever the main
    // loop is at least 8 k-iterations long (K >= 512: 1x1 512->256 @80x80 134 -> 108 us, 3x3 128->128 @20x20 19 -> 13 us --
    // also for launches of a single round of units, which an earlier rule excluded), and for K = 256 when the N tile is 256
    // wide (1x1 256->256 @160x160: 308 -> 286 us); K = 128 tiles are epilogue-bound and lose 3-10 % to the cross-CTA
    // accumulator hand-off.
    const long long K_total = (long long)p.taps * Cin;
    const bool cta2_legal = !p.halo && bn >= 128 && mtiles >= 2;
    p.cta2 = kn.cta2 == 0 ? 0 : kn.cta2 == 1 ? cta2_legal : cta2_legal && (K_total >= 512 || (K_total >= 256 && bn >= 256));
    if (p.cta2) p.num_units = (int)((mtiles + 1) / 2) * p.tiles_n;
    p.a_bytes = (uint32_t)(BLOCK_M * p.block_k * 2);
    if (p.halo) {
        p.halo_tx = (uint32_t)((p.ybx ? 10 * 2 * 10 : 10 * 18) * p.block_k * 2);
        p.a_bytes = (p.halo_tx + 1023u) & ~1023u;
    }
    p.b_bytes = (uint32_t)((p.cta2 ? bn / 2 : bn) * p.block_k * 2);       // a pair's CTA stages half of the weight tile
    const uint32_t stage_bytes = p.a_bytes + p.b_bytes;
    // 16-bit outputs leave through a swizzled staging tile + TMA store; fp32 outputs (raw head logits) store directly
    p.tma_store = (d.y.dtype != YRE_F32 && bn % 32 == 0 && kn.direct_store == 0) ? 1 : 0;
    // fp32 outputs (raw head logits): the full 32-column chunks of a tile go through a fp32 staging tile + TMA store on the
    // generic one-CTA kernel (a 16-column tail, Cout = 80, still stores directly): one 4 KB bulk store instead of eight
    // 16-byte stores per lane at a 576-byte pitch
    const bool f32_tma = d.y.dtype == YRE_F32 && bn >= 32 && !p.halo && !p.cta2 && kn.f32_tma != 0;
    if (f32_tma) p.tma_store = 1;
    p.stw = p.tw < 32 ? p.tw : 32;
    p.sth = (32 / p.stw) < p.th ? (32 / p.stw) : p.th;
    p.stb = 32 / (p.stw * p.sth);
    if (p.ybx) { p.stw = 8; p.stb = 2; p.sth = 2; }          // 32 rows of a (y, image, x) tile = 2 image rows x 2 images x 8 pixels
    // TMEM accumulator ring (nacc buffers of acc_stride columns), epilogue groups and (producer, MMA) pairs.
    // Tile j of a CTA uses accumulator j % nacc, epilogue group j % ngroups and pair j % npipes.  Every
    // mbarrier is waited on by parity, so a buffer must always be served by the SAME group and the SAME pair
    // (otherwise a waiter can fall two phases behind and the parity aliases): nacc % ngroups == 0 and
    // nacc % npipes == 0.
    // With one buffer per tile-group the group idles while its buffer is refilled, so keep nacc >= 2 * tgroups;
    // where TMEM only holds 2-3 buffers, split the chunks of each tile over the warpgroups instead.
    p.nthreads = bn <= 64 ? NT_3WG : NT_2WG;
    if ((kn.threads == NT_2WG || kn.threads == NT_3WG) && p.halo != 1) p.nthreads = kn.threads;
    if (p.cta2) p.nthreads = NT_2WG;
    const int maxg = (p.nthreads / 32 - 4) / 4;
    if (bn <= 64)       { p.acc_stride = 64;  p.nacc = 6; p.tgroups = maxg; p.csplit = 1; }
    else if (bn <= 128) { p.acc_stride = 128; p.nacc = 4; p.tgroups = 2; p.csplit = 1; }
    else if (bn <= 160) { p.acc_stride = 160; p.nacc = 3; p.tgroups = 1; p.csplit = maxg; }
    else                { p.acc_stride = 256; p.nacc = 2; p.tgroups = 1; p.csplit = maxg; }
    if (kn.tgroups >= 1 && kn.tgroups <= maxg && p.nacc % kn.tgroups == 0) { p.tgroups = kn.tgroups; if (p.tgroups * p.csplit > maxg) p.csplit = 1; }
    if (kn.split >= 1 && kn.split * p.tgroups <= maxg) p.csplit = kn.split;
    if (p.npair == 2) { p.nthreads = NT_2WG; p.acc_stride = 128; p.nacc = 4; p.tgroups = 2; p.csplit = 1; }   // group h <-> patch h
    while (p.csplit > 1 && p.csplit > (bn + 31) / 32) --p.csplit;   // every warpgroup owns at least one chunk
    p.ngroups = p.tgroups * p.csplit;
    // 64-column staging for the 384-thread kernels (they run the register-prefetching epilogue): N tiles that are whole units.
    // 1x1 convs only: they are store/epilogue-bound and gain 25-35 % from the halved store count (1x1 128->128 @160x160:
    // 208 -> 135 us), while every 3x3 kernel (generic, CTA pair, halo stream) is main-loop bound and LOSES 8-25 % to the
    // 32 KB of operand ring the larger staging tiles take (3x3 256->256 @80x80: 366 -> 467 us) -- per-layer sweep, r02_notes.md
    p.stage64 = (p.tma_store && p.nthreads == NT_2WG && bn % 64 == 0 && (kn.stage64 < 0 ? p.taps == 1 : kn.stage64 != 0)) ? 1 : 0;
    if (f32_tma) p.stage64 = 0;
    p.stage_out_bytes = p.tma_store ? ((p.stage64 || f32_tma) ? 4096u : 2048u) : 0u;      // 32 rows x 32 (or 64) bf16 / 32 fp32 channels per buffer
    const uint32_t n_stage_bufs = 8u * (uint32_t)p.ngroups;         // 4 warps x 2 buffers per group
    const uint32_t align_slack = p.cta2 ? 0u : 1024u;      // the pair kernel relies on (and checks) the declared 1024-byte alignment
    const uint32_t smem_cap = 227u * 1024u - align_slack - 256u - (uint32_t)Cout * 4u;   // alignment slack + barriers + bias copy
    int stages = (int)((smem_cap - n_stage_bufs * p.stage_out_bytes) / stage_bytes);
    if (p.halo == 1) stages = (int)((smem_cap - n_stage_bufs * p.stage_out_bytes - 9u * p.b_bytes) / p.a_bytes);
    if (stages > 8) stages = 8;
    if (p.halo == 2) {
        // weight ring: three taps per slot when that still leaves >= 3 slots (fewer, longer MMA batches per
        // mbarrier wait -- a single issuing thread needs ~450 cycles per wait + 4 MMAs), else one tap per slot
        const uint32_t room = smem_cap - n_stage_bufs * p.stage_out_bytes - 256u;
        const uint32_t a_slot = (uint32_t)p.npair * p.a_bytes;
        int sa = 2;
        p.tps = ((room - 2u * a_slot) / (3u * p.b_bytes) >= (p.npair == 2 ? 2u : 3u)) ? 3 : 1;
        if (kn.halo_tps == 1 || kn.halo_tps == 3) p.tps = kn.halo_tps;
        int sb = (int)((room - 2u * a_slot) / ((uint32_t)p.tps * p.b_bytes));
        if (sb > (p.tps == 3 ? 4 : 8)) {           // room to spare: a third halo slot
            const int sb3 = (int)((room - 3u * a_slot) / ((uint32_t)p.tps * p.b_bytes));
            if (sb3 >= (p.tps == 3 ? 3 : 5)) { sa = 3; sb = sb3; }
        }
        if (sb > 8) sb = 8;
        if (sb < 2) YRE_FAIL(YRE_EUNSUPPORTED, "conv_tc: halo tile does not fit shared memory");
        stages = sa; p.stages_b = sb;
    }
    if (kn.stages >= 2 && kn.stages <= stages) stages = kn.stages;
    if (stages < 2) YRE_FAIL(YRE_EUNSUPPORTED, "conv_tc: tile does not fit shared memory");
    // two (producer, MMA) pairs when the ring gives each at least 3 stages
    p.npipes = (stages >= 6 && p.nacc % 2 == 0 && !p.halo) ? 2 : 1;
    if (kn.pipes >= 1 && kn.pipes <= 2 && p.nacc % kn.pipes == 0 && stages >= 2 * kn.pipes) p.npipes = kn.pipes;
    if (p.npipes == 2 || p.halo == 1) stages &= ~1;
    p.stages = stages;
    // operand rings (the weight-stationary halo kernel keeps all nine weight taps resident), 8-byte mbarriers, 32 bytes of
    // TMEM slot and flags, the epilogue's staging buffers, the bias copy and the alignment slack
    const size_t rings = p.halo == 2 ? (size_t)stages * p.npair * p.a_bytes + (size_t)p.stages_b * p.tps * p.b_bytes
                       : p.halo      ? (size_t)stages * p.a_bytes + 9 * (size_t)p.b_bytes
                       :               (size_t)stages * stage_bytes;
    *smem = rings + 8 * (2 * stages + 16 + (p.halo == 2 ? 2 * p.stages_b : p.halo ? 2 : 0)) + 32 + n_stage_bufs * p.stage_out_bytes +
            (size_t)Cout * 4 + align_slack;
    // persistent grids: one CTA (pair) per work unit, at most one per SM
    *grid = p.cta2 ? 2 * std::min(p.num_units, sms / 2) : std::min(p.halo == 2 ? p.num_units : p.num_tiles, sms);
    // instruction descriptor: fp32 accumulator (bits 4-5), A and B bf16 (bits 7-9, 10-12; conv_tc_prepare clears them for
    // fp16 operands -- the tiling is the same for both 16-bit types), N >> 3, M >> 4
    p.idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(bn >> 3) << 17) | ((uint32_t)((p.cta2 ? 2 * BLOCK_M : BLOCK_M) >> 4) << 24);
    p.bias = d.bias; p.act = d.act;
    p.y = d.y.ptr; p.y_f32 = d.y.dtype == YRE_F32; p.y_ctot = d.y.C_total; p.y_coff = d.y.c_off;
    p.res = d.res.ptr; p.res_f32 = d.res.ptr ? d.res.dtype == YRE_F32 : 0;
    p.res_ctot = d.res.ptr ? d.res.C_total : 0; p.res_coff = d.res.ptr ? d.res.c_off : 0;
    return YRE_OK;
}

// ---- kernel table ----
typedef void (*TcKernelFn)(CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, TcParams);

// each kernel as the pair {bf16, fp16} of its instantiations for the two 16-bit activation types
template <int KSTEPS, int NT, bool CTA2, bool S64, bool F32T = false>
const TcKernelFn conv_tc_kernels[2] = {conv_tc_kernel<__nv_bfloat16, KSTEPS, NT, CTA2, S64, F32T>,
                                       conv_tc_kernel<__half, KSTEPS, NT, CTA2, S64, F32T>};
template <int KSTEPS, int COUT>
const TcKernelFn conv3_halo_kernels[2] = {conv3_halo_kernel<__nv_bfloat16, KSTEPS, COUT>, conv3_halo_kernel<__half, KSTEPS, COUT>};
template <int NT, bool S64>
const TcKernelFn conv3_halo_stream_kernels[2] = {conv3_halo_stream_kernel<__nv_bfloat16, NT, S64>, conv3_halo_stream_kernel<__half, NT, S64>};

// Every kernel (as its {bf16, fp16} pair of instantiations) with the TcParams values that select it.  The keys are exact (cout: Cout of the
// weight-stationary halo kernel, 0 elsewhere; f32_tma: fp32 output through the staged TMA store), so no two entries match
// the same parameters and the order of the rows does not matter.
struct TcKernel {
    const TcKernelFn* fn;                                // [0]: bf16 activations, [1]: fp16
    const char* name;                                    // for launch errors
    int halo, block_k, cout, cta2, f32_tma, nthreads, stage64;
};

const TcKernel TC_KERNELS[] = {
    //                                                                        halo  bk cout cta2 f32 nthreads s64
    {conv_tc_kernels<4, NT_2WG, false, false>,        "conv_tc",               0, 64,  0,  0,  0, NT_2WG, 0},
    {conv_tc_kernels<2, NT_2WG, false, false>,        "conv_tc",               0, 32,  0,  0,  0, NT_2WG, 0},
    {conv_tc_kernels<4, NT_2WG, false, true>,         "conv_tc",               0, 64,  0,  0,  0, NT_2WG, 1},
    {conv_tc_kernels<2, NT_2WG, false, true>,         "conv_tc",               0, 32,  0,  0,  0, NT_2WG, 1},
    {conv_tc_kernels<4, NT_3WG, false, false>,        "conv_tc",               0, 64,  0,  0,  0, NT_3WG, 0},
    {conv_tc_kernels<2, NT_3WG, false, false>,        "conv_tc",               0, 32,  0,  0,  0, NT_3WG, 0},
    {conv_tc_kernels<4, NT_2WG, true, false>,         "conv_tc (CTA pair)",    0, 64,  0,  1,  0, NT_2WG, 0},
    {conv_tc_kernels<2, NT_2WG, true, false>,         "conv_tc (CTA pair)",    0, 32,  0,  1,  0, NT_2WG, 0},
    {conv_tc_kernels<4, NT_2WG, true, true>,          "conv_tc (CTA pair)",    0, 64,  0,  1,  0, NT_2WG, 1},
    {conv_tc_kernels<2, NT_2WG, true, true>,          "conv_tc (CTA pair)",    0, 32,  0,  1,  0, NT_2WG, 1},
    {conv_tc_kernels<4, NT_2WG, false, false, true>,  "conv_tc (fp32 out)",    0, 64,  0,  0,  1, NT_2WG, 0},
    {conv_tc_kernels<2, NT_2WG, false, false, true>,  "conv_tc (fp32 out)",    0, 32,  0,  0,  1, NT_2WG, 0},
    {conv_tc_kernels<4, NT_3WG, false, false, true>,  "conv_tc (fp32 out)",    0, 64,  0,  0,  1, NT_3WG, 0},
    {conv_tc_kernels<2, NT_3WG, false, false, true>,  "conv_tc (fp32 out)",    0, 32,  0,  0,  1, NT_3WG, 0},
    {conv3_halo_stream_kernels<NT_2WG, false>,        "conv3_halo_stream",     2, 64,  0,  0,  0, NT_2WG, 0},
    {conv3_halo_stream_kernels<NT_2WG, true>,         "conv3_halo_stream",     2, 64,  0,  0,  0, NT_2WG, 1},
    {conv3_halo_stream_kernels<NT_3WG, false>,        "conv3_halo_stream",     2, 64,  0,  0,  0, NT_3WG, 0},
    {conv3_halo_kernels<4, 64>,                       "conv3_halo",            1, 64, 64,  0,  0, NT_3WG, 0},
    {conv3_halo_kernels<4, 32>,                       "conv3_halo",            1, 64, 32,  0,  0, NT_3WG, 0},
    {conv3_halo_kernels<2, 64>,                       "conv3_halo",            1, 32, 64,  0,  0, NT_3WG, 0},
    {conv3_halo_kernels<2, 32>,                       "conv3_halo",            1, 32, 32,  0,  0, NT_3WG, 0},
};

}  // namespace

struct ConvTcPlan {
    CUtensorMap tmA, tmB, tmY, tmAu;
    TcParams p;
    int grid;
    size_t smem;
    const TcKernel* kernel;
    int f16;                      // 1: fp16 activations and weights (kernel->fn[1]), 0: bf16
};

// ---- describe ----
// Human-readable kernel variant and tile shape of a conv: which of the tcgen05 kernels runs the layer and with which tiling,
// so that the selection rules above are visible per layer (plan.op_table(), bench --per-op).
static void tc_format(const TcParams& p, int grid, char* out, size_t n) {
    const char* k = p.halo == 1 ? "halo-ws" : p.halo == 2 ? (p.ybx ? "halo-stream-ybx" : "halo-stream") : (p.cta2 ? "generic-cta2" : "generic");
    snprintf(out, n, "%s M=%dx%dx%d N=%d K=%dx%d stages=%d%s%s%s thr=%d grid=%d", k, p.tb, p.th, p.tw, p.block_n, p.taps * p.kchunks, p.block_k,
             p.stages, p.npair == 2 ? " pair" : "", p.stage64 ? " s64" : "", p.tma_store ? (p.y_f32 ? " tma-f32" : " tma") : " direct", p.nthreads, grid);
}

void conv_tc_describe(const ConvTcPlan* pl, char* out, size_t n) { tc_format(pl->p, pl->grid, out, n); }

extern "C" int yre_conv_tc_describe(const yre_conv_desc* d, int32_t num_sms, char* out, int32_t cap) {
    if (!out || cap <= 0 || num_sms <= 0) YRE_FAIL(YRE_EINVAL, "conv_tc_describe: null output or non-positive size / SM count");
    if (int e = check_conv(d)) return e;
    char why[256] = "";
    if (!tc_shape_rules(*d, why, sizeof(why))) YRE_FAIL(YRE_EUNSUPPORTED, "conv_tc: %s", why);
    TcParams p; int grid; size_t smem;
    if (int e = conv_tc_select(*d, num_sms, tc_knobs(), &p, &grid, &smem)) return e;
    tc_format(p, grid, out, (size_t)cap);
    return YRE_OK;
}

// ---- prepare ----
int conv_tc_eligible(const yre_conv_desc& d, char* why, size_t n) {
    if (!tc_shape_rules(d, why, n)) return 0;
    // address rules: what the tensor maps need
    if (d.xu.ptr && (reinterpret_cast<uintptr_t>(d.xu.ptr) & 127)) NOPE("xu must be 128-byte aligned");
    if ((reinterpret_cast<uintptr_t>(d.x.ptr) & 127) || (reinterpret_cast<uintptr_t>(d.w) & 127)) NOPE("x and w must be 128-byte aligned");
    if (reinterpret_cast<uintptr_t>(d.y.ptr) & 127) NOPE("y must be 128-byte aligned");
    if (d.bias && (reinterpret_cast<uintptr_t>(d.bias) & 15)) NOPE("bias must be 16-byte aligned");
    if (!get_encode()) NOPE("cuTensorMapEncodeTiled unavailable");
    return 1;
}
#undef NOPE

// output tensor map of the staged TMA store: one box = the 32 pixels of a TMEM lane quarter x 32 (64 with stage64) channels;
// fp32 outputs use 128-byte rows (32 channels) in a 128B-swizzled tile.  Also used when an output buffer is re-bound.
static CUresult encode_y(ConvTcPlan* pl, void* ptr) {
    const auto& p = pl->p;
    const cuuint64_t es = p.y_f32 ? 4 : 2, ct = (cuuint64_t)p.y_ctot;
    cuuint64_t gdim[4] = {ct, (cuuint64_t)p.Wo, (cuuint64_t)p.Ho, (cuuint64_t)p.B};
    cuuint64_t gstr[3] = {ct * es, (cuuint64_t)p.Wo * ct * es, (cuuint64_t)p.Ho * p.Wo * ct * es};
    cuuint32_t box[4] = {p.stage64 ? 64u : 32u, (cuuint32_t)p.stw, (cuuint32_t)p.sth, (cuuint32_t)p.stb};
    if (p.ybx) {                                                   // {C, W, B, H}, like the input map
        gdim[2] = (cuuint64_t)p.B; gdim[3] = (cuuint64_t)p.Ho;
        const cuuint64_t sh = gstr[1], sb = gstr[2];
        gstr[1] = sb; gstr[2] = sh;
        box[2] = (cuuint32_t)p.stb; box[3] = (cuuint32_t)p.sth;
    }
    cuuint32_t est[4] = {1, 1, 1, 1};
    const CUtensorMapDataType dt = p.y_f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : pl->f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
    return get_encode()(&pl->tmY, dt, 4, ptr, gdim, gstr, box, est,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, (p.stage64 || p.y_f32) ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                        CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
}

int conv_tc_prepare(const yre_conv_desc& d, ConvTcPlan** out) {
    const EncodeTiledFn enc = get_encode();       // the address rules were checked by conv_tc_eligible
    if (!enc) YRE_FAIL(YRE_EUNSUPPORTED, "conv_tc: cuTensorMapEncodeTiled unavailable");
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const TcKnobs kn = tc_knobs();
    std::unique_ptr<ConvTcPlan> pl(new ConvTcPlan());
    TcParams& p = pl->p;
    if (int e = conv_tc_select(d, sms, kn, &p, &pl->grid, &pl->smem)) return e;
    pl->f16 = d.x.dtype == YRE_F16;
    if (pl->f16) p.idesc &= ~((7u << 7) | (7u << 10));      // A and B format 0 = F16
    const CUtensorMapDataType dt16 = pl->f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
    const int cout = p.halo == 1 ? p.Cout : 0, f32_tma = p.y_f32 && p.tma_store;
    for (const TcKernel& k : TC_KERNELS)
        if (k.halo == p.halo && k.block_k == p.block_k && k.cout == cout && k.cta2 == p.cta2 && k.f32_tma == f32_tma &&
            k.nthreads == p.nthreads && k.stage64 == p.stage64) pl->kernel = &k;
    if (!pl->kernel) YRE_FAIL(YRE_EUNSUPPORTED, "conv_tc: no kernel for halo %d, block_k %d, cta2 %d, %d threads, stage64 %d, "
                              "fp32 TMA store %d", p.halo, p.block_k, p.cta2, p.nthreads, p.stage64, f32_tma);
    if (kn.trace) {
        if (!g_trace_buf) cudaMalloc(&g_trace_buf, 8192 * sizeof(int));
        cudaMemset(g_trace_buf, 0, 8192 * sizeof(int));
        p.dbg = g_trace_buf;
    }

    // ---- tensor maps ----
    const CUtensorMapSwizzle swz = p.block_k == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
    const CUtensorMapL2promotion promoA = (CUtensorMapL2promotion)kn.l2promo_a;
    CUresult r;
    if (!p.phase4) {
        cuuint64_t gdim[4] = {(cuuint64_t)d.x.C_total, (cuuint64_t)d.x.W, (cuuint64_t)d.x.H, (cuuint64_t)d.x.B};
        cuuint64_t gstr[3] = {(cuuint64_t)d.x.C_total * 2, (cuuint64_t)d.x.W * d.x.C_total * 2, (cuuint64_t)d.x.H * d.x.W * d.x.C_total * 2};
        cuuint32_t box[4] = {(cuuint32_t)p.block_k, (cuuint32_t)p.tw, (cuuint32_t)p.th, (cuuint32_t)p.tb};
        if (p.halo) { box[1] = 10; box[2] = 18; box[3] = 1; }      // patch + 1-pixel halo
        if (p.ybx) {                                               // dimension order {C, W, B, H}: box {64, 10, 2 images, 10}
            gdim[2] = (cuuint64_t)d.x.B; gdim[3] = (cuuint64_t)d.x.H;
            const cuuint64_t sh = gstr[1], sb = gstr[2];
            gstr[1] = sb; gstr[2] = sh;
            box[2] = 2; box[3] = 10;
        }
        cuuint32_t est[4] = {1, 1, 1, 1};
        r = enc(&pl->tmA, dt16, 4, d.x.ptr, gdim, gstr, box, est, CU_TENSOR_MAP_INTERLEAVE_NONE, swz,
                promoA, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    } else {
        const cuuint64_t Hp = (cuuint64_t)(d.x.H + 1) / 2, Wp = (cuuint64_t)(d.x.W + 1) / 2, Ct = (cuuint64_t)d.x.C_total;
        cuuint64_t gdim[5] = {Ct, Wp, Hp, (cuuint64_t)d.x.B, 4};
        cuuint64_t gstr[4] = {Ct * 2, Wp * Ct * 2, Hp * Wp * Ct * 2, (cuuint64_t)d.x.B * Hp * Wp * Ct * 2};
        cuuint32_t box[5] = {(cuuint32_t)p.block_k, (cuuint32_t)p.tw, (cuuint32_t)p.th, (cuuint32_t)p.tb, 1};
        cuuint32_t est[5] = {1, 1, 1, 1, 1};
        r = enc(&pl->tmA, dt16, 5, d.x.ptr, gdim, gstr, box, est, CU_TENSOR_MAP_INTERLEAVE_NONE, swz,
                promoA, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    }
    if (r != CUDA_SUCCESS) YRE_FAIL(YRE_ECUDA, "conv_tc: cuTensorMapEncodeTiled(A) failed with %d", (int)r);
    pl->tmAu = pl->tmA;   // unused unless an upsampled source is given
    if (d.xu.ptr) {
        // {C, dup x, W/2, dup y, (H/2) * B}: the duplicated dimensions have stride 0 (accepted by the driver and the TMA
        // unit, scripts/ubench/tma_dup.cu), the images stack along the row dimension
        const cuuint64_t Ct = (cuuint64_t)d.xu.C_total, Wu = (cuuint64_t)d.xu.W, Hu = (cuuint64_t)d.xu.H;
        cuuint64_t gdim[5] = {Ct, 2, Wu, 2, Hu * (cuuint64_t)d.xu.B};
        cuuint64_t gstr[4] = {0, Ct * 2, 0, Wu * Ct * 2};
        cuuint32_t box[5] = {(cuuint32_t)p.block_k, 2, (cuuint32_t)(p.tw / 2), 2, (cuuint32_t)(p.th / 2)};
        cuuint32_t est[5] = {1, 1, 1, 1, 1};
        r = enc(&pl->tmAu, dt16, 5, d.xu.ptr, gdim, gstr, box, est, CU_TENSOR_MAP_INTERLEAVE_NONE, swz,
                promoA, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) YRE_FAIL(YRE_ECUDA, "conv_tc: cuTensorMapEncodeTiled(upsampled A) failed with %d", (int)r);
    }
    {
        const cuuint64_t K = (cuuint64_t)p.taps * p.Cin;
        cuuint64_t gdim[2] = {K, (cuuint64_t)p.Cout};
        cuuint64_t gstr[1] = {K * 2};
        cuuint32_t box[2] = {(cuuint32_t)p.block_k, (cuuint32_t)(p.cta2 ? p.block_n / 2 : p.block_n)};
        cuuint32_t est[2] = {1, 1};
        r = enc(&pl->tmB, dt16, 2, const_cast<void*>(d.w), gdim, gstr, box, est, CU_TENSOR_MAP_INTERLEAVE_NONE, swz,
                CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    }
    if (r != CUDA_SUCCESS) YRE_FAIL(YRE_ECUDA, "conv_tc: cuTensorMapEncodeTiled(W) failed with %d", (int)r);
    if (p.tma_store) {
        r = encode_y(pl.get(), d.y.ptr);
        if (r != CUDA_SUCCESS) YRE_FAIL(YRE_ECUDA, "conv_tc: cuTensorMapEncodeTiled(Y) failed with %d", (int)r);
    } else {
        pl->tmY = pl->tmB;   // unused
    }
    *out = pl.release();
    return YRE_OK;
}

// ---- launch ----
int conv_tc_launch(const ConvTcPlan* pl, cudaStream_t s) {
    static YrePerDeviceOnce once;
    if (int e = once.run([]() -> int {
            for (const TcKernel& k : TC_KERNELS)
                for (int t = 0; t < 2; ++t)
                    YRE_CUDA(cudaFuncSetAttribute(k.fn[t], cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
            return YRE_OK;
        })) return e;
    static const int pdl = tc_knobs().pdl;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)pl->grid); cfg.blockDim = dim3((unsigned)pl->p.nthreads); cfg.dynamicSmemBytes = pl->smem; cfg.stream = s;
    cudaLaunchAttribute at[2];
    int n = 0;
    if (pdl) {
        at[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[n].val.programmaticStreamSerializationAllowed = 1;
        ++n;
    }
    if (pl->p.cta2) {                     // CTA pairs: clusters of two (always on one TPC)
        at[n].id = cudaLaunchAttributeClusterDimension;
        at[n].val.clusterDim.x = 2; at[n].val.clusterDim.y = 1; at[n].val.clusterDim.z = 1;
        ++n;
    }
    cfg.attrs = at; cfg.numAttrs = n;
    YRE_CUDA(cudaLaunchKernelEx(&cfg, pl->kernel->fn[pl->f16], pl->tmA, pl->tmB, pl->tmY, pl->tmAu, pl->p));
    YRE_LAUNCH_CHECK(pl->kernel->name);
    return YRE_OK;
}

void conv_tc_free(ConvTcPlan* p) { delete p; }

void conv_tc_set_reverse(ConvTcPlan* pl, int rev) { pl->p.rev = rev ? 1 : 0; }

int conv_tc_rebind(ConvTcPlan* pl, const void* old_ptr, void* new_ptr) {
    int n = 0;
    if (pl->p.y == old_ptr) {
        if (pl->p.tma_store && encode_y(pl, new_ptr) != CUDA_SUCCESS) return -1;     // the output is baked into a TMA tensor map
        pl->p.y = new_ptr; ++n;
    }
    if (pl->p.res == old_ptr) { pl->p.res = new_ptr; ++n; }
    return n;
}

#ifdef YRE_TUNING
// debugging aid of tuning builds (not part of include/yre.h): copies the last trace buffer (8192 ints) to the host;
// returns 0 when tracing is off
extern "C" int yre_debug_read_trace(int* host, int n) {
    if (!g_trace_buf) return 0;
    cudaDeviceSynchronize();
    cudaMemcpy(host, g_trace_buf, sizeof(int) * (n < 8192 ? n : 8192), cudaMemcpyDeviceToHost);
    return n < 8192 ? n : 8192;
}
#endif
