// K7: batched class-aware NMS, bit-exact with the reference.
//
//   reference: non_max_suppression           src/yolo/utils/nms.py:19-94
//              torchvision.ops.nms via _nms   src/yolo/utils/nms.py:97-104
//
// Three launches for the whole batch (the reference loops over images in Python):
//   nms_init    zero the per-image counters
//   nms_filter  HBM-bound pass over pred[B][A][4+nc]: per-anchor first-max class, strict
//               `conf > thr` (+ optional class filter), xywh->xyxy, per-image max coordinate,
//               compaction of (score, anchor) sort keys
//   nms_select  one CTA (1024 threads) per image: the candidates' 64-bit keys in ascending order (== stable
//               descending score sort, ties -> lower anchor first) by a bitonic sort in shared memory; above
//               8192 candidates only the best ~3000 are selected (threshold from a sorted sample) and sorted,
//               because the scan below stops a few hundred candidates deep -- with an exact fallback to a
//               full segmented sort.  Then a chunked greedy scan: every chunk of CHUNK sorted candidates is
//               tested against the boxes kept so far (<= max_det, two threads per candidate), an IoU bitmask is
//               built inside the chunk (32 warps; pairs of different classes are skipped where that is provably
//               exact), and warp 0 resolves the chunk by walking the set bits of the survivors.  The scan stops
//               as soon as max_det boxes are kept, which is exactly `keep[:max_det]` of the reference -- there
//               is no pre-NMS top-k cap.
//
// Bit-exactness notes: every fp32 op is an explicitly rounded intrinsic (no FMA contraction);
// the class offset is `float(cls) * (max_coord + 1)` then `box + offset` as two rounded ops
// (nms.py:79-81); IoU is inter / ((area_i + area_j) - inter) in fp32, compared against the
// threshold as a DOUBLE, as torchvision's CPU kernel does.
#include "yre_common.cuh"

namespace {

constexpr int CHUNK = 512;            // candidates per greedy round
constexpr int NT_SEL = 1024;          // threads of nms_select (two per candidate of a chunk)
constexpr int MW = CHUNK / 32;        // 32-bit mask words per row
constexpr int SMEM_KEYS = 8192;       // keys sorted in shared memory at a time (one segment)
constexpr int NMS_MAX_DET = 4096;     // largest accepted max_det (sizes nms_select's shared-memory opt-in)

typedef unsigned long long u64;

// byte offsets of nms_select's fixed-size shared-memory arrays (the max_det-sized ones follow the key buffer)
constexpr unsigned OFF_CBOX = 0, OFF_UBOX = OFF_CBOX + 16 * CHUNK, OFF_MASK = OFF_UBOX + 16 * CHUNK,
                   OFF_AREA = OFF_MASK + 4 * CHUNK * MW, OFF_CONF = OFF_AREA + 4 * CHUNK, OFF_CLS = OFF_CONF + 4 * CHUNK,
                   OFF_ANC = OFF_CLS + 4 * CHUNK, OFF_KPOS = OFF_ANC + 4 * CHUNK, OFF_DEAD = OFF_KPOS + 4 * CHUNK,
                   OFF_INFO = OFF_DEAD + 4 * CHUNK, OFF_ALIVE = OFF_INFO + 4 * CHUNK, OFF_KEYS = OFF_ALIVE + 128,
                   OFF_KBOX = OFF_KEYS + 8 * SMEM_KEYS;
__device__ __forceinline__ float4 lds128(unsigned a) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ unsigned lds32(unsigned a) {
    unsigned v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts32(unsigned a, unsigned v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }

__device__ __forceinline__ unsigned f2ord(float f) {   // order-preserving float -> uint
    const unsigned u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ord2f(unsigned o) {
    return __uint_as_float((o & 0x80000000u) ? (o & 0x7fffffffu) : ~o);
}

struct NmsWs {           // carved out of the caller's workspace
    u64* keys;           // [B][cap]
    int* cls;            // [B][A]
    int* count;          // [B]
    unsigned* maxc;      // [B] (ordered-uint encoding)
    int cap;
};

__host__ __device__ inline int pow2ceil(int v) { int p = 1; while (p < v) p <<= 1; return p; }

#ifdef YRE_TUNING
// tuning builds: SM-clock stamps of image 0's CTA at the phase boundaries of nms_select (yre_debug_nms_prof reads them)
__device__ long long g_nms_prof[16];
// (BAR.SYNC blocks lazily, at the first consumer of barrier-protected state: a volatile shared-memory read pins the stamp
//  behind the barrier that precedes it)
#define NMS_STAMP(i) do { if (blockIdx.x == 0 && threadIdx.x == 0) { volatile int* vs = &s_newkept; long long t_ = clock64() + (long long)(*vs & 0); g_nms_prof[i] = t_; } } while (0)
#else
#define NMS_STAMP(i) do { } while (0)
#endif

__global__ void nms_init_kernel(int* count, unsigned* maxc, int B) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < B) { count[i] = 0; maxc[i] = 0u; }
}

// ---------------------------------------------------------------------------------------------
// filter: one warp per 32 consecutive anchors of one image; rows are read as coalesced float4
struct FilterParams {
    const float* pred; int B, A, nc; float conf; const int* classes; int n_classes;
    NmsWs ws;
};

__global__ void __launch_bounds__(128) nms_filter_kernel(const FilterParams p) {
    extern __shared__ __align__(16) unsigned char smraw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n4 = (4 + p.nc) / 4;                 // float4 per row (nc % 4 == 0)
    const int nparts = n4 - 1;
    const int pitch = nparts | 1;                  // odd pitch: conflict-free per-lane rows
    float* pv = reinterpret_cast<float*>(smraw) + (size_t)warp * 32 * pitch * 2;    // [32][pitch] best value
    int* pi = reinterpret_cast<int*>(pv + 32 * pitch);                               // [32][pitch] best class

    const int tiles = (p.A + 31) / 32;
    const int wglobal = blockIdx.x * (blockDim.x >> 5) + warp;
    if (wglobal >= tiles * p.B) return;
    const int b = wglobal / tiles, a0 = (wglobal % tiles) * 32;
    const int na = min(32, p.A - a0);
    const float4* base = reinterpret_cast<const float4*>(p.pred + ((size_t)b * p.A + a0) * (4 + p.nc));

    const bool vec = (p.nc & 3) == 0;        // rows are 16-byte aligned only when nc % 4 == 0
    // loads are issued 8 at a time into registers before anything is consumed (no load -> use -> load chain)
    for (int base0 = 0; vec && base0 < na * n4; base0 += 8 * 32) {
        float4 buf[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const int idx = base0 + q * 32 + lane;
            if (idx < na * n4) buf[q] = base[idx];
        }
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const int idx = base0 + q * 32 + lane;
            if (idx >= na * n4) continue;
            const int al = idx / n4, pos = idx - al * n4;
            if (pos == 0) continue;
            const float4 v = buf[q];
            float best = v.x; int bi = 0;
            if (v.y > best) { best = v.y; bi = 1; }
            if (v.z > best) { best = v.z; bi = 2; }
            if (v.w > best) { best = v.w; bi = 3; }
            pv[al * pitch + pos - 1] = best;
            pi[al * pitch + pos - 1] = (pos - 1) * 4 + bi;
        }
    }
    __syncwarp();

    bool cand = false;
    float conf = 0.f; int cls = 0;
    float x1 = 0, y1 = 0, x2 = 0, y2 = 0;
    if (lane < na) {
        if (vec) {
            conf = pv[lane * pitch]; cls = pi[lane * pitch];
            for (int q = 1; q < nparts; ++q) {
                const float v = pv[lane * pitch + q];
                if (v > conf) { conf = v; cls = pi[lane * pitch + q]; }     // strict > keeps the first max
            }
        } else {                              // generic class count: one lane walks its own row
            const float* row = p.pred + ((size_t)b * p.A + a0 + lane) * (4 + p.nc);
            conf = row[4];
            for (int q = 1; q < p.nc; ++q) {
                const float v = row[4 + q];
                if (v > conf) { conf = v; cls = q; }
            }
        }
        cand = conf > p.conf;
        if (cand && p.n_classes >= 0) {
            bool ok = false;
            for (int k = 0; k < p.n_classes; ++k) ok |= (p.classes[k] == cls);
            cand = ok;
        }
        if (cand) {
            const float* brow = p.pred + ((size_t)b * p.A + a0 + lane) * (4 + p.nc);
            const float4 bx = vec ? base[lane * n4] : make_float4(brow[0], brow[1], brow[2], brow[3]);
            const float hw = __fmul_rn(bx.z, 0.5f), hh = __fmul_rn(bx.w, 0.5f);   // w/2, h/2 (exact)
            x1 = __fsub_rn(bx.x, hw); y1 = __fsub_rn(bx.y, hh);
            x2 = __fadd_rn(bx.x, hw); y2 = __fadd_rn(bx.y, hh);
        }
    }
    const unsigned ballot = __ballot_sync(0xffffffffu, cand);
    if (ballot == 0u) return;
    // per-image max coordinate over candidate boxes
    unsigned mo = cand ? max(max(f2ord(x1), f2ord(y1)), max(f2ord(x2), f2ord(y2))) : 0u;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mo = max(mo, __shfl_xor_sync(0xffffffffu, mo, o));
    int slot0 = 0;
    if (lane == 0) {
        atomicMax(p.ws.maxc + b, mo);
        slot0 = atomicAdd(p.ws.count + b, __popc(ballot));
    }
    slot0 = __shfl_sync(0xffffffffu, slot0, 0);
    if (cand) {
        const int slot = slot0 + __popc(ballot & ((1u << lane) - 1u));
        const int a = a0 + lane;
        p.ws.keys[(size_t)b * p.ws.cap + slot] = ((u64)(~f2ord(conf)) << 32) | (unsigned)a;
        p.ws.cls[(size_t)b * p.A + a] = cls;
    }
}

// ---------------------------------------------------------------------------------------------
struct SelectParams {
    const float* pred; int B, A, nc; double iou; int max_det, agnostic;
    NmsWs ws;
    float* out; int* counts; long long* keep_anchor;
    const float* scale;   // optional [B][5] = pad_w, pad_h, gain, orig_w, orig_h (scale_boxes fused into the output)
    float iou_lo, iou_hi; // iou * (1 -+ 2^-18) as floats: the division-free shortcut of iou_gt (0 / 0: shortcut off)
};

// thresholds of the division-free shortcut in iou_gt: thr * (1 -+ 2^-18) as floats, computed once on the host (as
// kernel parameters they are constant-bank operands; derived in the kernel they were re-computed in fp64 at every use)
struct IouThr { double thr; float lo, hi; bool quick, nonneg; };

// IoU(a, b) > thr with the reference's arithmetic: inter / ((area_a + area_b) - inter) in fp32 (IEEE division), compared
// against the threshold as a double.  The division (~45 issued instructions with its special-case path) is skipped when
// the outcome is certain: an fp32 product and an fp32 quotient are each within 2^-24 of the exact value, so
// inter < thr (1 - 2^-18) union implies quotient < thr and inter > thr (1 + 2^-18) union implies quotient > thr; only ratios
// within 4e-6 of the threshold (and non-positive / tiny / NaN unions) take the exact path.
__device__ __forceinline__ bool iou_gt(const float4 a, const float aa, const float4 b, const float ab, const IouThr t) {
    const float w = fmaxf(0.f, __fsub_rn(fminf(a.z, b.z), fmaxf(a.x, b.x)));
    const float h = fmaxf(0.f, __fsub_rn(fminf(a.w, b.w), fmaxf(a.y, b.y)));
    const float inter = __fmul_rn(w, h);
    // inter == 0 -> IoU is +-0 or NaN, neither exceeds a threshold >= 0: skip the IEEE division (exact shortcut)
    if (inter == 0.f && t.nonneg) return false;
    const float uni = __fsub_rn(__fadd_rn(aa, ab), inter);
    if (t.quick && uni > 1e-30f && uni < 1e30f) {
        if (inter < __fmul_rn(t.lo, uni)) return false;
        if (inter > __fmul_rn(t.hi, uni)) return true;
    }
    const float iou = __fdiv_rn(inter, uni);
    return (double)iou > t.thr;
}

// bitonic network stages of merge size k with compare distances j = j_hi, j_hi/2, ..., 1 on the np_local keys in d
// (shared memory); `base` = global index of d[0] (the sort direction of an element depends on its GLOBAL index)
__device__ __forceinline__ void bitonic_local(u64* d, int np_local, int base, int k, int j_hi) {
    for (int j = j_hi; j > 0; j >>= 1) {
        for (int i = threadIdx.x; i < (np_local >> 1); i += blockDim.x) {
            const int lo = ((i & ~(j - 1)) << 1) | (i & (j - 1));
            const int hi = lo | j;
            const bool asc = ((base + lo) & k) == 0;
            const u64 a = d[lo], b = d[hi];
            if ((a > b) == asc) { d[lo] = b; d[hi] = a; }
        }
        __syncthreads();
    }
}

// one stage (merge size k, distance j >= SMEM_KEYS) over np keys in global memory; loads are batched ahead of the
// compare-exchange so that a thread has eight independent pairs in flight instead of one
__device__ __forceinline__ void bitonic_global_stage(u64* d, int np, int k, int j) {
    constexpr int U = 8;
    const int half = np >> 1;
    for (int i0 = threadIdx.x; i0 < half; i0 += blockDim.x * U) {
        u64 a[U], b[U];
        int lo[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int i = i0 + u * (int)blockDim.x;
            lo[u] = ((i & ~(j - 1)) << 1) | (i & (j - 1));
            if (i < half) { a[u] = d[lo[u]]; b[u] = d[lo[u] | j]; }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int i = i0 + u * (int)blockDim.x;
            if (i < half) {
                const bool asc = (lo[u] & k) == 0;
                if ((a[u] > b[u]) == asc) { d[lo[u]] = b[u]; d[lo[u] | j] = a[u]; }
            }
        }
    }
    __syncthreads();
}

// ascending sort of m keys that already sit in shared memory (padded to a power of two with ~0)
__device__ __forceinline__ void sort_smem(u64* skeys, int m) {
    const int np = pow2ceil(m);
    for (int i = m + threadIdx.x; i < np; i += blockDim.x) skeys[i] = ~0ull;
    __syncthreads();
    for (int k = 2; k <= np; k <<= 1) bitonic_local(skeys, np, 0, k, k >> 1);
}

// Full ascending sort of n > keys_in_smem keys in global memory (padded to np = pow2 with ~0): the bitonic network run
// segment-wise -- SEG-key segments are sorted / merged in shared memory, only the stages with a compare distance
// >= SEG touch global memory.  Rarely needed (see top_keys).
__device__ void sort_global(u64* gkeys, int n, u64* skeys, int SEG) {
    const int tid = threadIdx.x;
    const int np = pow2ceil(n);                          // a multiple of SEG (both powers of two)
    for (int i = n + tid; i < np; i += blockDim.x) gkeys[i] = ~0ull;
    __syncthreads();
    for (int s0 = 0; s0 < np; s0 += SEG) {               // every segment: all merge sizes up to SEG
        for (int i = tid; i < SEG; i += blockDim.x) skeys[i] = gkeys[s0 + i];
        __syncthreads();
        for (int k = 2; k <= SEG; k <<= 1) bitonic_local(skeys, SEG, s0, k, k >> 1);
        for (int i = tid; i < SEG; i += blockDim.x) gkeys[s0 + i] = skeys[i];
        __syncthreads();
    }
    for (int k = SEG << 1; k <= np; k <<= 1) {           // larger merge sizes
        for (int j = k >> 1; j >= SEG; j >>= 1) bitonic_global_stage(gkeys, np, k, j);
        for (int s0 = 0; s0 < np; s0 += SEG) {
            for (int i = tid; i < SEG; i += blockDim.x) skeys[i] = gkeys[s0 + i];
            __syncthreads();
            bitonic_local(skeys, SEG, s0, k, SEG >> 1);
            for (int i = tid; i < SEG; i += blockDim.x) gkeys[s0 + i] = skeys[i];
            __syncthreads();
        }
    }
}

// The greedy scan stops after max_det keeps, i.e. a few hundred candidates deep (measured: rank 360-730 of up to 33 600),
// so a full sort of a large candidate set is wasted work.  top_keys puts the SMALLEST m keys (= the m best candidates in
// reference order), sorted, into shared memory: a threshold is read off a sorted sample of <= 4096 keys so that about
// TARGET keys pass, those are compacted and sorted.  *partial tells the caller that candidates beyond the m exist; if the
// scan runs out of the m before max_det boxes are kept it redoes the image on the fully sorted list (sort_global).
constexpr int TOP_TARGET = 3072;
__device__ int top_keys(const u64* gkeys, int n, u64* skeys, int keys_in_smem, int* s_cnt, bool* partial) {
    const int tid = threadIdx.x;
    if (n <= keys_in_smem) {
        for (int i = tid; i < n; i += blockDim.x) skeys[i] = gkeys[i];
        __syncthreads();
        sort_smem(skeys, n);
        *partial = false;
        return n;
    }
    const int stride = (n + 4095) / 4096;
    const int ns = (n + stride - 1) / stride;            // <= 4096 samples
    for (int i = tid; i < ns; i += blockDim.x) skeys[i] = gkeys[(size_t)i * stride];
    __syncthreads();
    sort_smem(skeys, ns);
    const u64 thr = skeys[min(ns - 1, TOP_TARGET / stride)];
    if (tid == 0) *s_cnt = 0;
    __syncthreads();                                      // every thread holds thr: the sample buffer can be reused
    for (int i = tid; i < n; i += blockDim.x) {
        const u64 k = gkeys[i];
        if (k <= thr) {
            const int pos = atomicAdd(s_cnt, 1);
            if (pos < keys_in_smem) skeys[pos] = k;
        }
    }
    __syncthreads();
    const int m = *s_cnt;
    if (m > keys_in_smem) return -1;                      // pathological score distribution: caller sorts everything
    sort_smem(skeys, m);
    *partial = m < n;
    return m;
}

// packed (class, leaky) of a candidate -- see the cross-class shortcut in nms_select_kernel
__device__ __forceinline__ bool may_overlap(int ia, int ib) {
    const int ca = ia & 0x3fffffff, cb = ib & 0x3fffffff;
    if (ca == cb) return true;
    return ((ca > cb ? ia : ib) >> 30) & 1;               // the box of the HIGHER class must reach below -0.5 in x and y
}

__global__ void __launch_bounds__(NT_SEL) nms_select_kernel(const SelectParams p) {
    extern __shared__ __align__(16) unsigned char smraw[];
    // carve shared memory.  Every array the inner loops touch sits at a COMPILE-TIME offset (fixed-size arrays first, the
    // max_det-sized ones last): with run-time offsets and 64 registers per thread the compiler re-derived the bases from
    // the kernel parameters inside the loops -- ~25 of the ~65 instructions per 32 pairs (ncu source view, profiles/).
    float4* cbox = reinterpret_cast<float4*>(smraw + OFF_CBOX);      // [CHUNK] offset boxes
    float4* ubox = reinterpret_cast<float4*>(smraw + OFF_UBOX);      // [CHUNK] plain boxes
    unsigned* mask32 = reinterpret_cast<unsigned*>(smraw + OFF_MASK);// [CHUNK][MW] 32-bit mask words
    float* carea = reinterpret_cast<float*>(smraw + OFF_AREA);       // [CHUNK]
    float* cconf = reinterpret_cast<float*>(smraw + OFF_CONF);       // [CHUNK]
    int* ccls = reinterpret_cast<int*>(smraw + OFF_CLS);             // [CHUNK]
    int* canc = reinterpret_cast<int*>(smraw + OFF_ANC);             // [CHUNK]
    int* kpos = reinterpret_cast<int*>(smraw + OFF_KPOS);            // [CHUNK] chunk positions kept this round
    int* dead = reinterpret_cast<int*>(smraw + OFF_DEAD);            // [CHUNK] suppressed by an earlier chunk's keeps
    int* cinfo = reinterpret_cast<int*>(smraw + OFF_INFO);           // [CHUNK] class | leaky << 30
    unsigned* alive_w = reinterpret_cast<unsigned*>(smraw + OFF_ALIVE);   // [CHUNK/32]
    u64* skeys = reinterpret_cast<u64*>(smraw + OFF_KEYS);           // [SMEM_KEYS]
    float4* kbox = reinterpret_cast<float4*>(smraw + OFF_KBOX);      // [max_det] kept offset boxes
    float* karea = reinterpret_cast<float*>(kbox + p.max_det);       // [max_det]
    int* kinfo = reinterpret_cast<int*>(karea + p.max_det);          // [max_det]
    // 32-bit shared address of the carve, made opaque so that it stays in ONE register (the compiler otherwise re-derives
    // it from the cluster CTA id at every use): the mask phase addresses everything as sb + constant + index
    unsigned sb = (unsigned)__cvta_generic_to_shared(smraw);
    asm volatile("" : "+r"(sb));
    __shared__ int s_newkept, s_cnt;
    __shared__ bool s_partial;

    const int b = blockIdx.x, tid = threadIdx.x;
    const int n = min(p.ws.count[b], p.A);
    if (n == 0) { if (tid == 0) p.counts[b] = 0; return; }
    u64* gkeys = p.ws.keys + (size_t)b * p.ws.cap;
    NMS_STAMP(0);
    int n_scan = top_keys(gkeys, n, skeys, SMEM_KEYS, &s_cnt, &s_partial);
    __syncthreads();
    bool partial = s_partial;
    const u64* keys = skeys;
    if (n_scan < 0) { sort_global(gkeys, n, skeys, SMEM_KEYS); keys = gkeys; n_scan = n; partial = false; }
    NMS_STAMP(1);

    const float scale = __fadd_rn(ord2f(p.ws.maxc[b]), 1.0f);
    // Cross-class shortcut (exact).  Class-aware NMS adds cls * scale to every coordinate (nms.py:79-81), scale = max
    // coordinate + 1, so boxes of different classes sit in disjoint diagonal blocks -- unless a coordinate is negative
    // enough to reach back into the previous class's block (the reference's leakage, which must be reproduced).  While
    // nc * scale < 2^22 every rounding involved is <= 1/8: for classes c1 < c2 the two offsets differ by at least
    // scale - 0.25, scale >= max coordinate + 0.875, and every x2 / y2 of class c1 is <= max coordinate; rounding is
    // monotone, so the offset boxes can only intersect if the box of class c2 has x1 < -0.5 AND y1 < -0.5 ("leaky").
    // Pairs of different classes whose higher-class box is not leaky have an empty intersection: IoU = 0, never
    // suppressed, skipped without evaluating it.
    IouThr ithr;
    ithr.thr = p.iou; ithr.lo = p.iou_lo; ithr.hi = p.iou_hi; ithr.quick = p.iou_hi > 0.f; ithr.nonneg = p.iou >= 0.0;
    // (a threshold < 0 suppresses pairs whose IoU is 0 as well, so the shortcut then does not apply)
    const bool prune = !p.agnostic && ithr.nonneg && __fmul_rn(__int2float_rn(p.nc), scale) < 4194304.f;
    const int rowf = 4 + p.nc;
    int kept = 0;
    for (int pass = 0; pass < 2; ++pass) {
    kept = 0;
    for (int c0 = 0; c0 < n_scan && kept < p.max_det; c0 += CHUNK) {
        const int cnt = min(CHUNK, n_scan - c0);
        // ---- 1. load this chunk's candidates (threads 0 .. cnt-1) ----
        if (tid < CHUNK) dead[tid] = 0;
        if (tid < cnt) {
            const u64 key = keys[c0 + tid];
            const int a = (int)(unsigned)(key & 0xffffffffu);
            const float conf = ord2f(~(unsigned)(key >> 32));
            const int cls = p.ws.cls[(size_t)b * p.A + a];
            const float* row = p.pred + ((size_t)b * p.A + a) * rowf;
            const float4 bx = (p.nc & 3) ? make_float4(row[0], row[1], row[2], row[3]) : *reinterpret_cast<const float4*>(row);
            const float hw = __fmul_rn(bx.z, 0.5f), hh = __fmul_rn(bx.w, 0.5f);
            float4 u, mine;
            u.x = __fsub_rn(bx.x, hw); u.y = __fsub_rn(bx.y, hh); u.z = __fadd_rn(bx.x, hw); u.w = __fadd_rn(bx.y, hh);
            if (p.agnostic) mine = u;
            else {
                const float off = __fmul_rn(__int2float_rn(cls), scale);
                mine.x = __fadd_rn(u.x, off); mine.y = __fadd_rn(u.y, off);
                mine.z = __fadd_rn(u.z, off); mine.w = __fadd_rn(u.w, off);
            }
            ubox[tid] = u; cbox[tid] = mine;
            carea[tid] = __fmul_rn(__fsub_rn(mine.z, mine.x), __fsub_rn(mine.w, mine.y));
            cconf[tid] = conf; ccls[tid] = cls; canc[tid] = a;
            cinfo[tid] = cls | ((u.x < -0.5f && u.y < -0.5f) ? (1 << 30) : 0);
        }
        __syncthreads();
        if (c0 == 0) NMS_STAMP(2);
        // ---- 2. against everything kept by earlier chunks: two threads per candidate, each half of the kept list
        //         (whether ANY kept box suppresses the candidate is all that matters, so the split is exact) ----
        {
            constexpr int NPART = NT_SEL / CHUNK;
            const int c = tid % CHUNK, part = tid / CHUNK;
            if (c < cnt && kept > 0) {
                const int k0 = part * kept / NPART, k1 = (part + 1) * kept / NPART;
                const float4 mine = cbox[c];
                const float marea = carea[c];
                const int mi = cinfo[c];
                for (int k = k0; k < k1; ++k) {
                    if (prune && !may_overlap(kinfo[k], mi)) continue;
                    if (iou_gt(kbox[k], karea[k], mine, marea, ithr)) { dead[c] = 1; break; }
                }
            }
        }
        __syncthreads();
        if (tid < CHUNK) {
            const bool alive = tid < cnt && !dead[tid];
            const unsigned bal = __ballot_sync(0xffffffffu, alive);
            if ((tid & 31) == 0) alive_w[tid >> 5] = bal;
        }
        __syncthreads();
        if (c0 == 0) NMS_STAMP(3);
        // ---- 3. in-chunk suppression bitmask (row i: later boxes j > i it would suppress), 32-bit words ----
        // The lower triangle is cut into 32 x 32 tiles (column block cb, row block rb <= cb), dealt round-robin to the 32
        // warps.  In a tile every lane owns ONE column -- box / area / class held in registers -- and the warp walks the 32
        // rows: a few broadcast shared-memory loads per row, the IoU test against the lane's own column, one ballot = one
        // mask word.  (The first version walked columns per row with per-lane index arithmetic and loads: ~90 issued
        // instructions per 32 pairs, now ~45; dealing whole column blocks to warps left the last warp with 16x the work
        // of the first.  Measured alternatives that lost: two rows per turn (spills at 64 registers), a branch-free
        // classification (gives up the class shortcut), 512 threads with 128 registers (fewer warps to hide the
        // ~400-cycle dependent chain of a row).)
        {
            const int wid = tid >> 5, ln = tid & 31;
            const int nb = (cnt + 31) >> 5;                           // 32-candidate blocks in this chunk
            const int ntile = nb * (nb + 1) / 2;
            for (int t = wid; t < ntile; t += NT_SEL / 32) {
                int cb = 0;
                while ((cb + 1) * (cb + 2) / 2 <= t) ++cb;            // tile t -> (cb, rb), rb <= cb
                int rb = t - cb * (cb + 1) / 2;
                asm volatile("" : "+r"(rb), "+r"(cb));                // keep them in registers (not re-derived per row)
                const int j = cb * 32 + ln;
                const bool jv = j < cnt && ((lds32(sb + OFF_ALIVE + 4u * cb) >> ln) & 1u);
                float4 bj = make_float4(0.f, 0.f, 0.f, 0.f);
                float aj = 0.f;
                int ij = 0;
                if (jv) { bj = lds128(sb + OFF_CBOX + 16u * j); aj = __uint_as_float(lds32(sb + OFF_AREA + 4u * j)); ij = (int)lds32(sb + OFF_INFO + 4u * j); }
                unsigned rows = lds32(sb + OFF_ALIVE + 4u * rb);      // alive rows of the block (rows >= cnt are not alive)
                const unsigned a_mask = sb + OFF_MASK + 4u * (unsigned)cb;
                while (rows) {                                        // warp-uniform walk over the alive rows
                    const int i = rb * 32 + __ffs((int)rows) - 1;
                    rows &= rows - 1;
                    bool sup = false;
                    if (jv && j > i) {
                        const int ii = (int)lds32(sb + OFF_INFO + 4u * i);
                        if (!prune || may_overlap(ii, ij))
                            sup = iou_gt(lds128(sb + OFF_CBOX + 16u * i), __uint_as_float(lds32(sb + OFF_AREA + 4u * i)), bj, aj, ithr);
                    }
                    const unsigned bal = __ballot_sync(0xffffffffu, sup);
                    if (ln == 0) sts32(a_mask + 4u * MW * (unsigned)i, bal);
                }
            }
        }
        __syncthreads();
        if (c0 == 0) NMS_STAMP(4);
        // ---- 4. resolution of the chunk by warp 0: walk the set bits of (alive & ~removed) of one 32-candidate word at a
        //         time.  Every lane tracks the current word (same value in all lanes, no shuffle in the loop); lane v also
        //         accumulates word v of the removed set for the words still to come.  ~120 cycles per kept box
        //         (scripts/ubench/resolve_loop.cu), against ~160 for one thread with the whole set in its registers. ----
        if (tid < 32) {
            const int ln = tid, nw = (cnt + 31) >> 5;
            unsigned removed_own = 0u;                                // lane v < nw: word v of the removed set
            int nk = 0;
            bool full = false;
            for (int w = 0; w < nw && !full; ++w) {
                unsigned rem_w = __shfl_sync(0xffffffffu, removed_own, w);
                unsigned cand = alive_w[w] & ~rem_w;
                while (cand) {
                    const int i = w * 32 + __ffs((int)cand) - 1;
                    if (ln == 0) kpos[nk] = i;
                    ++nk;
                    if (kept + nk >= p.max_det) { full = true; break; }
                    const unsigned* mrow = mask32 + i * MW;
                    rem_w |= mrow[w];                                 // broadcast load: the word being walked
                    if (ln > w && ln < nw) removed_own |= mrow[ln];   // the later words, one per lane
                    cand &= cand - 1;                                 // this candidate is done
                    cand &= ~rem_w;                                   // and so is everything a keep suppresses
                }
            }
            if (ln == 0) s_newkept = nk;
#ifdef YRE_TUNING
            if (c0 == 0 && blockIdx.x == 0 && ln == 0) { g_nms_prof[8] = clock64(); g_nms_prof[9] = nk; g_nms_prof[10] = cnt; }
#endif
        }
        __syncthreads();
        if (c0 == 0) NMS_STAMP(5);
        // ---- 5. publish the newly kept boxes ----
        const int nk = s_newkept;
        for (int q = tid; q < nk; q += blockDim.x) {
            const int i = kpos[q], k = kept + q;
            kbox[k] = cbox[i]; karea[k] = carea[i]; kinfo[k] = cinfo[i];
            float* o = p.out + ((size_t)b * p.max_det + k) * 6;
            float4 u = ubox[i];
            if (p.scale) {        // scale_boxes (scripts/detect.py:74-109), same ops as scale_boxes_kernel (k_preproc.cu)
                const float* sc = p.scale + (size_t)b * 5;
                const float pw = sc[0], ph = sc[1], gain = sc[2], ow = sc[3], oh = sc[4];
                u.x = fminf(fmaxf(__fdiv_rn(__fsub_rn(u.x, pw), gain), 0.f), ow);
                u.y = fminf(fmaxf(__fdiv_rn(__fsub_rn(u.y, ph), gain), 0.f), oh);
                u.z = fminf(fmaxf(__fdiv_rn(__fsub_rn(u.z, pw), gain), 0.f), ow);
                u.w = fminf(fmaxf(__fdiv_rn(__fsub_rn(u.w, ph), gain), 0.f), oh);
            }
            o[0] = u.x; o[1] = u.y; o[2] = u.z; o[3] = u.w; o[4] = cconf[i]; o[5] = __int2float_rn(ccls[i]);
            p.keep_anchor[(size_t)b * p.max_det + k] = canc[i];
        }
        kept += nk;
        __syncthreads();
        if (c0 == 0) NMS_STAMP(6);
    }
    // the best TOP_TARGET candidates did not yield max_det boxes and there are more: redo the image on the full sorted list
    if (!(partial && kept < p.max_det)) break;
    sort_global(gkeys, n, skeys, SMEM_KEYS);
    keys = gkeys; n_scan = n; partial = false;
    }
    NMS_STAMP(7);
    if (tid == 0) p.counts[b] = kept;
}

size_t select_smem_bytes(int max_det) {
    return sizeof(float4) * (2 * CHUNK + (size_t)max_det) + sizeof(unsigned) * ((size_t)CHUNK * MW + 32) + sizeof(u64) * SMEM_KEYS +
           sizeof(float) * (2 * CHUNK + (size_t)max_det) + sizeof(int) * (5 * CHUNK + (size_t)max_det) + 64;
}

NmsWs carve(void* ws, int B, int A) {
    NmsWs w;
    w.cap = pow2ceil(A);
    unsigned char* p = reinterpret_cast<unsigned char*>(ws);
    w.keys = reinterpret_cast<u64*>(p); p += sizeof(u64) * (size_t)B * w.cap;
    w.cls = reinterpret_cast<int*>(p); p += sizeof(int) * (size_t)B * A;
    w.count = reinterpret_cast<int*>(p); p += sizeof(int) * (size_t)B;
    w.maxc = reinterpret_cast<unsigned*>(p);
    return w;
}

}  // namespace

extern "C" size_t yre_nms_workspace_bytes(int32_t B, int32_t A) {
    if (B <= 0 || A <= 0) return 0;
    return sizeof(u64) * (size_t)B * pow2ceil(A) + sizeof(int) * (size_t)B * A + 2 * sizeof(int) * (size_t)B + 256;
}

static int check_nms(const yre_nms_desc& d, bool outputs) {
    if (!d.pred || !d.workspace) YRE_FAIL(YRE_EINVAL, "nms: null pointer");
    if (outputs && (!d.out || !d.counts || !d.keep_anchor)) YRE_FAIL(YRE_EINVAL, "nms: null output pointer");
    if (d.B <= 0 || d.A <= 0 || d.nc <= 0) YRE_FAIL(YRE_EINVAL, "nms: bad extent B=%d A=%d nc=%d", d.B, d.A, d.nc);
    if (d.max_det <= 0 || d.max_det > NMS_MAX_DET) YRE_FAIL(YRE_EUNSUPPORTED, "nms: max_det=%d (supported 1..%d)", d.max_det, NMS_MAX_DET);
    if (d.workspace_bytes < yre_nms_workspace_bytes(d.B, d.A)) YRE_FAIL(YRE_EINVAL, "nms: workspace too small");
    if (d.n_classes > 0 && !d.classes) YRE_FAIL(YRE_EINVAL, "nms: classes pointer missing");
    if ((reinterpret_cast<uintptr_t>(d.pred) & 15) || (reinterpret_cast<uintptr_t>(d.workspace) & 15))
        YRE_FAIL(YRE_EINVAL, "nms: pred/workspace must be 16-byte aligned");
    return YRE_OK;
}

static int launch_nms_filter(const yre_nms_desc& d, const NmsWs& ws, cudaStream_t s) {
    nms_init_kernel<<<yre_cdiv(d.B, 256), 256, 0, s>>>(ws.count, ws.maxc, d.B);
    YRE_LAUNCH_CHECK("nms_init");

    FilterParams fp;
    fp.pred = d.pred; fp.B = d.B; fp.A = d.A; fp.nc = d.nc; fp.conf = d.conf_thres;
    fp.classes = d.classes; fp.n_classes = d.n_classes; fp.ws = ws;
    const size_t per_warp = (d.nc % 4 == 0) ? (size_t)32 * ((d.nc / 4) | 1) * 8 : 16;
    int warps = 4;
    while (warps > 1 && per_warp * warps > 40 * 1024) warps >>= 1;
    if (per_warp * warps > 48 * 1024) YRE_FAIL(YRE_EUNSUPPORTED, "nms: nc=%d too large", d.nc);
    const int tiles = yre_cdiv(d.A, 32) * d.B;
    nms_filter_kernel<<<yre_cdiv(tiles, warps), warps * 32, per_warp * warps, s>>>(fp);
    YRE_LAUNCH_CHECK("nms_filter");
    return YRE_OK;
}

extern "C" int yre_nms_filter_only(const yre_nms_desc* d, yre_stream_t s) {
    if (!d) YRE_FAIL(YRE_EINVAL, "nms: null descriptor");
    if (int e = check_nms(*d, false)) return e;
    return launch_nms_filter(*d, carve(d->workspace, d->B, d->A), (cudaStream_t)s);
}

int launch_nms(const yre_nms_desc& d, cudaStream_t s) {
    if (int e = check_nms(d, true)) return e;
    NmsWs ws = carve(d.workspace, d.B, d.A);
    if (int e = launch_nms_filter(d, ws, s)) return e;

    SelectParams sp;
    sp.pred = d.pred; sp.B = d.B; sp.A = d.A; sp.nc = d.nc; sp.iou = d.iou_thres; sp.max_det = d.max_det;
    sp.agnostic = d.agnostic; sp.ws = ws; sp.out = d.out; sp.counts = d.counts;
    sp.keep_anchor = reinterpret_cast<long long*>(d.keep_anchor);
    sp.scale = d.scale;
    sp.iou_lo = sp.iou_hi = 0.f;
    if (d.iou_thres > 1e-6 && d.iou_thres < 1e6) {
        sp.iou_lo = (float)(d.iou_thres * (1.0 - 1.0 / 262144.0));
        sp.iou_hi = (float)(d.iou_thres * (1.0 + 1.0 / 262144.0));
    }
    // opt in to the shared memory of the largest max_det check_nms accepts (227 520 B; sm_100 allows 232 448 B a block)
    static YrePerDeviceOnce once;
    if (int e = once.run([]() -> int {
            YRE_CUDA(cudaFuncSetAttribute(nms_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)select_smem_bytes(NMS_MAX_DET)));
            return YRE_OK;
        })) return e;
    nms_select_kernel<<<d.B, NT_SEL, select_smem_bytes(d.max_det), s>>>(sp);
    YRE_LAUNCH_CHECK("nms_select");
    return YRE_OK;
}

#ifdef YRE_TUNING
extern "C" int yre_debug_nms_prof(long long* host16) {
    cudaDeviceSynchronize();
    return cudaMemcpyFromSymbol(host16, g_nms_prof, sizeof(long long) * 16) == cudaSuccess ? 0 : -1;
}
#endif
