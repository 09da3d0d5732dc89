// K6: DFL softmax-integral box decode + anchor/stride generation + sigmoid class scoring.
//
//   reference: DetectDFL.forward tail   src/yolo/heads/detect.py:93-108
//              DFL.forward              src/yolo/heads/dfl.py:46-50
//              make_anchors/dist2bbox   src/yolo/heads/anchor.py:26-40, 57-64
//
// HBM-bound: per anchor it reads (64+nc) logits and writes 4+nc floats, nothing is reused.
// A CTA stages TILE anchors: the raw rows are fetched with fully coalesced 16-byte loads into
// shared memory, then one thread per (anchor, box side) does the 16-bin softmax expectation,
// sigmoid runs over the class logits, and the [TILE][4+nc] result leaves as one contiguous,
// coalesced block.  Anchor coordinates come from the anchor's linear index (no anchor tensor,
// no host sync).
// Segmentation heads (NM = 32, yre_dfl_decode_score_masks): the same launch also copies every anchor's NM mask coefficients
// from its level's mask-tower output into mc [B][A][NM], one coalesced 128-byte row per anchor.  Without YRE_DECODE_MASKS
// this file compiles the detection kernel, instruction for instruction.  The mask instantiations are compiled in their own
// translation unit (k_decode_masks.cu defines YRE_DECODE_MASKS and includes this file): ptxas allocates registers per
// module, and kernels added to this one would change the detection kernels' register assignment.
#include "yre_common.cuh"

namespace {

constexpr int TILE = 8;        // anchors per WARP; warps are independent (no block barrier anywhere)
constexpr int WARPS = 4;
constexpr int MAXL = 8;

struct DecodeParams {
    DView raw[MAXL];
    float stride[MAXL];
    int a_start[MAXL + 1];   // first anchor of every level
    int levels, nc, A, B;
    float dfl_w[16];
    float* y;
};

struct MaskParams {
    DView mask[MAXL];        // fp32 NHWC [B,Hl,Wl,>=NM] mask-tower outputs, levels as in DecodeParams::raw
    float* mc;               // [B][A][NM]
};

__device__ __forceinline__ float sigmoid_fast(float z) {      // ex2.approx + rcp.approx: ~3e-7 abs error
    return __fdividef(1.0f, 1.0f + __expf(-z));
}

// NC > 0: class count known at compile time (80 = COCO, the common case) so every index is a constant
// division; NC == 0: runtime class count.  With YRE_DECODE_MASKS the kernel also takes m and copies NM = 32
// coefficients per anchor (one per lane).
#ifdef YRE_DECODE_MASKS
constexpr int NM = 32;
#define DECODE_PARAMS const DecodeParams p, const MaskParams m
#define DECODE_ARGS p, m
#else
#define DECODE_PARAMS const DecodeParams p
#define DECODE_ARGS p
#endif
template <typename T, int NC>
__global__ void __launch_bounds__(WARPS * 32) decode_kernel(DECODE_PARAMS) {
    extern __shared__ __align__(16) float sm[];
    const int nc = NC > 0 ? NC : p.nc;
    const int CH = 64 + nc;                 // logits per raw row
    const int chunks = (CH + 3) / 4;        // 16-byte chunks per row (the last one may run into row padding when nc % 4 != 0)
    const int PITCH = chunks * 4 + 4;       // keeps 16B alignment, skews banks
    const int OC = 4 + nc;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* s_raw = sm + warp * (TILE * PITCH + TILE * OC);   // [TILE][PITCH]
    float* s_out = s_raw + TILE * PITCH;                      // [TILE][OC]

    const int tiles_per_img = (p.A + TILE - 1) / TILE;
    const long long wt = (long long)blockIdx.x * WARPS + warp;
    if (wt >= (long long)tiles_per_img * p.B) return;
    const int b = (int)(wt / tiles_per_img);
    const int a0 = (int)(wt % tiles_per_img) * TILE;
    const int na = min(TILE, p.A - a0);

    // ---- per-anchor geometry (lanes 0..TILE-1 own one anchor each) ----
    long long my_src = 0; int my_lvl = 0; float my_ax = 0.f, my_ay = 0.f, my_st = 0.f;
#ifdef YRE_DECODE_MASKS
    long long my_msrc = 0;                            // the anchor's pixel in its mask-tower view
#endif
    if (lane < na) {
        const int a = a0 + lane;
        int l = 0;
        while (l + 1 < p.levels && a >= p.a_start[l + 1]) ++l;
        const int r = a - p.a_start[l];
        const int W = p.raw[l].W;
        const int py = r / W, px = r - py * W;
        my_src = dview_pix(p.raw[l], b, py, px); my_lvl = l;
#ifdef YRE_DECODE_MASKS
        my_msrc = dview_pix(m.mask[l], b, py, px);
#endif
        my_ax = (float)px + 0.5f; my_ay = (float)py + 0.5f; my_st = p.stride[l];
    }
    const int total = na * chunks;
    // Fast path: the tile's anchors are consecutive pixels of ONE level whose view spans the whole buffer,
    // so their raw rows form one contiguous run of na*CH floats.  All loads of a lane are issued into
    // registers before the first shared-memory store (no load -> store -> load round-trip chain).
    const int lvl0 = __shfl_sync(0xffffffffu, my_lvl, 0), lvl1 = __shfl_sync(0xffffffffu, my_lvl, na - 1);
    const long long src0 = __shfl_sync(0xffffffffu, my_src, 0);
    constexpr int MAXQ = 10;                                  // one pass for nc <= 96 (9 loads per lane at nc = 80)
    if (lvl0 == lvl1 && p.raw[lvl0].C_total == chunks * 4) {
        const void* basep = p.raw[lvl0].ptr;
        for (int base0 = 0; base0 < total; base0 += 32 * MAXQ) {
            float4 buf[MAXQ];
#pragma unroll
            for (int q = 0; q < MAXQ; ++q) {
                const int i = base0 + q * 32 + lane;
                if (i < total) buf[q] = ld4<T>(basep, src0 + (long long)i * 4);
            }
#pragma unroll
            for (int q = 0; q < MAXQ; ++q) {
                const int i = base0 + q * 32 + lane;
                if (i < total) {
                    const int al = i / chunks, ck = i - al * chunks;
                    *reinterpret_cast<float4*>(s_raw + al * PITCH + ck * 4) = buf[q];
                }
            }
        }
    } else {
        for (int base0 = 0; base0 < total; base0 += 32) {        // rare: tile straddles two levels / windowed view
            const int i = base0 + lane;
            const bool act = i < total;
            const int al = act ? i / chunks : 0, ck = i - al * chunks;
            const long long src = __shfl_sync(0xffffffffu, my_src, al);
            const int lvl = __shfl_sync(0xffffffffu, my_lvl, al);
            if (act) *reinterpret_cast<float4*>(s_raw + al * PITCH + ck * 4) = ld4<T>(p.raw[lvl].ptr, src + ck * 4);
        }
    }
    __syncwarp();

    // ---- DFL expectation: lane = (anchor, side) ----
    float e = 0.f;
    {
        const int al = lane >> 2, side = lane & 3;
        if (al < na) {
            const float* z = s_raw + al * PITCH + side * 16;
            float v[16];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const float4 t = *reinterpret_cast<const float4*>(z + q * 4);
                v[q * 4] = t.x; v[q * 4 + 1] = t.y; v[q * 4 + 2] = t.z; v[q * 4 + 3] = t.w;
            }
            float mx = v[0];
#pragma unroll
            for (int k = 1; k < 16; ++k) mx = fmaxf(mx, v[k]);
            float den = 0.f, num = 0.f;
#pragma unroll
            for (int k = 0; k < 16; ++k) {
                const float ex = __expf(v[k] - mx);
                den += ex;
                num = fmaf(ex, p.dfl_w[k], num);
            }
            e = __fdividef(num, den);
        }
    }
    // ---- boxes: lane a (< TILE) gathers its four sides from lanes 4a..4a+3 ----
    {
        const int s0 = (lane & 7) * 4;
        const float e0 = __shfl_sync(0xffffffffu, e, s0), e1 = __shfl_sync(0xffffffffu, e, s0 + 1);
        const float e2 = __shfl_sync(0xffffffffu, e, s0 + 2), e3 = __shfl_sync(0xffffffffu, e, s0 + 3);
        if (lane < na) {
            const float x1 = my_ax - e0, y1 = my_ay - e1, x2 = my_ax + e2, y2 = my_ay + e3;
            float* o = s_out + lane * OC;
            o[0] = ((x1 + x2) / 2.f) * my_st;
            o[1] = ((y1 + y2) / 2.f) * my_st;
            o[2] = (x2 - x1) * my_st;
            o[3] = (y2 - y1) * my_st;
        }
    }
    // ---- class scores: float4 vectors, flat over (anchor, class/4) ----
    if ((nc & 3) == 0) {
        const int nc4 = nc / 4;
        for (int i = lane; i < na * nc4; i += 32) {
            const int al = i / nc4, c4 = i - al * nc4;
            const float4 z = *reinterpret_cast<const float4*>(s_raw + al * PITCH + 64 + c4 * 4);
            float4 r;
            r.x = sigmoid_fast(z.x); r.y = sigmoid_fast(z.y); r.z = sigmoid_fast(z.z); r.w = sigmoid_fast(z.w);
            *reinterpret_cast<float4*>(s_out + al * OC + 4 + c4 * 4) = r;
        }
    } else {                                // any class count (YOLO.from_yaml(num_classes=...)): scalar, rows are not 16-byte multiples
        for (int i = lane; i < na * nc; i += 32) {
            const int al = i / nc, c = i - al * nc;
            s_out[al * OC + 4 + c] = sigmoid_fast(s_raw[al * PITCH + 64 + c]);
        }
    }
    __syncwarp();

    // ---- contiguous coalesced store of na*OC floats ----
    float* dst = p.y + ((long long)b * p.A + a0) * OC;
    const int nfl = na * OC;
    if ((OC & 3) == 0 && ((a0 * OC) & 3) == 0) {
        for (int i = lane; i < nfl / 4; i += 32)
            reinterpret_cast<float4*>(dst)[i] = reinterpret_cast<const float4*>(s_out)[i];
    } else {
        for (int i = lane; i < nfl; i += 32) dst[i] = s_out[i];
    }

    // ---- mask coefficients: lane k copies coefficient k of each of the tile's anchors ----
#ifdef YRE_DECODE_MASKS
    {
        float v[TILE];
#pragma unroll
        for (int al = 0; al < TILE; ++al) {
            const long long src = __shfl_sync(0xffffffffu, my_msrc, al);
            const int lvl = __shfl_sync(0xffffffffu, my_lvl, al);
            if (al < na) v[al] = static_cast<const float*>(m.mask[lvl].ptr)[src + lane];
        }
        float* mdst = m.mc + ((long long)b * p.A + a0) * NM;
#pragma unroll
        for (int al = 0; al < TILE; ++al)
            if (al < na) mdst[al * NM + lane] = v[al];
    }
#endif
}

}  // namespace

// validates d and fills the kernel parameters, shared memory and grid of a decode launch for nb images
static int decode_setup(const yre_decode_desc& d, int nb, DecodeParams& p, size_t& smem, dim3& grid) {
    if (d.levels < 1 || d.levels > MAXL) YRE_FAIL(YRE_EINVAL, "decode: levels=%d", d.levels);
    if (!d.y) YRE_FAIL(YRE_EINVAL, "decode: null pointer");
    if (d.nc < 1) YRE_FAIL(YRE_EINVAL, "decode: nc=%d", d.nc);
    p.levels = d.levels; p.nc = d.nc; p.y = d.y;
    int A = 0;
    for (int l = 0; l < d.levels; ++l) {
        const yre_view& v = d.raw[l];
        if (yre_check_view(&v, "decode.raw")) return YRE_EINVAL;
        if (v.dtype == YRE_F16) YRE_FAIL(YRE_EUNSUPPORTED, "decode: raw logits must be fp32 or bf16 (level %d is fp16)", l);
        // rows are read as 16-byte chunks: the pixel pitch must be a multiple of 4 and, when nc % 4 != 0, leave room for the
        // last partial chunk (the host pads the raw buffer's channel count, engine.towers)
        if (v.layout != YRE_NHWC || v.C != 64 + d.nc || v.c_off % 4 || v.C_total % 4 || v.c_off + (64 + d.nc + 3) / 4 * 4 > v.C_total ||
            v.dtype != d.raw[0].dtype || v.B != d.raw[0].B)
            YRE_FAIL(YRE_EINVAL, "decode: level %d must be an NHWC [B,H,W,%d] view with a pixel pitch that is a multiple of 4", l, 64 + d.nc);
        p.raw[l] = make_dview(v);
        p.stride[l] = d.stride[l];
        p.a_start[l] = A;
        A += v.H * v.W;
    }
    p.a_start[d.levels] = A;
    p.A = A; p.B = nb;                               // rows of y and raw pixels are image-major
    for (int k = 0; k < 16; ++k) p.dfl_w[k] = d.dfl_w[k];
    const int CH4 = (64 + d.nc + 3) / 4 * 4, OC = 4 + d.nc;
    smem = (size_t)WARPS * (TILE * (CH4 + 4) + TILE * OC) * sizeof(float);
    const long long tiles = (long long)((A + TILE - 1) / TILE) * p.B;
    grid = dim3((unsigned)((tiles + WARPS - 1) / WARPS));
    if (smem > 200 * 1024) YRE_FAIL(YRE_EUNSUPPORTED, "decode: nc=%d too large for the staging tile", d.nc);
    return YRE_OK;
}

static int decode_launch(const yre_decode_desc& d, DECODE_PARAMS, size_t smem, dim3 grid, cudaStream_t s) {
    if (smem > 48 * 1024) {
        YRE_CUDA(cudaFuncSetAttribute(decode_kernel<float, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        YRE_CUDA(cudaFuncSetAttribute(decode_kernel<__nv_bfloat16, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
    const bool f32 = d.raw[0].dtype == YRE_F32;
    if (d.nc == 80) {
        if (f32) decode_kernel<float, 80><<<grid, WARPS * 32, smem, s>>>(DECODE_ARGS);
        else decode_kernel<__nv_bfloat16, 80><<<grid, WARPS * 32, smem, s>>>(DECODE_ARGS);
    } else {
        if (f32) decode_kernel<float, 0><<<grid, WARPS * 32, smem, s>>>(DECODE_ARGS);
        else decode_kernel<__nv_bfloat16, 0><<<grid, WARPS * 32, smem, s>>>(DECODE_ARGS);
    }
    #ifdef YRE_DECODE_MASKS
    YRE_LAUNCH_CHECK("dfl_decode_masks");
#else
    YRE_LAUNCH_CHECK("dfl_decode_score");
#endif
    return YRE_OK;
}

#ifndef YRE_DECODE_MASKS
int launch_decode(const yre_decode_desc& d, int nb, cudaStream_t s) {
    DecodeParams p;
    size_t smem;
    dim3 grid;
    if (int e = decode_setup(d, nb, p, smem, grid)) return e;
    return decode_launch(d, p, smem, grid, s);
}
#else

int launch_decode_masks(const yre_decode_masks_desc& d, int nb, cudaStream_t s) {
    DecodeParams p;
    size_t smem;
    dim3 grid;
    if (int e = decode_setup(d.dec, nb, p, smem, grid)) return e;
    if (d.nm != 32) YRE_FAIL(YRE_EINVAL, "decode_masks: nm=%d (32 mask coefficients only)", d.nm);
    if (!d.mc) YRE_FAIL(YRE_EINVAL, "decode_masks: null mc");
    MaskParams m;
    m.mc = d.mc;
    for (int l = 0; l < d.dec.levels; ++l) {
        const yre_view& v = d.mask[l];
        if (yre_check_view(&v, "decode_masks.mask")) return YRE_EINVAL;
        if (v.layout != YRE_NHWC || v.dtype != YRE_F32 || v.C != d.nm || v.B != d.dec.raw[l].B || v.H != d.dec.raw[l].H ||
            v.W != d.dec.raw[l].W)
            YRE_FAIL(YRE_EINVAL, "decode_masks: mask level %d must be an fp32 NHWC [B,H,W,%d] view of raw level %d's extent", l,
                     d.nm, l);
        m.mask[l] = make_dview(v);
    }
    return decode_launch(d.dec, p, m, smem, grid, s);
}
#endif
