// C ABI glue of libyre.so: error plumbing, standalone op entry points and the flat launch plan.
#include "yre_common.cuh"
#include <cstdlib>
#include <string>
#include <vector>
#include <new>

static thread_local char g_err[512] = "";

void yre_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

namespace {

enum OpKind { OP_CONV_FFMA, OP_CONV_TC, OP_STEM, OP_ADOWN, OP_SPP, OP_UP, OP_FUSE, OP_TO_VIEW, OP_TO_NCHW, OP_DECODE, OP_NMS, OP_DECODE_MASKS };

struct Op {
    OpKind kind;
    yre_conv_desc conv;
    ConvTcPlan* tc = nullptr;
    yre_stem_desc stem;
    yre_view v[10];
    int n_v = 0;
    const float* fin = nullptr;
    float* fout = nullptr;
    yre_decode_desc dec;
    yre_view mask[8];            // OP_DECODE_MASKS: the mask-tower views and mc (dec holds the rest)
    float* mc = nullptr;
    yre_nms_desc nms;
    double flops = 0.0;
};

// the batch an op was recorded for (the B of its views / descriptor)
int op_batch(const Op& o) {
    switch (o.kind) {
        case OP_CONV_FFMA:
        case OP_CONV_TC:   return o.conv.y.B;
        case OP_STEM:      return o.stem.y.B;
        case OP_DECODE:
        case OP_DECODE_MASKS: return o.dec.raw[0].B;
        case OP_NMS:       return o.nms.B;
        case OP_FUSE:      return o.v[1].B;
        default:           return o.v[0].B;
    }
}

// launches op o for its first nb images (nb == op_batch(o): the whole batch)
int run_op(Op& o, int nb, cudaStream_t s) {
    switch (o.kind) {
        case OP_CONV_FFMA: return launch_conv_ffma(o.conv, nb, s);
        case OP_CONV_TC:   return conv_tc_launch(o.tc, nb, s);
        case OP_STEM:      return launch_stem(o.stem, nb, s);
        case OP_ADOWN:     return launch_adown_prepool(o.v[0], o.v[1], o.v[2], nb, s);
        case OP_SPP:       return launch_spp_maxpool(o.v[0], o.v[1], o.v[2], o.v[3], nb, s);
        case OP_UP:        return launch_upsample2x(o.v[0], o.v[1], nb, s);
        case OP_FUSE:      return launch_cbfuse_sum(o.v + 2, o.n_v - 2, o.v[0], o.v[1], nb, s);
        case OP_TO_VIEW:   return launch_nchw_to_view(o.fin, o.v[0], nb, s);
        case OP_TO_NCHW:   return launch_view_to_nchw(o.v[0], o.fout, nb, s);
        case OP_DECODE:    return launch_decode(o.dec, nb, s);
        case OP_NMS:       return launch_nms(o.nms, nb, s);
        case OP_DECODE_MASKS: {
            yre_decode_masks_desc d;
            d.dec = o.dec; d.nm = 32; d.mc = o.mc;
            for (int l = 0; l < 8; ++l) d.mask[l] = o.mask[l];
            return launch_decode_masks(d, nb, s);
        }
    }
    return YRE_EINVAL;
}

const char* op_name(OpKind k) {
    switch (k) {
        case OP_CONV_FFMA: return "conv_ffma";
        case OP_CONV_TC:   return "conv_tc";
        case OP_STEM:      return "stem";
        case OP_ADOWN:     return "adown_prepool";
        case OP_SPP:       return "spp_maxpool";
        case OP_UP:        return "upsample2x";
        case OP_FUSE:      return "cbfuse_sum";
        case OP_TO_VIEW:   return "nchw_to_view";
        case OP_TO_NCHW:   return "view_to_nchw";
        case OP_DECODE:    return "dfl_decode_score";
        case OP_NMS:       return "nms";
        case OP_DECODE_MASKS: return "dfl_decode_masks";
    }
    return "?";
}

}  // namespace

// validates a conv descriptor for the plan, yre_conv and yre_conv_tc_describe
int check_conv(const yre_conv_desc* d) {
    if (!d || !d->w) YRE_FAIL(YRE_EINVAL, "conv: null descriptor/weights");
    if (yre_check_view(&d->x, "conv.x") || yre_check_view(&d->y, "conv.y")) return YRE_EINVAL;
    if (d->res.ptr && yre_check_view(&d->res, "conv.res")) return YRE_EINVAL;
    // bf16 and fp16 never mix: w has x's type, and a 16-bit y or residual must have the same one
    for (const yre_view* v : {&d->x, &d->y, &d->res})
        for (const yre_view* u : {&d->x, &d->y, &d->res})
            if (v->ptr && u->ptr && v->dtype != YRE_F32 && u->dtype != YRE_F32 && v->dtype != u->dtype)
                YRE_FAIL(YRE_EUNSUPPORTED, "conv: bf16 and fp16 operands mixed (x %d, y %d, res %d)", d->x.dtype, d->y.dtype,
                         d->res.ptr ? d->res.dtype : -1);
    if (d->k != 1 && d->k != 3) YRE_FAIL(YRE_EUNSUPPORTED, "conv: kernel size %d (1 or 3)", d->k);
    if (d->stride != 1 && d->stride != 2) YRE_FAIL(YRE_EUNSUPPORTED, "conv: stride %d (1 or 2)", d->stride);
    if (d->act != YRE_ACT_NONE && d->act != YRE_ACT_SILU) YRE_FAIL(YRE_EUNSUPPORTED, "conv: activation %d", d->act);
    const int pad = d->k / 2;
    const int Ho = (d->x.H + 2 * pad - d->k) / d->stride + 1, Wo = (d->x.W + 2 * pad - d->k) / d->stride + 1;
    if (d->y.H != Ho || d->y.W != Wo || d->y.B != d->x.B)
        YRE_FAIL(YRE_EINVAL, "conv: output extent %dx%d does not match input %dx%d k%d s%d", d->y.H, d->y.W, d->x.H, d->x.W, d->k, d->stride);
    if (d->y.layout != YRE_NHWC && d->engine == YRE_ENGINE_TCGEN05) YRE_FAIL(YRE_EUNSUPPORTED, "conv: tcgen05 engine writes NHWC only");
    if (d->res.ptr && (d->res.B != d->y.B || d->res.H != d->y.H || d->res.W != d->y.W || d->res.C != d->y.C))
        YRE_FAIL(YRE_EINVAL, "conv: residual shape mismatch");
    if (d->xu.ptr) {          // virtual cat([upsample2x(xu), x]) input
        if (yre_check_view(&d->xu, "conv.xu")) return YRE_EINVAL;
        if (d->k != 1 || d->stride != 1) YRE_FAIL(YRE_EUNSUPPORTED, "conv: an upsampled source needs a 1x1 stride-1 conv");
        if (d->xu.layout != YRE_NHWC || d->x.layout != YRE_NHWC || d->xu.dtype != d->x.dtype)
            YRE_FAIL(YRE_EUNSUPPORTED, "conv: upsampled source must be NHWC and of x's dtype");
        if (d->xu.B != d->x.B || 2 * d->xu.H != d->x.H || 2 * d->xu.W != d->x.W)
            YRE_FAIL(YRE_EINVAL, "conv: upsampled source %dx%d is not half of the input %dx%d", d->xu.H, d->xu.W, d->x.H, d->x.W);
    }
    return YRE_OK;
}

namespace {

// decides the engine; fills op
int make_conv_op(const yre_conv_desc* d, Op& o) {
    if (int e = check_conv(d)) return e;
    o.conv = *d;
    o.flops = conv_flops(*d);
    char why[256] = "";
    const bool elig = conv_tc_eligible(*d, why, sizeof(why)) != 0;
    if (d->engine == YRE_ENGINE_TCGEN05 && !elig) YRE_FAIL(YRE_EUNSUPPORTED, "conv: tcgen05 engine not eligible: %s", why);
    if (d->engine != YRE_ENGINE_FFMA && elig) {
        o.kind = OP_CONV_TC;
        return conv_tc_prepare(*d, &o.tc);
    }
    o.kind = OP_CONV_FFMA;
    return YRE_OK;
}

}  // namespace

struct yre_plan {
    std::vector<Op> ops;
    ~yre_plan() { for (auto& o : ops) if (o.tc) conv_tc_free(o.tc); }
};

extern "C" {

int yre_version(void) { return YRE_VERSION; }
const char* yre_last_error(void) { return g_err; }

int yre_device_check(void) {
    int dev = 0;
    YRE_CUDA(cudaGetDevice(&dev));
    cudaDeviceProp pr;
    YRE_CUDA(cudaGetDeviceProperties(&pr, dev));
    if (pr.major != 10) YRE_FAIL(YRE_EUNSUPPORTED, "device %d is sm_%d%d; libyre needs sm_100 (B200)", dev, pr.major, pr.minor);
    return YRE_OK;
}

int yre_conv(const yre_conv_desc* d, yre_stream_t s) {
    Op o;
    if (int e = make_conv_op(d, o)) return e;
    const int r = run_op(o, d->y.B, (cudaStream_t)s);
    if (o.tc) {   // the tensor maps are kernel parameters (copied at launch), safe to free now
        conv_tc_free(o.tc);
    }
    return r;
}

int yre_stem_conv(const yre_stem_desc* d, yre_stream_t s) {
    if (!d) YRE_FAIL(YRE_EINVAL, "stem: null descriptor");
    return launch_stem(*d, d->B, (cudaStream_t)s);
}
int yre_adown_prepool(const yre_view* x, const yre_view* lo, const yre_view* hi, yre_stream_t s) {
    if (!x || !lo || !hi) YRE_FAIL(YRE_EINVAL, "adown: null view");
    return launch_adown_prepool(*x, *lo, *hi, x->B, (cudaStream_t)s);
}
int yre_spp_maxpool(const yre_view* x, const yre_view* y5, const yre_view* y9, const yre_view* y13, yre_stream_t s) {
    if (!x || !y5 || !y9 || !y13) YRE_FAIL(YRE_EINVAL, "spp: null view");
    return launch_spp_maxpool(*x, *y5, *y9, *y13, x->B, (cudaStream_t)s);
}
int yre_upsample2x(const yre_view* x, const yre_view* y, yre_stream_t s) {
    if (!x || !y) YRE_FAIL(YRE_EINVAL, "upsample2x: null view");
    return launch_upsample2x(*x, *y, x->B, (cudaStream_t)s);
}
int yre_cbfuse_sum(const yre_view* srcs, int32_t n, const yre_view* t, const yre_view* y, yre_stream_t s) {
    if ((!srcs && n > 0) || !t || !y) YRE_FAIL(YRE_EINVAL, "cbfuse: null view");
    return launch_cbfuse_sum(srcs, n, *t, *y, y->B, (cudaStream_t)s);
}
int yre_nchw_to_view(const float* x, const yre_view* y, yre_stream_t s) {
    if (!y) YRE_FAIL(YRE_EINVAL, "nchw_to_view: null view");
    return launch_nchw_to_view(x, *y, y->B, (cudaStream_t)s);
}
int yre_view_to_nchw(const yre_view* x, float* y, yre_stream_t s) {
    if (!x) YRE_FAIL(YRE_EINVAL, "view_to_nchw: null view");
    return launch_view_to_nchw(*x, y, x->B, (cudaStream_t)s);
}
int yre_dfl_decode_score(const yre_decode_desc* d, yre_stream_t s) {
    if (!d) YRE_FAIL(YRE_EINVAL, "decode: null descriptor");
    return launch_decode(*d, d->raw[0].B, (cudaStream_t)s);
}
int yre_dfl_decode_score_masks(const yre_decode_masks_desc* d, yre_stream_t s) {
    if (!d) YRE_FAIL(YRE_EINVAL, "decode_masks: null descriptor");
    return launch_decode_masks(*d, d->dec.raw[0].B, (cudaStream_t)s);
}
int yre_nms_batched(const yre_nms_desc* d, yre_stream_t s) {
    if (!d) YRE_FAIL(YRE_EINVAL, "nms: null descriptor");
    return launch_nms(*d, d->B, (cudaStream_t)s);
}
int yre_nms_batched_multi_label(const yre_nms_desc* d, yre_stream_t s) {
    if (!d) YRE_FAIL(YRE_EINVAL, "nms: null descriptor");
    return launch_nms_multi_label(*d, d->B, (cudaStream_t)s);
}

// ---- plan -----------------------------------------------------------------------------------------
int yre_plan_create(yre_plan** out) {
    if (!out) YRE_FAIL(YRE_EINVAL, "plan_create: null out");
    *out = new (std::nothrow) yre_plan();
    if (!*out) YRE_FAIL(YRE_ENOMEM, "plan_create: out of memory");
    return YRE_OK;
}
void yre_plan_destroy(yre_plan* p) { delete p; }

#define PLAN_GUARD(p) if (!(p)) YRE_FAIL(YRE_EINVAL, "null plan")

// Tile-walk direction of the tcgen05 convs of a plan: 1 = alternate from one conv launch to the next (a layer then starts
// with what its producer wrote last, i.e. with what is still in L2), 0 = always first-to-last.
static int plan_rev_mode() {
#ifdef YRE_TUNING
    const char* v = getenv("YRE_TC_REV");
    if (v && *v) return atoi(v);
#endif
    return 0;
}

int yre_plan_add_conv(yre_plan* p, const yre_conv_desc* d) {
    PLAN_GUARD(p);
    Op o;
    if (int e = make_conv_op(d, o)) return e;
    if (o.tc && plan_rev_mode() == 1) {
        int n_tc = 0;
        for (const auto& q : p->ops) n_tc += q.kind == OP_CONV_TC;
        conv_tc_set_reverse(o.tc, n_tc & 1);
    }
    p->ops.push_back(o);
    return YRE_OK;
}
int yre_plan_add_stem(yre_plan* p, const yre_stem_desc* d) {
    PLAN_GUARD(p);
    if (!d) YRE_FAIL(YRE_EINVAL, "stem: null descriptor");
    Op o; o.kind = OP_STEM; o.stem = *d;
    o.flops = 2.0 * d->y.B * d->y.H * d->y.W * (double)d->y.C * d->Cin * 9;
    p->ops.push_back(o);
    return YRE_OK;
}
int yre_plan_add_adown_prepool(yre_plan* p, const yre_view* x, const yre_view* lo, const yre_view* hi) {
    PLAN_GUARD(p);
    if (!x || !lo || !hi) YRE_FAIL(YRE_EINVAL, "adown: null view");
    Op o; o.kind = OP_ADOWN; o.v[0] = *x; o.v[1] = *lo; o.v[2] = *hi; o.n_v = 3;
    p->ops.push_back(o);
    return YRE_OK;
}
int yre_plan_add_spp_maxpool(yre_plan* p, const yre_view* x, const yre_view* y5, const yre_view* y9, const yre_view* y13) {
    PLAN_GUARD(p);
    if (!x || !y5 || !y9 || !y13) YRE_FAIL(YRE_EINVAL, "spp: null view");
    Op o; o.kind = OP_SPP; o.v[0] = *x; o.v[1] = *y5; o.v[2] = *y9; o.v[3] = *y13; o.n_v = 4;
    p->ops.push_back(o);
    return YRE_OK;
}
int yre_plan_add_upsample2x(yre_plan* p, const yre_view* x, const yre_view* y) {
    PLAN_GUARD(p);
    if (!x || !y) YRE_FAIL(YRE_EINVAL, "upsample2x: null view");
    Op o; o.kind = OP_UP; o.v[0] = *x; o.v[1] = *y; o.n_v = 2;
    p->ops.push_back(o);
    return YRE_OK;
}
int yre_plan_add_cbfuse_sum(yre_plan* p, const yre_view* srcs, int32_t n, const yre_view* t, const yre_view* y) {
    PLAN_GUARD(p);
    if ((!srcs && n > 0) || !t || !y || n < 0 || n > 8) YRE_FAIL(YRE_EINVAL, "cbfuse: bad arguments");
    Op o; o.kind = OP_FUSE; o.v[0] = *t; o.v[1] = *y;
    for (int i = 0; i < n; ++i) o.v[2 + i] = srcs[i];
    o.n_v = 2 + n;
    p->ops.push_back(o);
    return YRE_OK;
}
int yre_plan_add_nchw_to_view(yre_plan* p, const float* x, const yre_view* y) {
    PLAN_GUARD(p);
    if (!x || !y) YRE_FAIL(YRE_EINVAL, "nchw_to_view: null argument");
    Op o; o.kind = OP_TO_VIEW; o.fin = x; o.v[0] = *y; o.n_v = 1;
    p->ops.push_back(o);
    return YRE_OK;
}
int yre_plan_add_view_to_nchw(yre_plan* p, const yre_view* x, float* y) {
    PLAN_GUARD(p);
    if (!x || !y) YRE_FAIL(YRE_EINVAL, "view_to_nchw: null argument");
    Op o; o.kind = OP_TO_NCHW; o.v[0] = *x; o.fout = y; o.n_v = 1;
    p->ops.push_back(o);
    return YRE_OK;
}
int yre_plan_add_decode(yre_plan* p, const yre_decode_desc* d) {
    PLAN_GUARD(p);
    if (!d) YRE_FAIL(YRE_EINVAL, "decode: null descriptor");
    Op o; o.kind = OP_DECODE; o.dec = *d;
    p->ops.push_back(o);
    return YRE_OK;
}
int yre_plan_add_decode_masks(yre_plan* p, const yre_decode_masks_desc* d) {
    PLAN_GUARD(p);
    if (!d) YRE_FAIL(YRE_EINVAL, "decode_masks: null descriptor");
    if (d->nm != 32) YRE_FAIL(YRE_EINVAL, "decode_masks: nm=%d (32 mask coefficients only)", d->nm);
    Op o; o.kind = OP_DECODE_MASKS; o.dec = d->dec; o.mc = d->mc;
    for (int l = 0; l < 8; ++l) o.mask[l] = d->mask[l];
    p->ops.push_back(o);
    return YRE_OK;
}
int yre_plan_add_nms(yre_plan* p, const yre_nms_desc* d) {
    PLAN_GUARD(p);
    if (!d) YRE_FAIL(YRE_EINVAL, "nms: null descriptor");
    Op o; o.kind = OP_NMS; o.nms = *d;
    p->ops.push_back(o);
    return YRE_OK;
}

int yre_plan_rebind(yre_plan* p, const void* old_ptr, void* new_ptr) {
    PLAN_GUARD(p);
    if (!old_ptr || !new_ptr) YRE_FAIL(YRE_EINVAL, "plan_rebind: null pointer");
    int n = 0;
    auto fix = [&](void*& f) { if (f == old_ptr) { f = new_ptr; ++n; } };
    auto fixc = [&](const void*& f) { if (f == old_ptr) { f = new_ptr; ++n; } };
    for (auto& o : p->ops) {
        switch (o.kind) {
            case OP_CONV_TC:
                if (o.conv.x.ptr == old_ptr || o.conv.w == old_ptr || (o.conv.xu.ptr && o.conv.xu.ptr == old_ptr))
                    YRE_FAIL(YRE_EUNSUPPORTED, "plan_rebind: buffer is baked into a TMA tensor map");
                {
                    const int r = conv_tc_rebind(o.tc, old_ptr, new_ptr);
                    if (r < 0) YRE_FAIL(YRE_EUNSUPPORTED, "plan_rebind: buffer is baked into a TMA tensor map");
                    n += r;
                }
                fix(o.conv.y.ptr); fix(o.conv.res.ptr);
                break;
            case OP_CONV_FFMA:
                fix(o.conv.x.ptr); fix(o.conv.y.ptr); fix(o.conv.res.ptr); fixc(o.conv.w);
                if (o.conv.xu.ptr) fix(o.conv.xu.ptr);
                break;
            case OP_STEM:
                if (o.stem.x_nchw == old_ptr) { o.stem.x_nchw = (const float*)new_ptr; ++n; }
                if (o.stem.x_u8_hwc == old_ptr) { o.stem.x_u8_hwc = (const uint8_t*)new_ptr; ++n; }
                fix(o.stem.y.ptr);
                break;
            case OP_DECODE:
            case OP_DECODE_MASKS:
                for (int l = 0; l < o.dec.levels; ++l) fix(o.dec.raw[l].ptr);
                if (o.dec.y == old_ptr) { o.dec.y = (float*)new_ptr; ++n; }
                if (o.kind == OP_DECODE_MASKS) {
                    for (int l = 0; l < o.dec.levels; ++l) fix(o.mask[l].ptr);
                    if (o.mc == old_ptr) { o.mc = (float*)new_ptr; ++n; }
                }
                break;
            case OP_NMS:
                if (o.nms.pred == old_ptr) { o.nms.pred = (const float*)new_ptr; ++n; }
                if (o.nms.out == old_ptr) { o.nms.out = (float*)new_ptr; ++n; }
                break;
            default:
                for (int i = 0; i < o.n_v; ++i) fix(o.v[i].ptr);
                if (o.fin == old_ptr) { o.fin = (const float*)new_ptr; ++n; }
                if (o.fout == old_ptr) { o.fout = (float*)new_ptr; ++n; }
                break;
        }
    }
    return n;
}

int yre_plan_run(yre_plan* p, yre_stream_t s) {
    PLAN_GUARD(p);
    for (auto& o : p->ops)
        if (int e = run_op(o, op_batch(o), (cudaStream_t)s)) return e;
    return YRE_OK;
}
int yre_plan_batch_capacity(const yre_plan* p) {
    PLAN_GUARD(p);
    if (p->ops.empty()) YRE_FAIL(YRE_EINVAL, "plan_batch_capacity: the plan has no ops");
    const int b = op_batch(p->ops[0]);
    for (size_t i = 1; i < p->ops.size(); ++i)
        if (op_batch(p->ops[i]) != b)
            YRE_FAIL(YRE_EINVAL, "plan_batch_capacity: op %zu (%s) was recorded for %d images, op 0 (%s) for %d", i,
                     op_name(p->ops[i].kind), op_batch(p->ops[i]), op_name(p->ops[0].kind), b);
    return b;
}
int yre_plan_run_batch(yre_plan* p, int32_t n, yre_stream_t s) {
    const int cap = yre_plan_batch_capacity(p);
    if (cap < 0) return cap;
    if (n < 1 || n > cap) YRE_FAIL(YRE_EINVAL, "plan_run_batch: %d images, the plan holds 1..%d", n, cap);
    for (auto& o : p->ops)
        if (int e = run_op(o, n, (cudaStream_t)s)) return e;
    return YRE_OK;
}
int yre_plan_run_op(yre_plan* p, int32_t i, yre_stream_t s) {
    PLAN_GUARD(p);
    if (i < 0 || (size_t)i >= p->ops.size()) YRE_FAIL(YRE_EINVAL, "plan_run_op: index %d out of range", i);
    return run_op(p->ops[i], op_batch(p->ops[i]), (cudaStream_t)s);
}
int yre_plan_num_ops(const yre_plan* p) { return p ? (int)p->ops.size() : 0; }
int yre_plan_num_launches(const yre_plan* p) {
    if (!p) return 0;
    int n = 0;
    for (auto& o : p->ops)     // NMS: 3 kernels; a stem writing parity planes of an odd extent zeroes their edge cells
        n += (o.kind == OP_NMS) ? 3 : (o.kind == OP_STEM && o.stem.y.layout == YRE_PHASE4 && ((o.stem.y.H | o.stem.y.W) & 1)) ? 2 : 1;
    return n;
}
int yre_plan_num_tcgen05(const yre_plan* p) {
    if (!p) return 0;
    int n = 0;
    for (auto& o : p->ops) n += o.kind == OP_CONV_TC;
    return n;
}
int yre_plan_op_flops(const yre_plan* p, double* flops, int32_t cap) {
    if (!p) return 0;
    for (size_t i = 0; i < p->ops.size() && (int)i < cap; ++i) flops[i] = p->ops[i].flops;
    return (int)p->ops.size();
}
const char* yre_plan_op_name(const yre_plan* p, int32_t i) {
    if (!p || i < 0 || (size_t)i >= p->ops.size()) return "";
    return op_name(p->ops[i].kind);
}
int yre_plan_op_variant(const yre_plan* p, int32_t i, char* out, int32_t cap) {
    if (!p || !out || cap <= 0 || i < 0 || (size_t)i >= p->ops.size()) return YRE_EINVAL;
    const Op& o = p->ops[i];
    if (o.kind == OP_CONV_TC && o.tc) conv_tc_describe(o.tc, out, (size_t)cap);
    else snprintf(out, (size_t)cap, "%s", op_name(o.kind));
    return YRE_OK;
}

}  // extern "C"
