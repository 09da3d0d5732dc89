"""Teacher-forced, per-element check of every launch of a compiled plan against float64 references (test helper).

`teacher_force(plan)` walks `plan.trace`.  For each op it snapshots the inputs that the op's outputs alias (an in-place
residual reads the buffer it writes), fills every output that aliases no input with NaN, runs `run_op(i)`, synchronizes
and checks every element of every output against a reference built from the exact operand values in the plan's
buffers.  The NaN fill makes an element the launch did not write fail the check.  References are computed on the
operands' device in float64, a slice of the batch at a time (at most `max_elems` elements per reference tensor), and
every slice is checked.  An op kind without a reference raises.  `run_reproduces(plan)` then requires one back-to-back
`plan.run()` to leave every buffer the plan owns bit for bit as the launch-by-launch pass left it.

u is the unit roundoff of the output type: bf16 2^-8, fp16 2^-11, fp32 2^-24.  Rounding a value v to the type changes
it by at most u |v|; for fp16 below 2^-14 the spacing is the subnormal one, so 2^-25 absolute is added (t16 below).
The bounds, per kernel family:

  * conv (tcgen05; fp32 accumulation of exact 16-bit products, fp32 epilogue, one rounding of the output):
        pre = conv(x [, upsample2x(xu)], w) + b,  ref = [res +] silu?(pre),  A = conv(|x|, |w|) + |b|,
        |y - ref| <= 2^-14 A + s 2^-11 |pre| + 2^-22 (|pre| + |ref|)  [+ u |ref| + t16 for a 16-bit output].
    The fp32 part is `check_bound` (derived in tests/test_gpu_conv_tc_exact.py: accumulation, tanh.approx SiLU with s = 1
    when the conv has one, bias and residual adds).  The 16-bit output is that fp32 value rounded once.  A is computed in
    fp32 with TF32 off: it only scales the bound.
  * stem (mma.sync on the image and weights rounded to the output's 16-bit type, fp32 accumulation, tanh.approx SiLU):
        |y - ref| <= u |ref| + s 2^-11 |pre| + 2^-20 A + t16,   ref from the rounded operands.
    K = 27 is padded to two k16 steps; each adds 16 exact products to the fp32 accumulator with one rounding (toward
    zero at worst, 2^-23 of the running sum), so with the bias add the accumulation error is below 3 * 2^-23 A = 2^-21.4 A.
    The SiLU term is the conv one.  The fp32 FMA stem (fp32 outputs, Cout != 64) reads the unrounded image: 27
    sequential FMAs and the bias add round 28 times, at most 28 * 2^-24 A = 2^-19.2 A, and silu_f (__expf and an IEEE
    division) adds 2^-21 |pre|; there the bound is u |ref| + 2^-18 A + t16.
  * ADown: lo = avg_pool2d(x, 2, 1, 0) over the first half of the channels, hi = max_pool2d(avg, 3, 2, 1) over the second.
    The 16-bit kernels sum the four pixels with three rounded adds.  Each rounds a partial sum bounded by the sum of
    |x|, so the error is below 3u(1 + u)^2 * 4 avg(|x|) before the exact x0.25.  Pairwise sums give (2u + u^2) instead,
    so the bound 4u avg(|x|) has a 2x margin there and covers a sequential order too.  The max of the computed
    averages is within the largest error in its window: hi is bounded by 4u max_pool(avg(|x|)).  fp16 adds 2^-23
    absolute, because subnormal sums and the x0.25 of a subnormal are inexact.  A parity-plane lo buffer must hold +0,
    bit for bit, in every cell without a source pixel: the stride-2 conv that reads it takes those cells as its zero
    padding.  The averaged map is (H-1) x (W-1), odd at every full-size level, so those cells exist.
  * SPP, upsample, the NCHW <-> view conversions and a CBFuse without sources (a concat copy): bit-exact against torch
    on the same values.
  * CBFuse: ref = sum_i nearest(src_i) + target, summed in fp32 in that order and rounded once.  With n sources the n + 1
    rounded adds stay below (n + 1) 2^-24 sum |terms|:  |y - ref| <= u |ref| + (n + 1) 2^-24 sum |terms| + t16.
  * decode: boxes (x, y, w, h) = dist2bbox of the softmax expectations e over 16 bins, times the level stride s, and
    scores sigmoid(z), against an fp64 restatement.
      - One expectation: __expf(d) for d = v - max <= 0 is within (2 + 1.17 |d|) ulp, at most (2 + 1.17 |d|) 2^-23
        relative.  Weighted by p_k = e^d_k / den, with den >= 1, and since e^-t t <= 1/e, these errors sum to at most
        (2 + 16 * 1.17 / e) 2^-23 = 2^-19.8 of the bins' weight.  As |w_k - e| <= 15 they move e by at most 2^-15.9.
        The 16-term fp32 sums of den and num each round 15 times on positive partial sums, (15 + 15) 2^-24 relative on
        e <= 15: 2^-15.2.  __fdividef adds 2 ulp of e <= 16: 2^-19.  Together 2^-14.4.
      - A width or height adds two expectations: 2^-13.4.  A centre averages two: 2^-14.4.  The 2^-14 s of the first
        draft of this bound is below that aligned worst case, so the constant is 2^-13.  The anchor coordinate
        a + 0.5 <= 160 and the roundings of a -/+ e, of the sum and of the product with s add 2^-23 (a_x + 15) per
        coordinate at most, inside 2^-21 (a_x + a_y) + 2^-13:
        |box - ref| <= s (2^-13 + 2^-21 (a_x + a_y)),  (a_x, a_y) the anchor centre in grid units.
      - Scores: __expf(-z) within (2 + 1.17 |z|) 2^-23 relative, which moves sigmoid by (1 - sigma) times that; 1 + E
        rounds once and __fdividef is within 2 ulp for 1 + E < 2^126.  At |z| <= 87.3 that is below 2^-16.2 sigma.
        Beyond, __fdividef returns 0 (or __expf overflows to inf) and sigma < 2^-126:
        |score - ref| <= 2^-15 sigma(z) + 2^-125.
Every output must be finite: a NaN or an infinity fails every bound.

What the bounds can see (tests/test_cpu_teacher_force.py checks each on the CPU): 2^-8 |y| added to one conv output
column before the 16-bit rounding, a bias skipped on a 16-channel tail, an average that drops a pixel, a nonzero
parity-plane edge cell, a CBFuse that rounds its partial sums, and a score or a box expectation computed from
bf16-rounded logits.

Measured worst log2(err / bound) per family and plan, NVIDIA B200 (148 SMs, power limit 1000 W).  A figure near 0 is
the bound's output-rounding term at work: a 16-bit result just above a power of two may sit half an ulp from its
reference, which is u |ref| to within a factor 1 + 2^-7.  Every plan's back-to-back run reproduced every buffer.
    plan                          conv   conv f32out  stem   adown  cbfuse  decode box  decode score
    config 2 bf16 64x640x640     -0.08      -7.71    -0.18  -1.02     -        -4.00       -4.13
    config 5 bf16 16x1280x1280   -0.08      -7.56    -0.18  -1.01     -        -3.50       -3.57
    config 4 bf16 16x640x640     -0.07      -7.62    -0.18  -1.02   -0.01      -4.15       -4.14
    config 2 fp16 64x640x640     -0.30      -7.41    -1.02  -1.02     -        -4.02       -4.17
    gelan-c bf16 64x384x640      -0.05      -8.03    -0.18  -1.02     -        -4.08       -5.20
    gelan-c fp16 64x384x640      -0.36      -7.81    -1.02  -1.03     -        -4.10       -5.20
    yolov9-c bf16 16x384x640     -0.05      -7.83    -0.18  -1.02   -0.01      -3.82       -5.26
    yolov9-c fp16 16x384x640     -0.34      -7.53    -1.02  -1.02   -0.00      -4.05       -5.23
SPP is bit-exact in every plan.  Scratch builds with one epilogue, decode or ADown change each fail this check:
2^-8 |f| added to output column 0 of every conv epilogue (op 1 of gelan-c bf16 64x384x640 already fails), scores
from bf16-rounded logits (19.5 M elements of the first level fail), and the parity-plane edge store of ADown skipped
(the first ADown fails).  The max-normalised loops this module replaced caught the first two, the first only through an
fp32-output conv, and passed the third.
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F

from yolo_b200 import _lib as L
from yolo_b200 import engine as E

UNIT = {L.BF16: 2.0 ** -8, L.F16: 2.0 ** -11, L.F32: 2.0 ** -24}
MAX_ELEMS = 1 << 27                      # elements per float64 reference tensor in one batch slice (1 GiB)
_INT = {1: torch.uint8, 2: torch.int16, 4: torch.int32, 8: torch.int64}
# op kind -> (input keys, output keys); "srcs" is a list of views
IO = {"conv": (("x", "xu", "res"), ("y",)), "stem": ((), ("y",)), "adown": (("x",), ("lo", "hi")),
      "spp": (("x",), ("y5", "y9", "y13")), "upsample": (("x",), ("y",)), "cbfuse": (("srcs", "target"), ("y",)),
      "decode": (("raws",), ("y",)), "nchw_to_view": ((), ("y",)), "view_to_nchw": (("x",), ("y",))}


# ---- bounds: pure functions of float64 tensors ----------------------------------------------------------------------
def _t16(dtype) -> float:
    return 2.0 ** -25 if dtype == L.F16 else 0.0


def conv_fp32_bound(ref, pre, A, silu: bool) -> torch.Tensor:
    return 2.0 ** -14 * A + (2.0 ** -11 if silu else 0.0) * pre.abs() + 2.0 ** -22 * (pre.abs() + ref.abs())


def conv_bound(ref, pre, A, silu: bool, dtype) -> torch.Tensor:
    b = conv_fp32_bound(ref, pre, A, silu)
    return b if dtype == L.F32 else b + UNIT[dtype] * ref.abs() + _t16(dtype)


def stem_bound(ref, pre, A, silu: bool, dtype, mma: bool) -> torch.Tensor:
    if not mma:
        return UNIT[dtype] * ref.abs() + 2.0 ** -18 * A + _t16(dtype)
    return UNIT[dtype] * ref.abs() + (2.0 ** -11 if silu else 0.0) * pre.abs() + 2.0 ** -20 * A + _t16(dtype)


def adown_bound(avg_abs, dtype) -> torch.Tensor:
    return 4.0 * UNIT[dtype] * avg_abs + (2.0 ** -23 if dtype == L.F16 else 0.0)


def cbfuse_bound(ref, terms_abs, n: int, dtype) -> torch.Tensor:
    return UNIT[dtype] * ref.abs() + (n + 1) * 2.0 ** -24 * terms_abs + _t16(dtype)


def box_bound(stride: float, ax, ay) -> torch.Tensor:
    return stride * (2.0 ** -13 + 2.0 ** -21 * (ax + ay))


def score_bound(sig) -> torch.Tensor:
    return 2.0 ** -15 * sig + 2.0 ** -125


def check_bound(got: torch.Tensor, ref, pre, A, silu: bool, what: str, tc: bool = True) -> float:
    """fp32 conv outputs: asserts the tcgen05 (tc) or FFMA per-element bound; returns the worst log2(err / A)"""
    err = (got.double() - ref).abs()
    bound = conv_fp32_bound(ref, pre, A, silu) if tc else 2.0 ** -19 * A + 2.0 ** -17 * ref.abs()
    over = err > bound
    if bool(over.any()):
        i = tuple(int(v) for v in torch.unravel_index((err / bound).argmax(), err.shape))
        raise AssertionError(f"{what}: {int(over.sum())} elements over the bound; worst at (b, y, x, c) = {i}: got "
                             f"{got[i].item():.9g}, ref {ref[i].item():.9g}, pre {pre[i].item():.6g}, A {A[i].item():.6g}, "
                             f"err / A = 2^{math.log2(err[i].item() / A[i].item()):.2f}")
    ratio = (err / A.clamp_min(1e-300)).max().item()
    return math.log2(ratio) if ratio > 0 else -math.inf


def within(got: torch.Tensor, ref: torch.Tensor, bound: torch.Tensor, what: str, b0: int = 0, dims="b, c, y, x") -> float:
    """asserts |got - ref| <= bound for every element (a non-finite output fails); returns max(err / bound).  b0 is the
    batch offset of the slice, added to the index in the message."""
    err = (got.double() - ref).abs()
    ok = err <= bound
    if not bool(ok.all()):
        r = torch.where(ok, torch.zeros_like(err), torch.nan_to_num(err / bound, nan=math.inf, posinf=math.inf))
        i = tuple(int(v) for v in torch.unravel_index(r.argmax(), r.shape))
        at = (i[0] + b0,) + i[1:]
        raise AssertionError(f"{what}: {int((~ok).sum())} elements over the bound; worst at ({dims}) = {at}: got "
                             f"{got[i].item():.9g}, ref {ref[i].item():.9g}, bound {bound[i].item():.3g}")
    r = torch.where(err == 0, torch.zeros_like(err), err / bound)
    return r.max().item() if r.numel() else 0.0


def exact(got: torch.Tensor, ref: torch.Tensor, what: str) -> float:
    assert got.shape == ref.shape and torch.equal(got, ref), f"{what}: differs from torch on the same values"
    return 0.0


# ---- views ----------------------------------------------------------------------------------------------------------
def window(v: E.V, b0: int, b1: int) -> torch.Tensor:
    """logical NHWC [b1 - b0, H, W, C] of a view, in the buffer's dtype"""
    if v.layout == L.NHWC:
        return v.t[b0:b1, :, :, v.c_off:v.c_off + v.C]
    t = v.t[:, b0:b1, :, :, v.c_off:v.c_off + v.C]
    out = t.new_empty((b1 - b0, v.H, v.W, v.C))
    for py in (0, 1):
        for px in (0, 1):
            sub = out[:, py::2, px::2]
            sub.copy_(t[py * 2 + px, :, :sub.shape[1], :sub.shape[2]])
    return out


def plane_edges(v: E.V, b0: int, b1: int) -> list[torch.Tensor]:
    """the cells of a parity-plane view that have no source pixel"""
    t = v.t[:, b0:b1, :, :, v.c_off:v.c_off + v.C]
    out = []
    for py in (0, 1):
        for px in (0, 1):
            h, w = (v.H - py + 1) // 2, (v.W - px + 1) // 2
            out += [t[py * 2 + px, :, h:], t[py * 2 + px, :, :h, w:]]
    return [e for e in out if e.numel()]


def nchw(t: torch.Tensor) -> torch.Tensor:
    return t.permute(0, 3, 1, 2)


def _views(a: dict, keys) -> list:
    out = []
    for k in keys:
        v = a.get(k)
        out += v if isinstance(v, list) else ([v] if v is not None else [])
    return out


def _overlap(p, q) -> bool:
    if not isinstance(p, E.V) or not isinstance(q, E.V) or p.t.data_ptr() != q.t.data_ptr():
        return False
    return p.c_off < q.c_off + q.C and q.c_off < p.c_off + p.C


def _frozen(v: E.V) -> E.V:
    t = v.t[..., v.c_off:v.c_off + v.C].clone()
    return E.V(t, v.B, v.H, v.W, v.C, 0, v.C, v.dtype, v.layout)


def _poison(o) -> None:
    if isinstance(o, E.V):
        o.t[..., o.c_off:o.c_off + o.C].fill_(math.nan)
    else:
        o.fill_(math.nan)


def _per_image(v) -> int:
    if isinstance(v, E.V):
        return v.H * v.W * v.C
    return v[0].numel() if isinstance(v, torch.Tensor) else 0


# ---- references, one batch slice [b0, b1) of one op -------------------------------------------------------------------
def stem_rounds_operands(a: dict) -> bool:
    """whether launch_stem (k_stem.cu) picks an mma.sync kernel, which rounds the image and weights to the output type"""
    y = a["y"]
    if y.dtype == L.F32 or y.C != 64:
        return False
    if a["u8"]:
        return a["stride"] == 2 and a["x"].shape[2] % 16 == 0
    return a["x"].shape[1] <= 3


def _conv(a, b0, b1, what):
    x = nchw(window(a["x"], b0, b1)).double()
    if a.get("xu") is not None:
        x = torch.cat((F.interpolate(nchw(window(a["xu"], b0, b1)).double(), scale_factor=2.0, mode="nearest"), x), 1)
    w, b, s, p = a["w"].double().permute(0, 3, 1, 2), a["b"].double(), a["stride"], a["k"] // 2
    pre = F.conv2d(x, w, b, s, p)
    A = F.conv2d(x.abs().float(), w.abs().float(), b.abs().float(), s, p).double()
    del x
    ref = F.silu(pre) if a["silu"] else pre
    if a["res"] is not None:
        ref = ref + nchw(window(a["res"], b0, b1)).double()
    y = a["y"]
    bound = conv_bound(ref, pre, A, a["silu"], y.dtype)
    fam = "conv f32out" if y.dtype == L.F32 else "conv"
    return {fam: within(nchw(window(y, b0, b1)), ref, bound, what, b0)}


def _stem(a, b0, b1, what):
    y = a["y"]
    if a["u8"]:     # BGR uint8 frames: the kernel's float(v) * (1/255), one fp32 rounding, and BGR -> RGB
        img = a["x"][b0:b1].flip(-1).permute(0, 3, 1, 2).float() * torch.tensor(1.0 / 255.0, dtype=torch.float32)
    else:
        img = a["x"][b0:b1].float()
    mma = stem_rounds_operands(a)
    tdt = E._TORCH_DT[y.dtype]
    x = (img.to(tdt) if mma else img).double()
    w = (a["w"].to(tdt) if mma else a["w"]).double().permute(0, 3, 1, 2)
    b = a["b"].double()
    pre = F.conv2d(x, w, b, a["stride"], 1)
    A = F.conv2d(x.abs(), w.abs(), b.abs(), a["stride"], 1)
    ref = F.silu(pre) if a["silu"] else pre
    out = {"stem": within(nchw(window(y, b0, b1)), ref, stem_bound(ref, pre, A, a["silu"], y.dtype, mma), what, b0)}
    if y.layout == L.PHASE4:
        _zero_edges(y, b0, b1, what)
    return out


def _zero_edges(v, b0, b1, what):
    for e in plane_edges(v, b0, b1):
        assert bool((e.contiguous().view(_INT[e.element_size()]) == 0).all()), \
            f"{what}: a parity-plane cell without a source pixel is not +0"


def _adown(a, b0, b1, what):
    x = nchw(window(a["x"], b0, b1)).double()
    half = x.shape[1] // 2
    avg, aabs = F.avg_pool2d(x, 2, 1, 0), F.avg_pool2d(x.abs(), 2, 1, 0)
    del x
    lo, hi = a["lo"], a["hi"]
    r1 = within(nchw(window(lo, b0, b1)), avg[:, :half], adown_bound(aabs[:, :half], lo.dtype), what + " avg", b0)
    if lo.layout == L.PHASE4:
        _zero_edges(lo, b0, b1, what + " avg")
    ref = F.max_pool2d(avg[:, half:], 3, 2, 1)
    r2 = within(nchw(window(hi, b0, b1)), ref, adown_bound(F.max_pool2d(aabs[:, half:], 3, 2, 1), hi.dtype), what + " max", b0)
    return {"adown": max(r1, r2)}


def _spp(a, b0, b1, what):
    x = nchw(window(a["x"], b0, b1)).float()
    for key, k in (("y5", 5), ("y9", 9), ("y13", 13)):
        exact(nchw(window(a[key], b0, b1)).float(), F.max_pool2d(x, k, 1, k // 2), f"{what} window {k}")
    return {"spp": 0.0}


def _upsample(a, b0, b1, what):
    ref = F.interpolate(nchw(window(a["x"], b0, b1)).float(), scale_factor=2.0, mode="nearest")
    return {"upsample": exact(nchw(window(a["y"], b0, b1)).float(), ref, what)}


def _cbfuse(a, b0, b1, what):
    tgt = nchw(window(a["target"], b0, b1)).float()
    got = nchw(window(a["y"], b0, b1))
    if not a["srcs"]:
        return {"copy": exact(got.float(), tgt, what)}
    size = tgt.shape[2:]
    terms = [F.interpolate(nchw(window(s, b0, b1)).float(), size=size, mode="nearest").double() for s in a["srcs"]] + [tgt.double()]
    ref = sum(terms[1:], terms[0])
    mag = sum((t.abs() for t in terms[1:]), terms[0].abs())
    return {"cbfuse": within(got, ref, cbfuse_bound(ref, mag, len(a["srcs"]), a["y"].dtype), what, b0)}


def decode_reference(z: torch.Tensor, stride: float, dfl_w):
    """z: raw logits [n, H, W, 64 + nc] of one level -> (boxes [n, H, W, 4], scores, anchor x, anchor y) in float64"""
    z = z.double()
    n, H, W, _ = z.shape
    e = (z[..., :64].reshape(n, H, W, 4, 16).softmax(-1) * torch.tensor(dfl_w, dtype=torch.float64, device=z.device)).sum(-1)
    gy, gx = torch.meshgrid(torch.arange(H, dtype=torch.float64, device=z.device) + 0.5,
                            torch.arange(W, dtype=torch.float64, device=z.device) + 0.5, indexing="ij")
    x1, y1, x2, y2 = gx - e[..., 0], gy - e[..., 1], gx + e[..., 2], gy + e[..., 3]
    box = torch.stack(((x1 + x2) / 2, (y1 + y2) / 2, x2 - x1, y2 - y1), -1) * stride
    return box, torch.sigmoid(z[..., 64:]), gx, gy


def _decode(a, b0, b1, what):
    y, a0, rb, rs = a["y"], 0, 0.0, 0.0
    for r, st in zip(a["raws"], a["strides"]):
        box, sig, gx, gy = decode_reference(window(r, b0, b1), st, a["dfl_w"])
        n, H, W, _ = box.shape
        got = y[b0:b1, a0:a0 + H * W].reshape(n, H, W, -1)
        a0 += H * W
        rb = max(rb, within(got[..., :4], box, box_bound(st, gx, gy)[..., None].expand_as(box), f"{what} boxes, stride {st:g}",
                            b0, "b, y, x, coordinate"))
        rs = max(rs, within(got[..., 4:], sig, score_bound(sig), f"{what} scores, stride {st:g}", b0, "b, y, x, class"))
    assert a0 == y.shape[1], f"{what}: {y.shape[1]} anchors in y, {a0} in the levels"
    return {"decode box": rb, "decode score": rs}


def _nchw_to_view(a, b0, b1, what):
    v = a["y"]
    ref = a["x"][b0:b1].permute(0, 2, 3, 1).to(E._TORCH_DT[v.dtype])
    return {"layout": exact(window(v, b0, b1).float(), ref.float(), what)}


def _view_to_nchw(a, b0, b1, what):
    return {"layout": exact(a["y"][b0:b1], nchw(window(a["x"], b0, b1)).float(), what)}


CHECK = {"conv": _conv, "stem": _stem, "adown": _adown, "spp": _spp, "upsample": _upsample, "cbfuse": _cbfuse,
         "decode": _decode, "nchw_to_view": _nchw_to_view, "view_to_nchw": _view_to_nchw}


# ---- the walk -----------------------------------------------------------------------------------------------------------
def teacher_force(plan, run_op=None, max_elems: int = MAX_ELEMS, label: str = "") -> dict[str, float]:
    """checks every element of every launch of the plan; returns the worst err / bound per kernel family (0 where the
    family is bit-exact).  run_op(i) runs op i (default plan.run_op, then a device synchronize)."""
    cuda = not plan.dry
    if run_op is None:
        def run_op(i):
            plan.run_op(i)
            torch.cuda.synchronize()
    descs = plan.op_descriptions()
    worst: dict[str, float] = {}
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        for i, (kind, a) in enumerate(plan.trace):
            if kind not in IO:
                raise ValueError(f"op {i}: no reference for the op kind {kind!r}")
            ins_k, outs_k = IO[kind]
            outs = _views(a, outs_k)
            a2 = dict(a)
            for k in ins_k:                      # inputs the op overwrites are read before it runs
                v = a.get(k)
                if isinstance(v, list):
                    a2[k] = [_frozen(s) if any(_overlap(s, o) for o in outs) else s for s in v]
                elif v is not None and any(_overlap(v, o) for o in outs):
                    a2[k] = _frozen(v)
            ins = _views(a, ins_k)
            for o in outs:
                if not any(_overlap(o, v) for v in ins):
                    _poison(o)
            run_op(i)
            per = max([_per_image(v) * (4 if k == "xu" else 1) for k in ins_k + outs_k for v in _views(a, (k,))]
                      + [_per_image(a["x"]) if kind in ("stem", "nchw_to_view") else 0] + [1])
            Bn = plan.batch
            step = max(1, min(Bn, max_elems // per))
            what = f"{label}op {i} ({descs[i]})"
            for b0 in range(0, Bn, step):
                for fam, r in CHECK[kind](a2, b0, min(Bn, b0 + step), what).items():
                    worst[fam] = max(worst.get(fam, 0.0), r)
            if cuda:
                torch.cuda.synchronize()
    finally:
        torch.backends.cudnn.allow_tf32 = old
    return worst


def report(worst: dict[str, float]) -> str:
    return ", ".join(f"{k} {'exact' if v == 0 else f'2^{math.log2(v):.2f}'}" for k, v in sorted(worst.items()))


# ---- back-to-back run ------------------------------------------------------------------------------------------------------
def digest(t: torch.Tensor, chunk: int = 1 << 26) -> torch.Tensor:
    """position-weighted sums of the bit patterns of t (int64, wrapping): a checksum for buffers too large to clone"""
    v = t.reshape(-1).view(_INT[t.element_size()])
    acc = torch.zeros(2, dtype=torch.int64, device=t.device)
    for c in range(0, v.numel(), chunk):
        x = v[c:c + chunk].long()
        i = torch.arange(c, c + x.numel(), dtype=torch.int64, device=t.device) * 2 + 1
        acc += torch.stack((x.sum(), (x * i).sum()))
    return acc


def snapshot(tensors: list[torch.Tensor], clone: bool) -> list[torch.Tensor]:
    return [t.clone() if clone else digest(t) for t in tensors]


def changed(tensors: list[torch.Tensor], snap: list[torch.Tensor], clone: bool) -> list[int]:
    """indices of the tensors whose bits differ from the snapshot"""
    out = []
    for j, (t, s) in enumerate(zip(tensors, snap)):
        it = _INT[t.element_size()]
        same = torch.equal(t.view(it), s.view(it)) if clone else torch.equal(digest(t), s)
        if not same:
            out.append(j)
    return out


def first_writers(plan) -> dict[int, int]:
    """data_ptr of a buffer -> index of the first op that writes it"""
    w = {}
    for i, (kind, a) in enumerate(plan.trace):
        for o in _views(a, IO.get(kind, ((), ()))[1]):
            w.setdefault((o.t if isinstance(o, E.V) else o).data_ptr(), i)
    return w


def run_reproduces(plan, run=None) -> None:
    """one plan.run() must leave every buffer of plan.keep (activations, outputs, weights) bit for bit as it is"""
    tensors = plan.keep
    nbytes = sum(t.numel() * t.element_size() for t in tensors)
    clone = plan.dry or nbytes < 0.5 * torch.cuda.mem_get_info()[0]
    snap = snapshot(tensors, clone)
    (run or plan.run)()
    if not plan.dry:
        torch.cuda.synchronize()
    bad = changed(tensors, snap, clone)
    if bad:
        writers = first_writers(plan)
        descs = plan.op_descriptions()
        ops = sorted((writers.get(tensors[j].data_ptr(), -1), j) for j in bad)
        lines = [f"buffer {j} {tuple(tensors[j].shape)} {tensors[j].dtype}: "
                 + (f"first written by op {i} ({descs[i]})" if i >= 0 else "written by no op (weights or bias)") for i, j in ops]
        raise AssertionError(f"the back-to-back run differs from the launch-by-launch run in {len(bad)} of {len(tensors)} "
                             f"buffers ({'clones' if clone else 'checksums'}); first differing op first:\n  " + "\n  ".join(lines))
