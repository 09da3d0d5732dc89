"""The fp16 precision on the device: every tcgen05 conv kernel per element against a float64 reference, the FFMA fallback,
the stem, pooling and layout kernels, the full-size plan teacher-forced launch by launch, detections, and properties of the
whole path.

Per-element conv bounds are the ones of tests/test_gpu_conv_tc_exact.py, with operands drawn there and rounded to fp16
instead of bf16.  fp16 x fp16 products are exact in fp32, as bf16 x bf16 products are, so the tensor cores accumulate the
same kind of exact products and the fp32 output obeys the same bound:
    |y_f32 - ref| <= 2^-14 A + s 2^-11 |pre| + 2^-22 (|pre| + |ref|),   A = conv(|x|, |w|) + |b|, s = 1 with SiLU,
and the fp16 output is the fp32 output rounded to nearest even, bit for bit.  The device must select the same TC_KERNELS
row as for the bf16 run of the case.

Worst log2(|y_f32 - ref| / A) per TC_KERNELS row over the cases, fp16 operands, NVIDIA B200 (148 SMs, power limit 1000 W),
within 0.3 of the bf16 file's figures:
    row  0: -21.13   row  1: -21.03   row  2: -19.78   row  3: -19.09   row  4: -19.58   row  5: -19.49   row  6: -20.80
    row  7: -21.05   row  8: -21.17   row  9: -21.05   row 10: -19.78   row 11: -19.09   row 12: -19.58   row 13: -19.49
    row 14: -20.76   row 16: -20.70   row 17: -20.87   row 18: -21.13   row 19: -20.52   row 20: -20.38

Full size, config 2: every launch is checked per element by tests/teacher_force.py, with the bounds derived there for
u = 2^-11, and one back-to-back run must reproduce every buffer bit for bit.

Detections against tests/golden/gelan-c_640_dets.npz: the fp16 head teacher-forced with the fp32 engine's neck features
recalls 0.999 of the reference's detections at precision 0.999; end to end fp16 recalls 0.681 at precision 0.682, where
bf16 recalls 0.123 at precision 0.123 in the same test.

Stem and ADown, derived from fp16 rounding (u = 2^-11, the unit roundoff of fp16):
  * stem (mma.sync on fp16 operands, fp32 accumulation, tanh.approx SiLU, one rounding of the output):
    |y - ref| <= u |ref| + s 2^-11 |pre| + 2^-20 A, with ref computed in float64 from the fp16-rounded image and weights;
  * ADown (three packed fp16 adds per 2x2 average, each rounding to fp16, and an exact x0.25; max is exact):
    |y - ref| <= 3 u avg(|x|) over the window, i.e. 2^-9.4 of the average of |x|, tested against 2^-9.
SPP, upsample, the NCHW <-> view conversions and CBFuse (fp32 sums in the kernel's order, one rounding) are exact."""
import ctypes as C
import math
import time
from collections import defaultdict

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from bench_data import make_inputs
from oracle import gelan_ref as G
from tests import teacher_force as TF
from tests.conftest import ROOT
from tests.conv_tc_cases import CASES, NUM_SMS, Case, desc, describe, row_key
from tests.test_gpu_conv_tc_exact import CHAINED, Operands, nan_buffer, ptrs, row_table, stream
from tests.test_gpu_round2 import BF16_HEAD_AGREEMENT, match_fraction

pytestmark = pytest.mark.gpu

import yolo_b200
from yolo_b200 import YOLO
from yolo_b200 import _lib as L
from yolo_b200 import engine as E

DEV = "cuda"
NAN = float("nan")
WORST = defaultdict(lambda: -math.inf)
GOLD = ROOT / "tests" / "golden"
U = 2.0 ** -11                     # unit roundoff of fp16
_INT = {torch.float16: torch.int16, torch.bfloat16: torch.int16, torch.float32: torch.int32}


def same_bits(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    return a.contiguous().view(_INT[a.dtype]) == b.contiguous().view(_INT[b.dtype])


def check_window(c: Case, y: torch.Tensor, what: str) -> torch.Tensor:
    fill = torch.full((), NAN, dtype=y.dtype, device=DEV)
    out = torch.cat((y[..., :c.y_off], y[..., c.y_off + c.Cout:]), -1)
    assert bool(same_bits(out, fill.expand_as(out)).all()), f"{what}: wrote outside its channel window"
    win = y[..., c.y_off:c.y_off + c.Cout]
    bad = (~torch.isfinite(win)).nonzero()
    assert bad.numel() == 0, f"{what}: {bad.shape[0]} non-finite outputs, first at {tuple(bad[0].tolist())}"
    return win


def f16_operands(c: Case, seed: int) -> Operands:
    """the operands of tests/test_gpu_conv_tc_exact.py (same draws), rounded to fp16 instead of bf16"""
    op = Operands.__new__(Operands)
    g = torch.Generator().manual_seed(seed)
    K = c.k * c.k * (c.Cin + c.cu)
    op.x = torch.randn((c.B, c.H, c.W, c.Cin), generator=g).half().to(DEV)
    op.xu = torch.randn((c.B, c.H // 2, c.W // 2, max(c.cu, 1)), generator=g).half().to(DEV)
    op.w = (torch.randn((c.Cout, c.k, c.k, c.Cin + c.cu), generator=g) * (2.5 / K ** 0.5)).half().to(DEV)
    op.b = (torch.rand((c.Cout,), generator=g) * 18 - 12).to(DEV) if c.bias else None
    r = torch.randn((c.B, c.Ho, c.Wo, c.Cout), generator=g) * 2
    op.res = None if c.res == "none" else r.to(torch.float32 if c.res == "f32" else torch.float16).to(DEV)
    return op


def f16_desc(c: Case, p: dict, y_f32: bool) -> L.ConvDesc:
    d = desc(c, p, y_f32=y_f32)
    for v in (d.x, d.y, d.res, d.xu):
        if v.ptr and v.dtype == L.BF16:
            v.dtype = L.F16
    return d


@pytest.fixture(scope="module", autouse=True)
def report():
    yield
    if WORST:
        print("\nfp16 operands: worst log2(|y_f32 - ref| / A) per TC_KERNELS row:")
        for r in sorted(WORST):
            print(f"  row {r:2d}: {WORST[r]:7.2f}")


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_fp16_tcgen05_conv_matches_fp64(case):
    c = case
    op = f16_operands(c, seed=1000 + CASES.index(c))
    ref, pre, A = op.reference(c)
    bufs = op.buffers(c, torch.float16)
    outs = {}
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    for f32 in (False, True):
        y = nan_buffer((c.B, c.Ho, c.Wo, c.yct), torch.float32 if f32 else torch.float16)
        d = f16_desc(c, ptrs(bufs, y, op.b), f32)
        expect = row_table().index(row_key(describe(desc(c, y_f32=f32), NUM_SMS)))     # the bf16 run's row
        assert row_table().index(row_key(describe(d, sms))) == expect, f"{c.name}: fp16 selects another kernel than bf16"
        L.check(L.lib().yre_conv(C.byref(d), stream()), f"yre_conv {c.name}")
        torch.cuda.synchronize()
        outs[f32] = (check_window(c, y, f"{c.name} {'fp32' if f32 else 'fp16'}"), expect)
    (yh, rowh), (y32, row32) = outs[False], outs[True]
    same = same_bits(yh, y32.to(torch.float16))
    if not bool(same.all()):
        i = tuple((~same).nonzero()[0].tolist())
        raise AssertionError(f"{c.name}: fp16 output differs from the rounded fp32 output in {int((~same).sum())} elements, "
                             f"first at {i}: {yh[i].item()} vs {y32[i].item():.9g}")
    worst = TF.check_bound(y32, ref, pre, A, c.silu, c.name)
    WORST[row32] = max(WORST[row32], worst)
    WORST[rowh] = max(WORST[rowh], worst)


@pytest.mark.parametrize("case,f32,row", CHAINED, ids=[f"row{r}-{c.name}-{'fp32' if f else 'fp16'}" for c, f, r in CHAINED])
def test_fp16_tcgen05_conv_waits_for_its_producer(case, f32, row):
    c = case
    lib = L.lib()
    op = f16_operands(c, seed=2000 + CASES.index(c))
    bufs = op.buffers(c, torch.float16)
    bufs["x"].fill_(NAN)
    g = torch.Generator().manual_seed(3000 + row)
    src = torch.randn((c.B, c.H, c.W, 512), generator=g).half().to(DEV)
    w1 = (torch.randn((c.Cin, 1, 1, 512), generator=g) / 512 ** 0.5).half().to(DEV)
    null = L.View(None, 0, 0, 0, 0, 0, 0, 0, 0)
    d1 = L.ConvDesc(L.View(src.data_ptr(), L.F16, L.NHWC, c.B, c.H, c.W, 512, 0, 512),
                    L.View(bufs["x"].data_ptr(), L.F16, L.NHWC, c.B, c.H, c.W, c.xct, c.x_off, c.Cin),
                    null, w1.data_ptr(), None, 1, 1, L.ACT_NONE, L.ENGINE_TCGEN05, null)
    y = nan_buffer((c.B, c.Ho, c.Wo, c.yct), torch.float32 if f32 else torch.float16)
    d2 = f16_desc(c, ptrs(bufs, y, op.b), f32)
    h = C.c_void_p()
    L.check(lib.yre_plan_create(C.byref(h)), "plan_create")
    try:
        L.check(lib.yre_plan_add_conv(h, C.byref(d1)), "plan_add_conv producer")
        L.check(lib.yre_plan_add_conv(h, C.byref(d2)), f"plan_add_conv {c.name}")
        assert lib.yre_plan_num_tcgen05(h) == 2
        L.check(lib.yre_plan_run(h, stream()), "plan_run")
        torch.cuda.synchronize()
    finally:
        lib.yre_plan_destroy(h)
    x = bufs["x"][..., c.x_off:c.x_off + c.Cin]
    assert bool(torch.isfinite(x).all()), f"{c.name}: the producer left part of the input window unwritten"
    ref, pre, A = op.reference(c, x=x)
    got = check_window(c, y, f"{c.name} after a producer")
    err = (got.double() - ref).abs()
    bound = 2.0 ** -14 * A + (2.0 ** -11 if c.silu else 0.0) * pre.abs() + 2.0 ** -22 * (pre.abs() + ref.abs())
    if not f32:
        bound = bound + U * ref.abs()          # plus half an ulp of fp16
    assert bool((err <= bound).all()), f"{c.name} after a producer: {int((err > bound).sum())} elements over the bound"


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_fp16_ffma_conv_matches_fp64(case):
    """the FFMA fallback on fp16 operands: fp32 output within the bf16 file's FFMA bound, fp16 output = rounded fp32"""
    c = case
    op = f16_operands(c, seed=1000 + CASES.index(c))
    ref, pre, A = op.reference(c)
    bufs = op.buffers(c, torch.float16)
    outs = []
    for f32 in (True, False):
        y = nan_buffer((c.B, c.Ho, c.Wo, c.yct), torch.float32 if f32 else torch.float16)
        d = f16_desc(c, ptrs(bufs, y, op.b), f32)
        d.engine = L.ENGINE_FFMA
        L.check(L.lib().yre_conv(C.byref(d), stream()), f"yre_conv ffma {c.name}")
        torch.cuda.synchronize()
        outs.append(check_window(c, y, f"{c.name} ffma"))
    TF.check_bound(outs[0], ref, pre, A, c.silu, f"{c.name} ffma", tc=False)
    assert bool(same_bits(outs[1], outs[0].to(torch.float16)).all()), f"{c.name} ffma: fp16 output != rounded fp32 output"


def check_planes(planes: torch.Tensor, nhwc: torch.Tensor, what: str):
    zero = torch.zeros((), dtype=planes.dtype, device=DEV)
    for py in (0, 1):
        for px in (0, 1):
            p = planes[py * 2 + px]
            sub = nhwc[:, py::2, px::2]
            h, w = sub.shape[1], sub.shape[2]
            assert bool(same_bits(p[:, :h, :w], sub).all()), f"{what}: plane {py * 2 + px} differs from the NHWC output"
            for rest in (p[:, h:], p[:, :, w:]):
                assert bool(same_bits(rest, zero.expand_as(rest)).all()), f"{what}: plane {py * 2 + px} cells without a source are not +0"


# (B, H, W, Cout, stride): the MMA stems (Cout 64: vectorised stride-2 for W % 4 == 0, scalar gather otherwise, stride 1)
# and the generic FMA stem (Cout 32)
STEMS = [(2, 45, 36, 64, 2), (2, 45, 37, 64, 2), (2, 33, 35, 32, 2), (2, 24, 20, 64, 1), (2, 45, 48, 64, 2)]


@pytest.mark.parametrize("Bn,H,W,Cout,stride", STEMS)
def test_fp16_stem(Bn, H, W, Cout, stride):
    """fp32 image and uint8 frames, NHWC and parity planes (odd output extents, zeroed edge cells), within the fp16 bound;
    the uint8 frames give the fp32-image output bit for bit"""
    g = torch.Generator().manual_seed(H * W + Cout + stride)
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    frames = torch.randint(0, 256, (Bn, H, W, 3), generator=g, dtype=torch.uint8)
    img = frames.flip(-1).permute(0, 3, 1, 2).contiguous().float() / 255.0
    w = torch.randn((Cout, 3, 3, 3), generator=g) * 0.3
    b = torch.randn((Cout,), generator=g)
    img_d, fr_d, w_d, b_d = img.to(DEV), frames.to(DEV), w.to(DEV), b.to(DEV)
    outs = {}
    for src in ("f32", "u8"):
        for layout in ((L.NHWC, L.PHASE4) if stride == 2 else (L.NHWC,)):
            shape = (Bn, Ho, Wo, Cout) if layout == L.NHWC else (4, Bn, (Ho + 1) // 2, (Wo + 1) // 2, Cout)
            y = nan_buffer(shape, torch.float16)
            d = L.StemDesc(img_d.data_ptr() if src == "f32" else None, Bn, 3, H, W,
                           L.View(y.data_ptr(), L.F16, layout, Bn, Ho, Wo, Cout, 0, Cout), w_d.data_ptr(), b_d.data_ptr(),
                           stride, L.ACT_SILU, fr_d.data_ptr() if src == "u8" else None)
            L.check(L.lib().yre_stem_conv(C.byref(d), stream()), "yre_stem_conv")
            torch.cuda.synchronize()
            outs[src, layout] = y
    got = outs["f32", L.NHWC]
    assert bool(torch.isfinite(got).all())
    if stride == 2:
        for src in ("f32", "u8"):
            check_planes(outs[src, L.PHASE4], outs[src, L.NHWC], f"stem {src} {H}x{W}")
    mma = Cout == 64
    if mma and stride == 2 and W % 16 == 0:
        # where the uint8 frames take the MMA kernel, fp16(v * (1/255)) == fp16(v / 255) makes them the fp32 image's twin
        assert bool(same_bits(outs["u8", L.NHWC], got).all())
    xr = img.half().double() if mma else img.double()
    wr = w.half().double() if mma else w.double()
    pre = F.conv2d(xr, wr.permute(0, 3, 1, 2), b.double(), stride=stride, padding=1)
    A = F.conv2d(xr.abs(), wr.abs().permute(0, 3, 1, 2), b.double().abs(), stride=stride, padding=1)
    ref = F.silu(pre)
    nhwc = lambda t: t.permute(0, 2, 3, 1).to(DEV)
    ref, pre, A = nhwc(ref), nhwc(pre), nhwc(A)
    bound = U * ref.abs() + 2.0 ** -11 * pre.abs() + 2.0 ** -20 * A
    if not mma:     # the FMA stem reads the fp32 image: only the output rounding and __expf / division in silu_f
        bound = U * ref.abs() + 2.0 ** -20 * A
    err = (got.double() - ref).abs()
    assert bool((err <= bound).all()), f"stem {H}x{W}: {int((err > bound).sum())} over the bound, worst {(err / bound).max():.3f}"


@pytest.mark.parametrize("Bn,H,W,Cn", [(2, 40, 38, 128), (3, 22, 36, 96), (1, 41, 39, 256)])
def test_fp16_adown(Bn, H, W, Cn):
    """tiled (packed fp16) and per-pixel kernels, NHWC and parity-plane averages, within 2^-9 of the averaged |x|"""
    g = torch.Generator().manual_seed(H + W + Cn)
    x = (torch.randn((Bn, H, W, Cn), generator=g) * 4).half().to(DEV)
    half, Ha, Wa = Cn // 2, H - 1, W - 1
    Ho, Wo = (Ha - 1) // 2 + 1, (Wa - 1) // 2 + 1
    xv = L.View(x.data_ptr(), L.F16, L.NHWC, Bn, H, W, Cn, 0, Cn)
    outs = {}
    for layout in (L.NHWC, L.PHASE4):
        lo = nan_buffer((Bn, Ha, Wa, half) if layout == L.NHWC else (4, Bn, (Ha + 1) // 2, (Wa + 1) // 2, half), torch.float16)
        hi = nan_buffer((Bn, Ho, Wo, half), torch.float16)
        L.check(L.lib().yre_adown_prepool(C.byref(xv), C.byref(L.View(lo.data_ptr(), L.F16, layout, Bn, Ha, Wa, half, 0, half)),
                                          C.byref(L.View(hi.data_ptr(), L.F16, L.NHWC, Bn, Ho, Wo, half, 0, half)), stream()), "adown")
        torch.cuda.synchronize()
        outs[layout] = (lo, hi)
    assert bool(same_bits(outs[L.PHASE4][1], outs[L.NHWC][1]).all())
    check_planes(outs[L.PHASE4][0], outs[L.NHWC][0], f"adown {H}x{W} C {Cn}")
    xn = x.double().permute(0, 3, 1, 2)
    avg, aabs = F.avg_pool2d(xn, 2, 1, 0), F.avg_pool2d(xn.abs(), 2, 1, 0)
    lo, hi = (t.double().permute(0, 3, 1, 2) for t in outs[L.NHWC])
    assert bool(((lo - avg[:, :half]).abs() <= 2.0 ** -9 * aabs[:, :half]).all())
    ref_hi = F.max_pool2d(avg[:, half:], 3, 2, 1)
    assert bool(((hi - ref_hi).abs() <= 2.0 ** -9 * F.max_pool2d(aabs[:, half:], 3, 2, 1)).all())


@pytest.mark.parametrize("Hs,Cn", [(20, 128), (40, 64), (13, 24)])
def test_fp16_spp_upsample_cbfuse_conversions_are_exact(Hs, Cn):
    """SPP (plane-resident max.f16x2 kernel, and the fp32-staged one for planes too large), upsample, CBFuse and the
    NCHW <-> view conversions, against torch on the same fp16 values"""
    g = torch.Generator().manual_seed(Hs * Cn)
    lib, s = L.lib(), stream()
    x = (torch.randn((2, Hs, Hs, Cn), generator=g) * 100).half().to(DEV)
    v = lambda t, H_, W_, C_: L.View(t.data_ptr(), L.F16, L.NHWC, t.shape[0], H_, W_, C_, 0, C_)
    ys = [torch.empty_like(x) for _ in range(3)]
    L.check(lib.yre_spp_maxpool(C.byref(v(x, Hs, Hs, Cn)), *[C.byref(v(y, Hs, Hs, Cn)) for y in ys], s), "spp")
    up = torch.empty((2, 2 * Hs, 2 * Hs, Cn), dtype=torch.float16, device=DEV)
    L.check(lib.yre_upsample2x(C.byref(v(x, Hs, Hs, Cn)), C.byref(v(up, 2 * Hs, 2 * Hs, Cn)), s), "upsample")
    tgt = (torch.randn((2, 2 * Hs, 2 * Hs, Cn), generator=g) * 100).half().to(DEV)
    fused = torch.empty_like(tgt)
    srcs = (L.View * 1)(v(x, Hs, Hs, Cn))
    L.check(lib.yre_cbfuse_sum(srcs, 1, C.byref(v(tgt, 2 * Hs, 2 * Hs, Cn)), C.byref(v(fused, 2 * Hs, 2 * Hs, Cn)), s), "cbfuse")
    img = torch.randn((2, Cn, Hs, Hs), generator=g).to(DEV) * 1000
    view = torch.empty((2, Hs, Hs, Cn), dtype=torch.float16, device=DEV)
    L.check(lib.yre_nchw_to_view(img.data_ptr(), C.byref(v(view, Hs, Hs, Cn)), s), "nchw_to_view")
    back = torch.empty((2, Cn, Hs, Hs), dtype=torch.float32, device=DEV)
    L.check(lib.yre_view_to_nchw(C.byref(v(view, Hs, Hs, Cn)), back.data_ptr(), s), "view_to_nchw")
    torch.cuda.synchronize()
    xn = x.float().permute(0, 3, 1, 2)
    for y, k in zip(ys, (5, 9, 13)):
        assert torch.equal(y.float().permute(0, 3, 1, 2), F.max_pool2d(xn, k, 1, k // 2)), f"spp {k}"
    assert torch.equal(up.float().permute(0, 3, 1, 2), F.interpolate(xn, scale_factor=2.0, mode="nearest"))
    ref = (F.interpolate(xn, scale_factor=2.0, mode="nearest") + tgt.float().permute(0, 3, 1, 2)).half()
    assert bool(same_bits(fused.permute(0, 3, 1, 2), ref).all())
    assert bool(same_bits(view.permute(0, 3, 1, 2), img.half()).all())
    assert torch.equal(back, view.float().permute(0, 3, 1, 2))


# ---- full size -------------------------------------------------------------------------------------------------------------
CONFIGS = {2: ("gelan-c", 640, 64), 5: ("gelan-c", 1280, 16), 4: ("yolov9-c", 640, 16)}


def _model(name, request, prec="fp16"):
    nodes, nc, sd = request.getfixturevalue("gelan_c" if name == "gelan-c" else "yolov9_c")
    m = YOLO.from_yaml(ROOT / "configs/models" / f"{name}.yaml")
    m.load_state_dict(sd, strict=True)
    return m.to(DEV).eval().set_precision(prec)


def test_fp16_every_launch_of_the_config2_plan_teacher_forced(request):
    name, img, Bn = CONFIGS[2]
    model = _model(name, request)
    x = make_inputs(Bn, img, seed=7).to(DEV)
    with torch.cuda.device(x.device):
        p = E.compile_model(model, x)
        names = [n for n, _ in p.op_table()]
        assert "conv_ffma" not in names
        t0 = time.perf_counter()
        worst = TF.teacher_force(p, label="fp16 config 2 ")
        t1 = time.perf_counter()
        TF.run_reproduces(p)
        print(f"fp16 config 2: {len(names)} launches checked per element in {t1 - t0:.1f} s, worst err / bound per kernel "
              f"family: {TF.report(worst)}; the back-to-back run reproduces every buffer")


@pytest.mark.parametrize("config", [2, 4, 5])
def test_fp16_full_size_outputs_are_finite_and_on_tcgen05(config, request):
    name, img, Bn = CONFIGS[config]
    model = _model(name, request)
    x = make_inputs(Bn, img, seed=7).to(DEV)
    y, raws = model(x)
    torch.cuda.synchronize()
    ys = y if isinstance(y, list) else [y]
    rs = [r for rr in raws for r in rr] if isinstance(y, list) else raws
    assert all(bool(torch.isfinite(t).all()) for t in ys + rs), f"config {config}: non-finite outputs in fp16"
    plan = next(iter(model._plans.values()))
    assert "conv_ffma" not in plan.op_variants()
    assert plan.num_tcgen05 == sum(1 for n, _ in plan.op_table() if n.startswith("conv"))
    feats = [v for v in plan.vals.values() if isinstance(v, E.V)]
    assert all(v.dtype in (L.F16, L.F32) for v in feats)


# ---- detections --------------------------------------------------------------------------------------------------------------
def test_fp16_detection_level_agreement(gelan_c):
    """against the reference's detections (tests/golden/gelan-c_640_dets.npz): the fp16 head teacher-forced with the fp32
    engine's neck features scores at least BF16_HEAD_AGREEMENT; end to end, fp16's recall and precision are at least
    bf16's minus 0.02, measured in the same test"""
    nodes, nc, sd = gelan_c
    gd = np.load(GOLD / "gelan-c_640_dets.npz")
    Bn, S = int(gd["batch"]), int(gd["size"])
    x = G.fractal(Bn, S, torch.Generator().manual_seed(int(gd["seed"]))).to(DEV)
    ref = [gd[f"det{i}"] for i in range(Bn)]

    def agreement(dets):
        return (float(np.mean([match_fraction(ref[i], dets[i]) for i in range(Bn)])),
                float(np.mean([match_fraction(dets[i], ref[i]) for i in range(Bn)])))

    def dets(y):
        return [d.cpu().numpy() for d in yolo_b200.non_max_suppression(y.permute(0, 2, 1), 0.25, 0.45)]

    m = YOLO.from_yaml(ROOT / "configs/models/gelan-c.yaml")
    m.load_state_dict(sd, strict=True)
    m = m.to(DEV).eval().set_precision("fp32")
    y32, _ = m(x)
    p32 = next(iter(m._plans.values()))
    det_name = list(m.layers.keys())[-1]
    feats = []
    for n in m.connections[det_name]:
        v = p32.vals[n]
        feats.append(v.t[..., v.c_off:v.c_off + v.C].float().permute(0, 3, 1, 2).contiguous())
    with yolo_b200.precision("fp16"):
        yh, _ = m.layers[det_name](feats)
    rh = agreement(dets(yh))
    res = {}
    for prec in ("bf16", "fp16"):
        y, _ = m.set_precision(prec)(x)
        res[prec] = agreement(dets(y))
    print(f"\nfp16 head (teacher-forced): recall {rh[0]:.3f} precision {rh[1]:.3f}; end to end: fp16 recall {res['fp16'][0]:.3f} "
          f"precision {res['fp16'][1]:.3f}, bf16 recall {res['bf16'][0]:.3f} precision {res['bf16'][1]:.3f}")
    assert rh[0] >= BF16_HEAD_AGREEMENT and rh[1] >= BF16_HEAD_AGREEMENT
    assert res["fp16"][0] >= res["bf16"][0] - 0.02 and res["fp16"][1] >= res["bf16"][1] - 0.02


# ---- whole path --------------------------------------------------------------------------------------------------------------
def test_fp16_uint8_frames_graph_and_precision_switch(gelan_c):
    nodes, nc, sd = gelan_c
    x = G.fractal(2, 256, torch.Generator().manual_seed(5))
    frames = (x.permute(0, 2, 3, 1).flip(-1) * 255.0).round().clamp(0, 255).to(torch.uint8).contiguous()
    xf = (frames.flip(-1).permute(0, 3, 1, 2).contiguous().float() / 255.0).to(DEV)
    m = YOLO.from_yaml(ROOT / "configs/models/gelan-c.yaml")
    m.load_state_dict(sd, strict=True)
    m = m.to(DEV).eval().set_precision("fp16")
    y_f, raws_f = m(xf)
    y_u, raws_u = m(frames.to(DEV))
    assert torch.equal(y_f, y_u) and all(torch.equal(a, b) for a, b in zip(raws_f, raws_u))
    # CUDA-graph replay equals eager
    m.fresh_outputs, m.use_cuda_graph = False, True
    y_g, _ = m(xf)
    y_g2, _ = m(xf)
    assert torch.equal(y_g, y_f) and torch.equal(y_g2, y_f)
    m.fresh_outputs, m.use_cuda_graph = True, False
    # switching precisions recompiles and gives each precision its own result
    out = {}
    for prec in ("bf16", "fp16", "fp32", "fp16", "bf16"):
        y, _ = m.set_precision(prec)(xf)
        if prec in out:
            assert torch.equal(y, out[prec]), prec
        out[prec] = y.clone()
    assert torch.equal(out["fp16"], y_f)
    assert not torch.equal(out["fp16"], out["bf16"])
    e16 = (out["fp16"] - out["fp32"]).abs().max().item()
    eb = (out["bf16"] - out["fp32"]).abs().max().item()
    print(f"\nmax |y - y_fp32|: fp16 {e16:.4g}, bf16 {eb:.4g}")


def test_fp16_yolov9c_dual_head_and_main_only(yolov9_c):
    """the dual head runs in fp16 (finite outputs), and main_only equals the dual model's main half bit for bit"""
    nodes, nc, sd = yolov9_c
    x = G.fractal(2, 128, torch.Generator().manual_seed(10)).to(DEV)
    m = YOLO.from_yaml(ROOT / "configs/models/yolov9-c.yaml")
    m.load_state_dict(sd, strict=True)
    m = m.to(DEV).eval().set_precision("fp16")
    (ya, ym), (ra, rm) = m(x)
    assert all(bool(torch.isfinite(t).all()) for t in [ya, ym, *ra, *rm])
    m.main_only = True
    y1, r1 = m(x)
    assert torch.equal(y1, ym) and all(torch.equal(a, b) for a, b in zip(r1, rm))
