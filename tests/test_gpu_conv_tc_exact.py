"""Per-element check of every tcgen05 conv kernel against a float64 reference (cases: tests/conv_tc_cases.py).

Each case runs through `yre_conv` on the tcgen05 engine twice: once with a bf16 output and once with an fp32 output.
Both y buffers are wider than their channel window and are NaN-filled first.  So are the channels around the x and
residual windows, so a read outside a window also shows up as a NaN.  The bias is spread over [-12, 6], which puts the
pre-activations over about [-20, 8] and tests the negative tail of the SiLU.  For every element:
  * the window is finite, and every channel outside it still holds the NaN fill, bit for bit;
  * y_bf16 == y_f32.to(bfloat16), bit for bit.  The epilogue computes the same fp32 value for both outputs and rounds
    it once, to nearest even.  The MMA order of a tile does not depend on the output dtype;
  * |y_f32 - ref| <= 2^-14 A + s 2^-11 |pre| + 2^-22 (|pre| + |ref|).  Here pre = conv(x, w) + b, A = conv(|x|, |w|) + |b|,
    and s = 1 with SiLU.  The first term covers fp32 accumulation in the tensor cores.  Sequential round-to-nearest
    accumulation of bf16 products stays below 2^-23 A, and round-toward-zero reaches 2^-17.7 A at K = 9216.  A dropped
    64-channel K chunk gives a median error of 2^-9.8 A at K = 9216.  The second term covers the SiLU's tanh.approx:
    2^-10.987 relative on tanh, times |pre| / 2, with a 2x margin.  The third covers the bias and residual adds.
The kernel each run uses (`yre_conv_tc_describe` at the device's SM count) must be the TC_KERNELS row that the CPU
coverage test expects at 148 SMs.

What the bound can see: an error of 2^-8 |y| in one output column, a skipped bias or a bf16 round trip of an fp32 output
fails it.  A perturbation near 2^-12 |y| can hide under the accumulation term when K is long, because A grows with K
while |y| does not.

Worst log2(|y_f32 - ref| / A) per TC_KERNELS row over the cases, NVIDIA B200 (148 SMs, power limit 1000 W).  Rows
10-13 are the fp32 runs of the cases of rows 0-5 and show the same figures; the largest ratios come from short-K 1x1
convs, where the tanh.approx error, which scales with |pre|, is a larger share of A:
    row  0: -21.25   row  1: -21.20   row  2: -19.81   row  3: -19.10   row  4: -19.59   row  5: -19.45   row  6: -21.08
    row  7: -21.15   row  8: -21.14   row  9: -21.23   row 10: -19.81   row 11: -19.10   row 12: -19.59   row 13: -19.45
    row 14: -20.88   row 16: -20.73   row 17: -20.85   row 18: -21.06   row 19: -20.51   row 20: -20.33
No row comes near 2^-16, where the error would be more than rounding.

Epilogue mutations, each built from a scratch copy of the sources, all fail test_tcgen05_conv_matches_fp64:
  * pack_bf16x2 rounding toward zero: all 40 cases (bf16 output != rounded fp32 output);
  * 2^-8 |f| added to output column 0: 38 of 40 cases (fp32 bound);
  * the bias skipped in the 16-column tail: all 10 cases that have such a tail and a bias (fp32 bound).

The file also checks:
  * chained launches: one case per row with an NHWC input runs as the second conv of a two-conv plan.  The first conv
    writes that case's NaN-filled input window.  This tests each kernel's programmatic-dependent-launch wait before its
    first activation read;
  * the FFMA validation engine on the same cases with fp32 operands: |y - ref| <= 2^-19 A + 2^-17 |ref|.  This is
    derived from its sequential fp32 FMAs (the products of bf16-valued operands are exact), __expf and the IEEE division
    of silu_f;
  * the producers of parity-plane (PHASE4) inputs, yre_stem_conv and yre_adown_prepool, on odd extents: every cell that
    has a source pixel equals the NHWC output bit for bit, and every cell without one is +0."""
import ctypes as C
import math
from collections import defaultdict

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from tests.conv_tc_cases import CASES, NUM_SMS, Case, desc, describe, row_key
from tests.teacher_force import check_bound, conv_fp32_bound

from yolo_b200 import _lib as L

DEV = "cuda"
NAN = float("nan")
WORST = defaultdict(lambda: -math.inf)        # row -> worst log2(err / A) over the runs of this module


def row_table():
    from tests.test_cpu_conv_tc_coverage import KEYS
    return KEYS


def stream():
    return torch.cuda.current_stream().cuda_stream


def same_bits(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    it = {torch.bfloat16: torch.int16, torch.float32: torch.int32}[a.dtype]
    return a.contiguous().view(it) == b.contiguous().view(it)


def nan_buffer(shape, dtype):
    return torch.full(shape, NAN, dtype=dtype, device=DEV)


def to_phase4(x: torch.Tensor, ct: int, off: int) -> torch.Tensor:
    """parity planes [4][B][Hp][Wp][ct] of the logical NHWC map x in channels [off, off + C); cells without a source pixel
    hold zeros in the window, everything outside the window is NaN"""
    Bn, H, W, Cn = x.shape
    buf = nan_buffer((4, Bn, (H + 1) // 2, (W + 1) // 2, ct), x.dtype)
    buf[..., off:off + Cn] = 0
    for py in (0, 1):
        for px in (0, 1):
            sub = x[:, py::2, px::2]
            buf[py * 2 + px, :, :sub.shape[1], :sub.shape[2], off:off + Cn] = sub
    return buf


class Operands:
    """Seeded operands of one case: logical tensors on the device and the float64 reference."""

    def __init__(self, c: Case, seed: int):
        g = torch.Generator().manual_seed(seed)
        K = c.k * c.k * (c.Cin + c.cu)
        self.x = torch.randn((c.B, c.H, c.W, c.Cin), generator=g).bfloat16().to(DEV)
        self.xu = torch.randn((c.B, c.H // 2, c.W // 2, max(c.cu, 1)), generator=g).bfloat16().to(DEV)
        self.w = (torch.randn((c.Cout, c.k, c.k, c.Cin + c.cu), generator=g) * (2.5 / K ** 0.5)).bfloat16().to(DEV)
        self.b = (torch.rand((c.Cout,), generator=g) * 18 - 12).to(DEV) if c.bias else None
        r = torch.randn((c.B, c.Ho, c.Wo, c.Cout), generator=g) * 2
        self.res = None if c.res == "none" else r.to(torch.float32 if c.res == "f32" else torch.bfloat16).to(DEV)

    def reference(self, c: Case, x: torch.Tensor | None = None):
        """(ref, pre, A) in float64, NHWC; x overrides the logical input"""
        x = self.x if x is None else x
        inp = x.double().permute(0, 3, 1, 2)
        if c.cu:
            inp = torch.cat((F.interpolate(self.xu.double().permute(0, 3, 1, 2), scale_factor=2.0, mode="nearest"), inp), 1)
        w = self.w.double().permute(0, 3, 1, 2)
        b = self.b.double() if self.b is not None else torch.zeros(c.Cout, dtype=torch.float64, device=DEV)
        pre = F.conv2d(inp, w, b, stride=c.stride, padding=c.k // 2)
        A = F.conv2d(inp.abs(), w.abs(), b.abs(), stride=c.stride, padding=c.k // 2)
        ref = F.silu(pre) if c.silu else pre
        if self.res is not None:
            ref = ref + self.res.double().permute(0, 3, 1, 2)
        nhwc = lambda t: t.permute(0, 2, 3, 1)
        return nhwc(ref), nhwc(pre), nhwc(A)

    def buffers(self, c: Case, dt=torch.bfloat16) -> dict:
        """device buffers in the case's layout (x, xu and w in dtype dt): windows inside NaN-filled wider buffers"""
        if c.phase4:
            x = to_phase4(self.x.to(dt), c.xct, c.x_off)
        else:
            x = nan_buffer((c.B, c.H, c.W, c.xct), dt)
            x[..., c.x_off:c.x_off + c.Cin] = self.x.to(dt)
        bufs = dict(x=x, xu=self.xu.to(dt), w=self.w.to(dt).contiguous())
        if self.res is not None:
            res = nan_buffer((c.B, c.Ho, c.Wo, c.yct), self.res.dtype)
            res[..., c.y_off:c.y_off + c.Cout] = self.res
            bufs["res"] = res
        return bufs


def ptrs(bufs: dict, y: torch.Tensor, b) -> dict:
    return dict(x=bufs["x"].data_ptr(), y=y.data_ptr(), res=bufs["res"].data_ptr() if "res" in bufs else None,
                w=bufs["w"].data_ptr(), bias=b.data_ptr() if b is not None else None, xu=bufs["xu"].data_ptr())


def check_window(c: Case, y: torch.Tensor, what: str) -> torch.Tensor:
    """the output window (finite); the channels around it must still hold the NaN fill"""
    fill = torch.full((), NAN, dtype=y.dtype, device=DEV)
    out = torch.cat((y[..., :c.y_off], y[..., c.y_off + c.Cout:]), -1)
    assert bool(same_bits(out, fill.expand_as(out)).all()), f"{what}: wrote outside its channel window"
    win = y[..., c.y_off:c.y_off + c.Cout]
    bad = (~torch.isfinite(win)).nonzero()
    assert bad.numel() == 0, f"{what}: {bad.shape[0]} non-finite outputs, first at (b, y, x, c) = {tuple(bad[0].tolist())}"
    return win


def device_row(d: L.ConvDesc) -> int:
    return row_table().index(row_key(describe(d, torch.cuda.get_device_properties(0).multi_processor_count)))


@pytest.fixture(scope="module", autouse=True)
def report():
    yield
    if WORST:
        print("\nworst log2(|y_f32 - ref| / A) per TC_KERNELS row:")
        for r in sorted(WORST):
            print(f"  row {r:2d}: {WORST[r]:7.2f}")


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_tcgen05_conv_matches_fp64(case):
    c = case
    op = Operands(c, seed=1000 + CASES.index(c))
    ref, pre, A = op.reference(c)
    bufs = op.buffers(c)
    outs = {}
    for f32 in (False, True):
        y = nan_buffer((c.B, c.Ho, c.Wo, c.yct), torch.float32 if f32 else torch.bfloat16)
        d = desc(c, ptrs(bufs, y, op.b), y_f32=f32)
        expect = row_table().index(row_key(describe(d, NUM_SMS)))
        assert device_row(d) == expect, f"{c.name}: the device selects another kernel than the CPU coverage test expects"
        L.check(L.lib().yre_conv(C.byref(d), stream()), f"yre_conv {c.name}")
        torch.cuda.synchronize()
        outs[f32] = (check_window(c, y, f"{c.name} {'fp32' if f32 else 'bf16'}"), expect)
    (y16, _), (y32, row32) = outs[False], outs[True]
    same = same_bits(y16, y32.to(torch.bfloat16))
    if not bool(same.all()):
        i = tuple((~same).nonzero()[0].tolist())
        raise AssertionError(f"{c.name}: bf16 output differs from the rounded fp32 output in {int((~same).sum())} elements, "
                             f"first at {i}: {y16[i].item()} vs {y32[i].item():.9g}")
    worst = check_bound(y32, ref, pre, A, c.silu, c.name)
    WORST[row32] = max(WORST[row32], worst)
    WORST[outs[False][1]] = max(WORST[outs[False][1]], worst)


def chained_cases():
    """one (case, fp32 output) per reachable row with an NHWC input, first in list order"""
    seen, out = set(), []
    for c in CASES:
        if c.phase4:
            continue
        for f32 in (False, True):
            r = row_table().index(row_key(describe(desc(c, y_f32=f32))))
            if r not in seen:
                seen.add(r)
                out.append((c, f32, r))
    return out


CHAINED = chained_cases()


@pytest.mark.parametrize("case,f32,row", CHAINED, ids=[f"row{r}-{c.name}-{'fp32' if f else 'bf16'}" for c, f, r in CHAINED])
def test_tcgen05_conv_waits_for_its_producer(case, f32, row):
    c = case
    lib = L.lib()
    op = Operands(c, seed=2000 + CASES.index(c))
    bufs = op.buffers(c)
    bufs["x"].fill_(NAN)                        # the whole input buffer; the producer writes the window
    g = torch.Generator().manual_seed(3000 + row)
    src = torch.randn((c.B, c.H, c.W, 512), generator=g).bfloat16().to(DEV)
    w1 = (torch.randn((c.Cin, 1, 1, 512), generator=g) / 512 ** 0.5).bfloat16().to(DEV)
    d1 = L.ConvDesc(L.View(src.data_ptr(), L.BF16, L.NHWC, c.B, c.H, c.W, 512, 0, 512),
                    L.View(bufs["x"].data_ptr(), L.BF16, L.NHWC, c.B, c.H, c.W, c.xct, c.x_off, c.Cin),
                    L.View(None, 0, 0, 0, 0, 0, 0, 0, 0), w1.data_ptr(), None, 1, 1, L.ACT_NONE, L.ENGINE_TCGEN05,
                    L.View(None, 0, 0, 0, 0, 0, 0, 0, 0))
    y = nan_buffer((c.B, c.Ho, c.Wo, c.yct), torch.float32 if f32 else torch.bfloat16)
    d2 = desc(c, ptrs(bufs, y, op.b), y_f32=f32)
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
    if f32:
        check_bound(got, ref, pre, A, c.silu, f"{c.name} after a producer")
    else:   # a bf16 output: the fp32 bound plus half an ulp of bf16
        err = (got.double() - ref).abs()
        bound = conv_fp32_bound(ref, pre, A, c.silu) + 2.0 ** -8 * ref.abs()
        assert bool((err <= bound).all()), f"{c.name} after a producer: {int((err > bound).sum())} elements over the bound"


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_ffma_conv_matches_fp64(case):
    c = case
    op = Operands(c, seed=1000 + CASES.index(c))
    ref, pre, A = op.reference(c)
    bufs = op.buffers(c, torch.float32)
    y = nan_buffer((c.B, c.Ho, c.Wo, c.yct), torch.float32)
    d = desc(c, ptrs(bufs, y, op.b), y_f32=True)
    d.x.dtype = d.xu.dtype = L.F32
    d.engine = L.ENGINE_FFMA
    L.check(L.lib().yre_conv(C.byref(d), stream()), f"yre_conv ffma {c.name}")
    torch.cuda.synchronize()
    check_bound(check_window(c, y, f"{c.name} ffma"), ref, pre, A, c.silu, f"{c.name} ffma", tc=False)


def check_planes(planes: torch.Tensor, nhwc: torch.Tensor, what: str):
    """planes [4][B][Hp][Wp][C] against the NHWC map [B][H][W][C]: source cells bit for bit, the others +0"""
    H, W = nhwc.shape[1], nhwc.shape[2]
    zero = torch.zeros((), dtype=planes.dtype, device=DEV)
    for py in (0, 1):
        for px in (0, 1):
            p = planes[py * 2 + px]
            sub = nhwc[:, py::2, px::2]
            h, w = sub.shape[1], sub.shape[2]
            assert bool(same_bits(p[:, :h, :w], sub).all()), f"{what}: plane {py * 2 + px} differs from the NHWC output"
            for rest in (p[:, h:], p[:, :, w:]):
                assert bool(same_bits(rest, zero.expand_as(rest)).all()), \
                    f"{what}: plane {py * 2 + px} cells without a source pixel are not +0 ({H}x{W} map)"


# (frames as uint8, B, H, W, Cout, fp32 output): the MMA stems (64 bf16 channels; uint8, 4-aligned and unaligned widths)
# and the generic stem kernel
STEMS = [(False, 2, 45, 36, 64, False), (False, 2, 45, 37, 64, False), (False, 2, 33, 35, 32, False), (False, 1, 33, 35, 64, True),
         (True, 2, 45, 48, 64, False), (True, 2, 33, 37, 32, False)]


@pytest.mark.parametrize("u8,Bn,H,W,Cout,f32", STEMS)
def test_stem_parity_planes_are_complete(u8, Bn, H, W, Cout, f32):
    g = torch.Generator().manual_seed(H * W + Cout)
    Ho, Wo = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    img = torch.rand((Bn, 3, H, W), generator=g).to(DEV)
    frames = (torch.rand((Bn, H, W, 3), generator=g) * 255).to(torch.uint8).to(DEV)
    w = torch.randn((Cout, 3, 3, 3), generator=g).to(DEV)
    b = torch.randn((Cout,), generator=g).to(DEV)
    ydt, yl = (torch.float32, L.F32) if f32 else (torch.bfloat16, L.BF16)
    outs = {}
    for layout in (L.NHWC, L.PHASE4):
        shape = (Bn, Ho, Wo, Cout) if layout == L.NHWC else (4, Bn, (Ho + 1) // 2, (Wo + 1) // 2, Cout)
        y = nan_buffer(shape, ydt)
        d = L.StemDesc(None if u8 else img.data_ptr(), Bn, 3, H, W, L.View(y.data_ptr(), yl, layout, Bn, Ho, Wo, Cout, 0, Cout),
                       w.data_ptr(), b.data_ptr(), 2, L.ACT_SILU, frames.data_ptr() if u8 else None)
        L.check(L.lib().yre_stem_conv(C.byref(d), stream()), "yre_stem_conv")
        torch.cuda.synchronize()
        outs[layout] = y
    assert bool(torch.isfinite(outs[L.NHWC]).all())
    check_planes(outs[L.PHASE4], outs[L.NHWC], f"stem u8={u8} {H}x{W} Cout {Cout}")


@pytest.mark.parametrize("Bn,H,W,Cn", [(2, 40, 38, 128), (3, 22, 36, 96), (1, 41, 39, 256)])
def test_adown_parity_planes_are_complete(Bn, H, W, Cn):
    """the tiled kernel (128 bytes of channels per CTA) and the per-pixel one (half = 48 channels)"""
    g = torch.Generator().manual_seed(H + W + Cn)
    x = torch.randn((Bn, H, W, Cn), generator=g).bfloat16().to(DEV)
    half, Ha, Wa = Cn // 2, H - 1, W - 1
    Ho, Wo = (Ha - 1) // 2 + 1, (Wa - 1) // 2 + 1
    xv = L.View(x.data_ptr(), L.BF16, L.NHWC, Bn, H, W, Cn, 0, Cn)
    outs = {}
    for layout in (L.NHWC, L.PHASE4):
        lo = nan_buffer((Bn, Ha, Wa, half) if layout == L.NHWC else (4, Bn, (Ha + 1) // 2, (Wa + 1) // 2, half), torch.bfloat16)
        hi = nan_buffer((Bn, Ho, Wo, half), torch.bfloat16)
        L.check(L.lib().yre_adown_prepool(C.byref(xv), C.byref(L.View(lo.data_ptr(), L.BF16, layout, Bn, Ha, Wa, half, 0, half)),
                                          C.byref(L.View(hi.data_ptr(), L.BF16, L.NHWC, Bn, Ho, Wo, half, 0, half)), stream()), "adown")
        torch.cuda.synchronize()
        outs[layout] = (lo, hi)
    assert bool(torch.isfinite(outs[L.NHWC][0]).all())
    assert bool(same_bits(outs[L.PHASE4][1], outs[L.NHWC][1]).all())
    check_planes(outs[L.PHASE4][0], outs[L.NHWC][0], f"adown {H}x{W} C {Cn}")
