"""The teacher-forcing checker (tests/teacher_force.py) without a GPU: each family's bound accepts its reference rounded
to the output type and rejects the perturbation its docstring says it can see; a dry plan replayed op by op with the CPU
interpreter passes every launch, every batch slice is checked, and the back-to-back comparison names the first op
whose buffer differs."""
import pytest
import torch
import torch.nn.functional as F

from oracle import gelan_ref as G
from tests import cpu_plan_exec as X
from tests import teacher_force as TF
from tests.conftest import ROOT

from yolo_b200 import YOLO, _lib as L
from yolo_b200 import engine as E

TDT = {L.BF16: torch.bfloat16, L.F16: torch.float16, L.F32: torch.float32}


def view(t: torch.Tensor, dtype, layout=L.NHWC, hw=None) -> E.V:
    if layout == L.NHWC:
        Bn, H, W, Cn = t.shape
    else:
        _, Bn, _, _, Cn = t.shape
        H, W = hw
    return E.V(t, Bn, H, W, Cn, 0, Cn, dtype, layout)


def fails(fn, *args, match: str = "over the bound"):
    with pytest.raises(AssertionError, match=match):
        fn(*args)


# ---- conv --------------------------------------------------------------------------------------------------------------
def conv_op(dtype, perturb=None, seed=0):
    """a 3x3 48 -> 48 conv with a 16-channel tail in the 32 + 16 tiling, SiLU and a bias over [-12, 6]; y is the fp64 result
    rounded to fp32 (the epilogue's value), perturbed, then rounded to the output type"""
    g = torch.Generator().manual_seed(seed)
    tdt = TDT[dtype] if dtype != L.F32 else torch.bfloat16
    x = torch.randn((2, 12, 10, 32), generator=g).to(tdt)
    w = (torch.randn((48, 3, 3, 32), generator=g) * (2.5 / 288 ** 0.5)).to(tdt)
    b = torch.rand((48,), generator=g) * 18 - 12
    pre = F.conv2d(x.double().permute(0, 3, 1, 2), w.double().permute(0, 3, 1, 2), b.double(), 1, 1)
    if perturb == "no tail bias":
        pre[:, 32:] -= b.double()[32:, None, None]
    f = F.silu(pre).float().permute(0, 2, 3, 1).contiguous()
    if perturb == "column":        # the column with the largest bias: outside the SiLU's negative tail, where 2^-11 |pre| hides it
        c = int(b.argmax())
        f[..., c] += 2.0 ** -8 * f[..., c].abs()
    y = f.to(TDT[dtype])
    return dict(x=view(x, L.F16 if tdt == torch.float16 else L.BF16), xu=None, res=None, w=w, b=b, k=3, stride=1, silu=True,
                y=view(y, dtype))


@pytest.mark.parametrize("dtype", [L.BF16, L.F16, L.F32])
def test_conv_bound(dtype):
    assert TF._conv(conv_op(dtype), 0, 2, "conv")["conv f32out" if dtype == L.F32 else "conv"] < 1
    fails(TF._conv, conv_op(dtype, "column"), 0, 2, "conv")
    fails(TF._conv, conv_op(dtype, "no tail bias"), 0, 2, "conv")


def test_check_bound_is_the_fp32_conv_bound():
    g = torch.Generator().manual_seed(1)
    ref, pre, A = (torch.randn((2, 3, 4, 5), generator=g, dtype=torch.float64) for _ in range(3))
    A = A.abs() + pre.abs()
    assert torch.equal(TF.conv_bound(ref, pre, A, True, L.F32), TF.conv_fp32_bound(ref, pre, A, True))
    assert TF.check_bound(ref.float(), ref, pre, A, True, "fp32") < -14
    fails(TF.check_bound, (ref * (1 + 2.0 ** -8)).float(), ref, pre, A, False, "fp32")


# ---- stem --------------------------------------------------------------------------------------------------------------
def stem_op(dtype, perturb=None, u8=False):
    g = torch.Generator().manual_seed(2)
    frames = torch.randint(0, 256, (2, 20, 32, 3), generator=g, dtype=torch.uint8)
    img = frames.flip(-1).permute(0, 3, 1, 2).float() * torch.tensor(1 / 255, dtype=torch.float32)
    w = torch.randn((64, 3, 3, 3), generator=g) * 0.3
    b = torch.randn((64,), generator=g)
    tdt = TDT[dtype]
    pre = F.conv2d(img.to(tdt).double(), w.to(tdt).double().permute(0, 3, 1, 2), b.double(), 2, 1)
    if perturb == "no tail bias":
        pre[:, 48:] -= b.double()[48:, None, None]
    y = view(F.silu(pre).permute(0, 2, 3, 1).to(tdt).contiguous(), dtype)
    return dict(x=frames if u8 else img.contiguous(), y=y, w=w, b=b, stride=2, silu=True, u8=u8)


@pytest.mark.parametrize("dtype", [L.BF16, L.F16])
@pytest.mark.parametrize("u8", [False, True])
def test_stem_bound(dtype, u8):
    a = stem_op(dtype, u8=u8)
    assert TF.stem_rounds_operands(a)
    assert TF._stem(a, 0, 2, "stem")["stem"] < 1
    fails(TF._stem, stem_op(dtype, "no tail bias", u8), 0, 2, "stem")


# ---- ADown -------------------------------------------------------------------------------------------------------------
def adown_op(dtype, perturb=None):
    g = torch.Generator().manual_seed(3)
    x = (torch.randn((3, 14, 12, 32), generator=g) * 4).to(TDT[dtype])
    xn = x.double().permute(0, 3, 1, 2)
    avg = F.avg_pool2d(xn, 2, 1, 0)
    if perturb == "three pixels":
        avg[1, 3, 4, 5] = (xn[1, 3, 4, 5] + xn[1, 3, 4, 6] + xn[1, 3, 5, 5]) / 4
    lo = torch.zeros((4, 3, 7, 6, 16), dtype=TDT[dtype])
    lov = view(lo, dtype, L.PHASE4, (13, 11))
    X.write(lov, avg[:, :16].permute(0, 2, 3, 1))
    if perturb == "edge":
        lo[3, 2, 6, 0, 7] = 1.0          # plane (1, 1) has 6 rows with a source pixel: row 6 is an edge row
    if perturb == "-0 edge":
        lo[1, 0, 3, 5, 0] = -0.0         # plane (0, 1) has 5 columns with a source pixel
    hi = F.max_pool2d(avg[:, 16:], 3, 2, 1).permute(0, 2, 3, 1).to(TDT[dtype]).contiguous()
    return dict(x=view(x, dtype), lo=lov, hi=view(hi, dtype))


@pytest.mark.parametrize("dtype", [L.BF16, L.F16])
def test_adown_bound(dtype):
    assert TF._adown(adown_op(dtype), 0, 3, "adown")["adown"] < 1
    fails(TF._adown, adown_op(dtype, "three pixels"), 0, 3, "adown")
    fails(TF._adown, adown_op(dtype, "edge"), 0, 3, "adown", match="not \\+0")
    fails(TF._adown, adown_op(dtype, "-0 edge"), 0, 3, "adown", match="not \\+0")


# ---- CBFuse ------------------------------------------------------------------------------------------------------------
def cbfuse_op(dtype, perturb=None):
    g = torch.Generator().manual_seed(4)
    tdt = TDT[dtype]
    srcs = [(torch.randn((2, 4, 6, 16), generator=g) * 50).to(tdt), (torch.randn((2, 2, 3, 16), generator=g) * 50).to(tdt)]
    tgt = (torch.randn((2, 8, 12, 16), generator=g) * 50).to(tdt)
    terms = [F.interpolate(s.float().permute(0, 3, 1, 2), size=(8, 12), mode="nearest") for s in srcs] + [tgt.float().permute(0, 3, 1, 2)]
    if perturb == "dropped source":
        terms = terms[1:]
    acc = torch.zeros_like(terms[0])
    for t in terms:
        acc = acc + t
        if perturb == "rounded partial sums":
            acc = acc.to(tdt).float()
    y = acc.permute(0, 2, 3, 1).to(tdt).contiguous()
    return dict(srcs=[view(s, dtype) for s in srcs], target=view(tgt, dtype), y=view(y, dtype))


@pytest.mark.parametrize("dtype", [L.BF16, L.F16])
def test_cbfuse_bound(dtype):
    assert TF._cbfuse(cbfuse_op(dtype), 0, 2, "cbfuse")["cbfuse"] < 1
    fails(TF._cbfuse, cbfuse_op(dtype, "dropped source"), 0, 2, "cbfuse")
    fails(TF._cbfuse, cbfuse_op(dtype, "rounded partial sums"), 0, 2, "cbfuse")


# ---- decode -----------------------------------------------------------------------------------------------------------
def decode_op(perturb=None):
    g = torch.Generator().manual_seed(5)
    raws, outs = [], []
    dfl = [float(k) for k in range(16)]
    for H, W, st in ((8, 12, 8.0), (4, 6, 16.0), (2, 3, 32.0)):
        z = torch.cat((torch.randn((2, H, W, 64), generator=g) * 3, torch.randn((2, H, W, 80), generator=g) * 4 - 4), -1)
        raws.append(view(z, L.F32))
        zb = z.bfloat16().float()
        e = ((zb if perturb == "bf16 bins" else z)[..., :64].reshape(2, H, W, 4, 16).softmax(-1) * torch.tensor(dfl)).sum(-1)
        gy, gx = torch.meshgrid(torch.arange(H) + 0.5, torch.arange(W) + 0.5, indexing="ij")
        box = torch.stack((gx + (e[..., 2] - e[..., 0]) / 2, gy + (e[..., 3] - e[..., 1]) / 2, e[..., 0] + e[..., 2], e[..., 1] + e[..., 3]), -1) * st
        sc = ((zb if perturb == "bf16 scores" else z)[..., 64:]).sigmoid()
        outs.append(torch.cat((box, sc), -1).reshape(2, H * W, -1))
    return dict(raws=raws, strides=[8.0, 16.0, 32.0], nc=80, dfl_w=dfl, y=torch.cat(outs, 1))


def test_decode_bounds():
    r = TF._decode(decode_op(), 0, 2, "decode")
    assert r["decode box"] < 1 and r["decode score"] < 1
    fails(TF._decode, decode_op("bf16 scores"), 0, 2, "decode")
    fails(TF._decode, decode_op("bf16 bins"), 0, 2, "decode")


def test_score_bound_at_the_float_limits():
    z = torch.tensor([-200.0, -100.0, -87.0, 0.0, 30.0], dtype=torch.float64)
    sig = torch.sigmoid(z)
    device_like = torch.where(z < -87.3, torch.zeros_like(sig), sig * (1 - 2.0 ** -16.5))
    assert bool(((device_like - sig).abs() <= TF.score_bound(sig)).all())


# ---- a dry plan, op by op -----------------------------------------------------------------------------------------------
@pytest.fixture()
def dry():
    E._ALLOW_CPU_DRY_RUN = True
    yield
    E._ALLOW_CPU_DRY_RUN = False


def cpu_runner(plan, inject=None):
    """runs op i with the CPU interpreter; an mma.sync stem rounds the image and weights first, as on the device.
    inject(i, a) may perturb op i's outputs after it ran."""
    def run(i):
        kind, a = plan.trace[i]
        if kind == "stem" and TF.stem_rounds_operands(a):
            tdt = TDT[a["y"].dtype]
            y = F.conv2d(a["x"].to(tdt).float(), a["w"].to(tdt).float().permute(0, 3, 1, 2), a["b"], a["stride"], 1)
            X.write(a["y"], X.nhwc(F.silu(y) if a["silu"] else y))
        else:
            X.run_op(kind, a)
        if inject is not None:
            inject(i, a)
    return run


def dry_plan(request, name, prec, Bn=3, H=64, W=96):
    nodes, nc, sd = request.getfixturevalue("gelan_c" if name == "gelan-c" else "yolov9_c")
    m = YOLO.from_yaml(ROOT / "configs/models" / f"{name}.yaml")
    m.load_state_dict(sd)
    m.eval().set_precision(prec)
    x = G.fractal(Bn, H, torch.Generator().manual_seed(8), w=W)
    return E.compile_model(m, x), x


@pytest.mark.parametrize("name,prec", [("gelan-c", "bf16"), ("gelan-c", "fp16"), ("yolov9-c", "bf16")])
def test_dry_plan_passes_op_by_op_and_reproduces(dry, request, name, prec):
    p, x = dry_plan(request, name, prec, Bn=3 if name == "gelan-c" else 2, H=64, W=96 if name == "gelan-c" else 64)
    worst = TF.teacher_force(p, run_op=cpu_runner(p), max_elems=1)      # one image per slice
    fams = {"conv", "conv f32out", "stem", "adown", "spp", "decode box", "decode score"}
    fams |= {"cbfuse"} if name == "yolov9-c" else set()
    assert fams <= set(worst), worst
    assert all(v < 1 for v in worst.values()), worst
    print(f"\n{name} {prec} dry plan: {TF.report(worst)}")
    run_op = cpu_runner(p)

    def run():
        for i in range(len(p.trace)):
            run_op(i)
    TF.run_reproduces(p, run=run)
    conv = next(i for i, (k, _) in enumerate(p.trace) if k == "conv" and p.trace[i][1]["res"] is None)

    def bad_run():
        run()
        y = p.trace[conv][1]["y"]
        y.t[-1, -1, -1, y.c_off] += 1.0
    with pytest.raises(AssertionError, match=f"first written by op {conv} "):
        TF.run_reproduces(p, run=bad_run)


@pytest.mark.parametrize("where", ["conv", "adown", "decode"])
def test_every_batch_slice_is_checked(dry, request, where):
    """slices of two images over a batch of three: one element perturbed in the last image of the last slice fails"""
    p, _ = dry_plan(request, "gelan-c", "bf16")
    j = next(i for i, (k, a) in enumerate(p.trace) if k == where and (k != "conv" or a["res"] is None))
    a = p.trace[j][1]
    per = {"conv": lambda: a["y"].H * a["y"].W * a["y"].C, "adown": lambda: a["x"].H * a["x"].W * a["x"].C,
           "decode": lambda: a["y"][0].numel()}[where]()

    def inject(i, a_):
        if i != j:
            return
        if where == "decode":
            a_["y"][-1, -1, -1] += 2.0 ** -10 * a_["y"][-1, -1, -1].abs() + 2.0 ** -100
        else:
            v = a_["y"] if where == "conv" else a_["hi"]
            e = v.t[-1, -1, -1, v.c_off + v.C - 1]
            v.t[-1, -1, -1, v.c_off + v.C - 1] = e + 2.0 ** -5 * e.abs() + 1e-3
    with pytest.raises(AssertionError, match=f"op {j} .*worst at \\(b, [^)]*\\) = \\(2, "):
        TF.teacher_force(p, run_op=cpu_runner(p, inject), max_elems=2 * per)


def test_unwritten_output_fails(dry, request):
    """outputs are NaN-filled before their launch: an op that leaves part of its window alone fails"""
    p, _ = dry_plan(request, "gelan-c", "bf16", Bn=2, H=64, W=64)
    j = next(i for i, (k, _) in enumerate(p.trace) if k == "spp")

    def skip(i):
        if i == j:
            a = p.trace[j][1]
            for k in ("y5", "y9"):
                X.write(a[k], X.nhwc(F.max_pool2d(X.nchw(X.read(a["x"])), 5 if k == "y5" else 9, 1, 2 if k == "y5" else 4)))
        else:
            cpu_runner(p)(i)
    with pytest.raises(AssertionError, match=f"op {j} .*window 13"):
        TF.teacher_force(p, run_op=skip)


def test_unknown_op_kind_raises(dry, request):
    p, _ = dry_plan(request, "gelan-c", "bf16", Bn=1, H=64, W=64)
    p.trace.insert(0, ("mystery", {}))
    with pytest.raises(ValueError, match="mystery"):
        TF.teacher_force(p, run_op=lambda i: None)


def test_checksums_see_one_bit():
    ts = [torch.randn(1000).bfloat16(), torch.randn(7, 9), torch.arange(10, dtype=torch.int64)]
    for clone in (True, False):
        snap = TF.snapshot(ts, clone)
        assert TF.changed(ts, snap, clone) == []
        ts[1].view(torch.int32)[3, 4] ^= 1
        assert TF.changed(ts, snap, clone) == [1]
        ts[1].view(torch.int32)[3, 4] ^= 1
        t0 = ts[0].clone()
        ts[0][[5, 6]] = ts[0][[6, 5]]                            # a swap keeps the plain sum: the weighted one sees it
        assert TF.changed(ts, snap, clone) == ([0] if not torch.equal(t0, ts[0]) else [])
        ts[0].copy_(t0)
