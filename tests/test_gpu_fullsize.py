"""Parity at BASELINE.json's FULL sizes (configs 2, 4, 5).

The small-shape tests do not reach the kernel variants a full-size plan selects (CTA pairs with many rounds, paired halo
streams, 8x8 two-image halo tiles, 64-column staging, fp32 TMA stores ...), and a whole forward cannot be compared with the
oracle at these sizes in a test's time budget.  So:

  * every launch of the full-size plan is checked TEACHER-FORCED: the launch's inputs are read back from the plan's own
    buffers, the op is restated with plain torch fp32 ops on the device (cuDNN with TF32 off -- the independent
    reference), and the launch's output must agree within the per-kernel tolerance written below;
  * size-independent properties of the whole path: a permutation of the batch permutes the outputs bit for bit, and NMS
    on the full-size bf16 predictions is bit-identical to the oracle's NMS (C restatement of the reference).
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from bench_data import make_inputs
from oracle import nms_ref as N
from tests import cpu_plan_exec as X
from tests.conftest import ROOT
from tests.test_cpu_conv_tc_select import tc_variant

pytestmark = pytest.mark.gpu

from yolo_b200 import YOLO, nms_raw
from yolo_b200 import _lib as L
from yolo_b200 import engine as E

DEV = "cuda"
# tolerances, as a fraction of max|reference| of the launch's output tensor
TOL_CONV_BF16 = 1.0e-2     # bf16 rounding of the output (2^-9 of the value) + tanh.approx + accumulation order
TOL_STEM = 2.0e-2          # the stem also rounds the fp32 IMAGE to bf16 operands (27 taps of 2^-9 input error on top)
TOL_CONV_F32 = 1.0e-3      # fp32 outputs (raw head logits): bf16 operands, fp32 accumulation, no rounding of the result
TOL_POOL = 1.0e-2          # ADown pre-pool averages in packed bf16
TOL_DECODE = 1.0e-4        # DFL softmax expectation + sigmoid in fp32

CONFIGS = {2: ("gelan-c", 640, 64), 5: ("gelan-c", 1280, 16), 4: ("yolov9-c", 640, 16)}


def _model(name, request):
    nodes, nc, sd = request.getfixturevalue("gelan_c" if name == "gelan-c" else "yolov9_c")
    m = YOLO.from_yaml(ROOT / "configs/models" / f"{name}.yaml")
    m.load_state_dict(sd, strict=True)
    return m.to(DEV).eval().set_precision("bf16")


def _rel(got, ref):
    return (got - ref).abs().max().item() / max(1e-6, ref.abs().max().item())


@pytest.mark.parametrize("config", [2, 5, 4])
def test_every_launch_of_the_full_size_plan_teacher_forced(config, request):
    name, img, Bn = CONFIGS[config]
    model = _model(name, request)
    x = make_inputs(Bn, img, seed=7).to(DEV)
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.cuda.device(x.device):
            p = E.compile_model(model, x)
            names = [n for n, _ in p.op_table()]
            assert len(names) == len(p.trace)
            assert "conv_ffma" not in names
            worst = {}
            for i, (kind, a) in enumerate(p.trace):
                if kind == "conv":
                    xin = X.nchw(X.read(a["x"]))
                    if a.get("xu") is not None:
                        xin = torch.cat((F.interpolate(X.nchw(X.read(a["xu"])), scale_factor=2.0, mode="nearest"), xin), 1)
                    res = X.nchw(X.read(a["res"])) if a["res"] is not None else None
                    p.run_op(i)
                    ref = F.conv2d(xin, a["w"].float().permute(0, 3, 1, 2), a["b"].float(), a["stride"], a["k"] // 2)
                    del xin
                    if a["silu"]:
                        ref = F.silu(ref)
                    if res is not None:
                        ref = ref + res
                    got = X.nchw(X.read(a["y"]))
                    f32 = a["y"].dtype == L.F32
                    err, tol = _rel(got, ref), (TOL_CONV_F32 if f32 else TOL_CONV_BF16)
                    key = "conv f32out" if f32 else "conv"
                elif kind == "stem":
                    p.run_op(i)
                    ref = F.conv2d(a["x"].float(), a["w"].float().permute(0, 3, 1, 2), a["b"].float(), a["stride"], 1)
                    if a["silu"]:
                        ref = F.silu(ref)
                    got = X.nchw(X.read(a["y"]))
                    err, tol, key = _rel(got, ref), TOL_STEM, "stem"
                elif kind == "adown":
                    xin = X.nchw(X.read(a["x"]))
                    p.run_op(i)
                    avg = F.avg_pool2d(xin, 2, 1, 0)
                    half = xin.shape[1] // 2
                    e1 = _rel(X.nchw(X.read(a["lo"])), avg[:, :half])
                    e2 = _rel(X.nchw(X.read(a["hi"])), F.max_pool2d(avg[:, half:], 3, 2, 1))
                    err, tol, key = max(e1, e2), TOL_POOL, "adown"
                elif kind == "spp":
                    xin = X.nchw(X.read(a["x"]))
                    p.run_op(i)
                    err = 0.0
                    for k_, win in (("y5", 5), ("y9", 9), ("y13", 13)):
                        assert torch.equal(X.nchw(X.read(a[k_])), F.max_pool2d(xin, win, 1, win // 2)), f"spp window {win}"
                    tol, key = 0.0, "spp"
                elif kind == "upsample":
                    xin = X.nchw(X.read(a["x"]))
                    p.run_op(i)
                    assert torch.equal(X.nchw(X.read(a["y"])), F.interpolate(xin, scale_factor=2.0, mode="nearest"))
                    err, tol, key = 0.0, 0.0, "upsample"
                elif kind == "cbfuse":
                    tgt = X.nchw(X.read(a["target"]))
                    acc = torch.zeros_like(tgt)
                    for s_ in a["srcs"]:
                        acc = acc + F.interpolate(X.nchw(X.read(s_)), size=tgt.shape[2:], mode="nearest")
                    p.run_op(i)
                    err, tol, key = _rel(X.nchw(X.read(a["y"])), acc + tgt), TOL_POOL, "cbfuse"
                elif kind == "decode":
                    p.run_op(i)
                    outs = []
                    for r, st in zip(a["raws"], a["strides"]):
                        z = X.read(r)
                        b_, H, W, _ = z.shape
                        e = (z[..., :64].reshape(b_, H, W, 4, 16).softmax(-1) * torch.tensor(a["dfl_w"], device=z.device)).sum(-1)
                        gy, gx = torch.meshgrid(torch.arange(H, device=z.device) + 0.5, torch.arange(W, device=z.device) + 0.5, indexing="ij")
                        x1, y1, x2, y2 = gx - e[..., 0], gy - e[..., 1], gx + e[..., 2], gy + e[..., 3]
                        box = torch.stack(((x1 + x2) / 2, (y1 + y2) / 2, x2 - x1, y2 - y1), -1) * st
                        outs.append(torch.cat((box, z[..., 64:].sigmoid()), -1).reshape(b_, H * W, -1))
                    ref = torch.cat(outs, 1)
                    got = a["y"]
                    eb = (got[..., :4] - ref[..., :4]).abs().max().item() / img            # boxes: fraction of the image size
                    es = (got[..., 4:] - ref[..., 4:]).abs().max().item()                  # scores: absolute
                    err, tol, key = max(eb, es), TOL_DECODE, "decode"
                else:
                    raise AssertionError(f"unexpected op {kind}")
                torch.cuda.synchronize()
                assert np.isfinite(err) and err <= tol, f"config {config} op {i} ({names[i]}: {p.op_descriptions()[i]}): error {err:.3e} > {tol:.1e}"
                worst[key] = max(worst.get(key, 0.0), err)
            print(f"config {config}: {len(names)} launches checked, worst error per kernel family (fraction of max|ref|): "
                  + ", ".join(f"{k} {v:.2e}" for k, v in worst.items()))
    finally:
        torch.backends.cudnn.allow_tf32 = old


def test_full_size_batch_permutation_and_nms(request):
    """Config 2 at full size: permuting the 64 images permutes y and the raw logits bit for bit (every output pixel is
    computed independently of its position in the batch, whatever tile it lands in), and NMS of the full-size bf16
    predictions equals the oracle's NMS bit for bit."""
    name, img, Bn = CONFIGS[2]
    model = _model(name, request)
    x = make_inputs(Bn, img, seed=11).to(DEV)
    perm = torch.randperm(Bn, generator=torch.Generator().manual_seed(3)).to(DEV)
    y, raws = model(x)
    yp, rawsp = model(x[perm].contiguous())
    torch.cuda.synchronize()
    assert torch.equal(yp, y[perm])
    for a, b in zip(rawsp, raws):
        assert torch.equal(a, b[perm])
    pred = y.permute(0, 2, 1).contiguous()
    out, counts, keep = nms_raw(pred, 0.25, 0.45, 300)
    ref = N.non_max_suppression(pred.cpu(), 0.25, 0.45, 300)
    cnt = counts.cpu().tolist()
    assert sum(cnt) > 1000                            # the calibrated weights give NMS real work
    for b_ in range(Bn):
        assert cnt[b_] == len(ref[b_])
        assert np.array_equal(out[b_, :cnt[b_]].cpu().numpy(), ref[b_])


def test_kernel_selection_rules_at_config_2(request):
    """The per-layer kernel selection (conv_tc_select, rules measured in profiles/r02_notes.md) is visible through
    yre_plan_op_variant; pin what the full-size config-2 plan gets so that a rule change shows up here.  The host-only
    query yre_conv_tc_describe must report exactly what the plan prepared on the device."""
    name, img, Bn = CONFIGS[2]
    model = _model(name, request)
    x = make_inputs(Bn, img, seed=7).to(DEV)
    with torch.cuda.device(x.device):
        p = E.compile_model(model, x)
    rows = [(d, v) for (n, _), d, v in zip(p.op_table(), p.op_descriptions(), p.op_variants()) if n == "conv_tc"]
    assert len(rows) == p.num_tcgen05 and "conv_ffma" not in [n for n, _ in p.op_table()]
    sms = torch.cuda.get_device_properties(x.device).multi_processor_count
    convs = [(v, a) for (kind, a), v in zip(p.trace, p.op_variants()) if kind == "conv"]
    assert len(convs) == len(rows)
    for v, a in convs:
        assert tc_variant(a, sms) == v

    def variants(prefix):
        got = {v.split(" thr=")[0] for d, v in rows if d.startswith(prefix)}
        assert got, prefix
        return got

    for d, v in rows:
        if d.startswith("conv3x3"):
            assert " s64" not in v, (d, v)                                   # 64-column staging is for 1x1 convs only
        if "f32out" in d:
            assert " tma-f32" in v, (d, v)                                   # raw logits leave through the fp32 TMA store
        else:
            assert " tma" in v and " direct" not in v, (d, v)
    assert all(v.startswith("generic-cta2") and " N=256 " in v for v in variants("conv3x3s1 256->256 @80x80"))
    assert all(v.startswith("halo-stream ") and " pair" in v and " N=128 " in v for v in variants("conv3x3s1 128->128 @80x80"))
    assert all(v.startswith("halo-stream ") and " pair" in v and " N=64 " in v for v in variants("conv3x3s1 256->64 @80x80"))
    assert all(v.startswith("halo-stream-ybx") and " pair" in v for v in variants("conv3x3s1 512->64 @40x40"))
    assert all(v.startswith("halo-ws") for v in variants("conv3x3s1 32->32 @160x160") | variants("conv3x3s1 64->64 @80x80"))
    assert all(v.startswith("generic ") and " s64" in v for v in variants("conv1x1s1 128->128 @80x80"))     # K = 128: no CTA pairs
    assert all(v.startswith("generic-cta2") and " s64" in v for v in variants("conv1x1s1 256->256 @160x160"))
    assert all(v.startswith("generic-cta2") for v in variants("conv3x3s1 128->128 @20x20") | variants("conv3x3s1 128->128 @40x40")
               | variants("conv1x1s1 1024->512 @40x40") | variants("conv3x3s2 64->128 @160x160"))
