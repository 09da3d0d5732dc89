"""Parity at BASELINE.json's FULL sizes (configs 2, 4, 5).

The small-shape tests do not reach the kernel variants a full-size plan selects (CTA pairs with many rounds, paired halo
streams, 8x8 two-image halo tiles, 64-column staging, fp32 TMA stores ...), and a whole forward cannot be compared with the
oracle at these sizes in a test's time budget.  So:

  * every launch of the full-size plan is checked TEACHER-FORCED, element by element, against a float64 reference built
    from the operand values in the plan's own buffers, within the per-family bounds derived in tests/teacher_force.py;
    then one back-to-back run of the plan (programmatic dependent launch overlapping consecutive convs) must reproduce
    every buffer bit for bit;
  * size-independent properties of the whole path: a permutation of the batch permutes the outputs bit for bit, and NMS
    on the full-size bf16 predictions is bit-identical to the oracle's NMS (C restatement of the reference).
"""
import time

import numpy as np
import pytest
import torch

from bench_data import make_inputs
from oracle import nms_ref as N
from tests import teacher_force as TF
from tests.conftest import ROOT
from tests.test_cpu_conv_tc_select import tc_variant

pytestmark = pytest.mark.gpu

from yolo_b200 import YOLO, nms_raw
from yolo_b200 import engine as E

DEV = "cuda"
CONFIGS = {2: ("gelan-c", 640, 64), 5: ("gelan-c", 1280, 16), 4: ("yolov9-c", 640, 16)}


def _model(name, request):
    nodes, nc, sd = request.getfixturevalue("gelan_c" if name == "gelan-c" else "yolov9_c")
    m = YOLO.from_yaml(ROOT / "configs/models" / f"{name}.yaml")
    m.load_state_dict(sd, strict=True)
    return m.to(DEV).eval().set_precision("bf16")


@pytest.mark.parametrize("config", [2, 5, 4])
def test_every_launch_of_the_full_size_plan_teacher_forced(config, request):
    name, img, Bn = CONFIGS[config]
    model = _model(name, request)
    x = make_inputs(Bn, img, seed=7).to(DEV)
    with torch.cuda.device(x.device):
        p = E.compile_model(model, x)
        names = [n for n, _ in p.op_table()]
        assert len(names) == len(p.trace)
        assert "conv_ffma" not in names
        t0 = time.perf_counter()
        worst = TF.teacher_force(p, label=f"config {config} ")
        t1 = time.perf_counter()
        TF.run_reproduces(p)
        print(f"config {config}: {len(names)} launches checked per element in {t1 - t0:.1f} s, worst err / bound per kernel "
              f"family: {TF.report(worst)}; the back-to-back run reproduces every buffer")


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
