"""CPU pin of the plan compiler's output: the launch list of every plan below, written in a canonical form, must hash
line for line to tests/golden/plan_launch_lists.json.  A compiler change that moves one window, drops one op or swaps
one weight shows up here, before the plan ever runs.

Canonical form of a plan (one line each):
  * every Plan.trace op: its kind, then every argument in sorted key order.  A view is
    ``b<id>:dtype/layout/BxHxWxC_total[c_off+C]``, the buffer id counting buffers in order of first appearance in the
    trace.  ``w`` and ``b`` are shape, dtype and a hash of their bytes; other tensors (image inputs, ``y``) are
    uninitialised, so they are shape and dtype only.  Scalars are written with repr;
  * every ``p.vals`` entry that is a view, as ``layer -> view``;
  * the totals: op names and FLOPs, launch count, activation bytes, the multiset of (shape, dtype) of the tensors the plan
    keeps, and the structure of ``p.result`` (or of the outputs of ``compile_module``).

The weights are drawn from fixed seeds, with every BatchNorm affine term and running statistic randomised so that a
BN folded into the wrong conv changes a hash.  (The oracle's calibrated state_dict takes its running statistics from
a CPU forward pass whose last bits depend on the machine's thread count, so it cannot feed a byte hash.)

Regenerate with ``python -m tests.test_cpu_plan_launch_list --write`` only when a change to what is emitted is meant."""
import hashlib
import json
import sys
from collections import Counter

import pytest
import torch

from tests.conftest import ROOT

from yolo_b200 import YOLO, _lib as L, blocks as B, engine
from yolo_b200.heads import DetectDFL

GOLDEN = ROOT / "tests/golden/plan_launch_lists.json"
_LAYOUT = {L.NHWC: "nhwc", L.PHASE4: "phase4"}


def _randomize_bn(m: torch.nn.Module, seed: int) -> None:
    g = torch.Generator().manual_seed(seed)
    for mod in m.modules():
        if isinstance(mod, torch.nn.BatchNorm2d):
            mod.weight.data.uniform_(0.8, 1.2, generator=g)
            mod.bias.data.normal_(0, 0.2, generator=g)
            mod.running_mean.normal_(0, 0.3, generator=g)
            mod.running_var.uniform_(0.5, 1.5, generator=g)


def _model_plan(cfg, shape, prec="bf16", u8=False, num_classes=None, fuse_upsample=True, main_only=False):
    torch.manual_seed(0)
    m = YOLO.from_yaml(ROOT / "configs/models" / f"{cfg}.yaml", num_classes=num_classes)
    _randomize_bn(m, 1)
    m.eval().set_precision(prec)
    m.fuse_upsample, m.main_only = fuse_upsample, main_only
    x = torch.empty(shape, dtype=torch.uint8 if u8 else torch.float32)
    return engine.compile_model(m, x), None


def _detect_head():
    m = DetectDFL(80, (64, 128, 256))
    m.stride = torch.tensor([8.0, 16.0, 32.0])
    m.init_bias()
    return m, [torch.empty(1, c, s, s) for c, s in ((64, 16), (128, 8), (256, 4))]


# the block cases of test_cpu_host.py::test_block_plans, a stem Conv and a detection head
_MODULES = {
    "elan": lambda: (B.RepNCSPELAN4(128, 256, 128, 64, 1), torch.empty(1, 128, 16, 16)),
    "adown": lambda: (B.ADown(128, 256), torch.empty(1, 128, 16, 16)),
    "adown_odd": lambda: (B.ADown(64, 64), torch.empty(1, 64, 13, 13)),
    "sppelan": lambda: (B.SPPELAN(64, 64, 32), torch.empty(1, 64, 10, 10)),
    "csp": lambda: (B.RepNCSP(64, 64, 2), torch.empty(1, 64, 8, 8)),
    "stem": lambda: (B.Conv(3, 32, 3, 2), torch.empty(1, 3, 32, 32)),
    "detect": _detect_head,
}


def _module_plan(case, prec):
    torch.manual_seed(0)
    m, x = _MODULES[case]()
    _randomize_bn(m, 1)
    return engine.compile_module(m.eval(), x, prec)


PLANS = {
    "gelan-c_2x640_bf16": lambda: _model_plan("gelan-c", (2, 3, 640, 640)),
    "gelan-c_2x640_fp16": lambda: _model_plan("gelan-c", (2, 3, 640, 640), "fp16"),
    "gelan-c_2x640_fp32": lambda: _model_plan("gelan-c", (2, 3, 640, 640), "fp32"),
    "gelan-c_2x640x384_u8_bf16": lambda: _model_plan("gelan-c", (2, 640, 384, 3), u8=True),
    "gelan-c_2x384x640_bf16": lambda: _model_plan("gelan-c", (2, 3, 384, 640)),
    "gelan-c_3x64x96_bf16": lambda: _model_plan("gelan-c", (3, 3, 64, 96)),
    "gelan-c_1x224x352_bf16": lambda: _model_plan("gelan-c", (1, 3, 224, 352)),
    "gelan-c_2x640_bf16_no_fuse_upsample": lambda: _model_plan("gelan-c", (2, 3, 640, 640), fuse_upsample=False),
    "gelan-c_2x640_bf16_nc3": lambda: _model_plan("gelan-c", (2, 3, 640, 640), num_classes=3),
    "gelan-c_64x640_bf16": lambda: _model_plan("gelan-c", (64, 3, 640, 640)),
    "gelan-c_16x1280_bf16": lambda: _model_plan("gelan-c", (16, 3, 1280, 1280)),
    "yolov9-c_16x640_bf16": lambda: _model_plan("yolov9-c", (16, 3, 640, 640)),
    "yolov9-c_16x640_bf16_main_only": lambda: _model_plan("yolov9-c", (16, 3, 640, 640), main_only=True),
    **{f"module_{case}_{prec}": (lambda case=case, prec=prec: _module_plan(case, prec))
       for case in _MODULES for prec in ("bf16", "fp32")},
}


class _Writer:
    def __init__(self):
        self.buf_ids: dict[int, int] = {}

    def __call__(self, v, key: str = "") -> str:
        if isinstance(v, engine.V):
            bid = self.buf_ids.setdefault(id(v.t), len(self.buf_ids))
            dt = str(engine._TORCH_DT[v.dtype]).removeprefix("torch.")
            return f"b{bid}:{dt}/{_LAYOUT[v.layout]}/{v.B}x{v.H}x{v.W}x{v.C_total}[{v.c_off}+{v.C}]"
        if isinstance(v, torch.Tensor):
            s = f"{tuple(v.shape)} {str(v.dtype).removeprefix('torch.')}"
            if key in ("w", "b"):
                s += " " + hashlib.sha256(v.contiguous().view(torch.uint8).numpy().tobytes()).hexdigest()[:16]
            return s
        if isinstance(v, (list, tuple)):
            return "[" + ", ".join(self(o, key) for o in v) + "]"
        return repr(v)


def canonical_lines(p: engine.Plan, outputs=None) -> list[str]:
    fmt = _Writer()
    lines = [kind + " " + " ".join(f"{k}={fmt(a[k], k)}" for k in sorted(a)) for kind, a in p.trace]
    vals = getattr(p, "vals", {})
    lines += [f"{n} -> {fmt(v)}" for n, v in sorted(vals.items()) if isinstance(v, engine.V)]
    keep = sorted(Counter((tuple(t.shape), str(t.dtype)) for t in p.keep).items())
    if p.result is not None:
        kind, y, raws = p.result
        result = f"{kind} y={fmt(y)} raws={fmt(raws)}"
    else:
        result = f"outputs={fmt(outputs)}"
    lines.append(f"ops={p.op_table()!r} launches={p.num_launches} act_bytes={p.act_bytes} keep={keep!r} {result}")
    return lines


def _hash(line: str) -> str:
    return hashlib.sha256(line.encode()).hexdigest()[:16]


@pytest.fixture()
def dry():
    engine._ALLOW_CPU_DRY_RUN = True
    yield
    engine._ALLOW_CPU_DRY_RUN = False


@pytest.mark.parametrize("name", sorted(PLANS))
def test_launch_list_matches_the_pinned_one(dry, name):
    golden = json.loads(GOLDEN.read_text())[name]
    p, outputs = PLANS[name]()
    lines = canonical_lines(p, outputs)
    for i, (line, h) in enumerate(zip(lines, golden["hashes"])):
        if _hash(line) != h:
            where = f"op {i}: {p.op_descriptions()[i]}" if i < len(p.trace) else f"line {i} (after the {len(p.trace)} ops)"
            pytest.fail(f"{name}: first difference at {where}\n  {line}")
    assert len(lines) == golden["lines"], (len(lines), golden["lines"])


def test_wiring_needs_only_the_graph_and_the_input_extent():
    """engine.wire_model decides extents, concat windows, lazy upsamples, main_only pruning and the stem's layout from
    the module graph alone, before a plan allocates anything"""
    m = YOLO.from_yaml(ROOT / "configs/models/gelan-c.yaml")
    w = engine.wire_model(m, 384, 640, 3)
    assert [(w[n].H, w[n].W, w[n].C) for n in ("stem1", "down1", "down3", "up1", "concat1")] == \
        [(192, 320, 64), (48, 80, 256), (12, 20, 512), (24, 40, 512), (24, 40, 1024)]
    assert {n for n in w if w[n].lazy} == {"up1", "up2"}
    assert (w["stage3"].dest, w["pan_down1"].dest, w["fpn1"].dest) == (("concat1", 0), ("concat3", 0), ("concat3", 256))
    assert w["stem1"].phase4 and not w["stem2"].phase4
    m.fuse_upsample = False
    m.set_precision("fp32")
    w = engine.wire_model(m, 384, 640, 3)
    assert not any(v.lazy for v in w.values()) and (w["up1"].dest, w["stage3"].dest) == (("concat1", 0), ("concat1", 512))
    assert not w["stem1"].phase4                         # the fp32 stem writes NHWC

    m = YOLO.from_yaml(ROOT / "configs/models/yolov9-c.yaml")
    w = engine.wire_model(m, 640, 640, 3)
    assert w["stem1"].srcs == w["aux_stem1"].srcs == ["input"]       # both read the image through input_silence
    assert all(v.needed for v in w.values()) and len(w["detect"].srcs) == 6
    m.main_only = True
    w = engine.wire_model(m, 640, 640, 3)
    assert w["detect"].srcs == ["fpn2", "pan1", "pan2"]
    assert {n for n in w if not w[n].needed} == {n for n in w if n.startswith(("aux_", "cb_route"))}


if __name__ == "__main__":
    if "--write" not in sys.argv:
        sys.exit("usage: python -m tests.test_cpu_plan_launch_list --write")
    engine._ALLOW_CPU_DRY_RUN = True
    out = {}
    for name in sorted(PLANS):
        lines = canonical_lines(*PLANS[name]())
        out[name] = {"lines": len(lines), "hashes": [_hash(l) for l in lines]}
        print(f"{name}: {len(lines)} lines")
    GOLDEN.write_text(json.dumps(out, indent=0) + "\n")
