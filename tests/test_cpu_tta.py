"""Test-time augmentation without a GPU: the branch geometry of yre_tta_geometry against upstream's Python arithmetic,
the tcgen05 kernel selection of the branch plans, which plans model(x, augment=True) compiles, oracle/tta_ref.py against
upstream's code, K12's fp32 formula against torch's bilinear resize, and the ABI of the new descriptors."""
import contextlib
import ctypes as C
import math
import subprocess

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import gelan_ref as G
from oracle import tta_ref as T
from tests.conftest import ROOT
from tests.test_cpu_conv_tc_select import tc_variant

from yolo_b200 import YOLO, _lib as L, engine, tta

SIZES = [(64, 96), (128, 128), (192, 320), (384, 640), (640, 384), (640, 640), (736, 1280), (1280, 1280), (32, 32),
         (32, 2048), (4096, 96)]


def upstream_sizes(h, w):
    """scale_img's sizes for the three ratios, in upstream's own expressions"""
    out = []
    for ratio in (1.0, 0.83, 0.67):
        if ratio == 1.0:
            out.append(((h, w), (h, w)))
            continue
        s = (int(h * ratio), int(w * ratio))
        out.append((s, tuple(math.ceil(x * ratio / 32) * 32 for x in (h, w))))
    return out


@pytest.mark.parametrize("h,w", SIZES)
def test_geometry_matches_scale_img_and_clip_augmented(h, w):
    g = tta.geometry(h, w)
    assert (g.h, g.w) == (h, w)
    ups = upstream_sizes(h, w)
    assert T.branch_shapes(h, w) == ups
    A_tot = 0
    for i, ((rh, rw), (oh, ow)) in enumerate(ups):
        assert (g.rh[i], g.rw[i], g.out_h[i], g.out_w[i]) == (rh, rw, oh, ow), i
        assert g.scale[i] == np.float32((1.0, 0.83, 0.67)[i]) and g.flip[i] == (i == 1)
        # _clip_augmented on a y with one column per anchor: which anchors survive
        A = sum((oh // s) * (ow // s) for s in (8, 16, 32))
        assert (g.A[i], g.a_begin[i], g.a_end[i]) == T.windows(h, w)[i]
        assert g.A[i] == A
        A_tot += g.a_end[i] - g.a_begin[i]
    ys = [torch.arange(g.A[i]).view(1, 1, -1) for i in range(3)]
    kept = T.clip_augmented(list(ys))
    for i in range(3):
        assert torch.equal(kept[i].flatten(), torch.arange(g.a_begin[i], g.a_end[i])), i
    assert g.A_tot == A_tot


def test_geometry_of_the_issue_table():
    g = tta.geometry(640, 640)
    assert [(g.out_h[i], g.out_w[i]) for i in range(3)] == [(640, 640), (544, 544), (448, 448)]
    assert [g.a_end[i] - g.a_begin[i] for i in range(3)] == [8000, 6069, 980] and g.A_tot == 15049
    g = tta.geometry(384, 640)
    assert [(g.rh[i], g.rw[i], g.out_h[i], g.out_w[i]) for i in range(3)] == [(384, 640, 384, 640), (318, 531, 320, 544),
                                                                            (257, 428, 288, 448)]
    assert g.A_tot == 9000
    assert tta.geometry(1280, 1280).A_tot == 59921


@pytest.mark.parametrize("h,w", [(0, 64), (64, 0), (63, 64), (64, 100), (96, 33), (-32, 64), (65568, 64)])
def test_sizes_that_are_not_multiples_of_32_are_rejected(h, w):
    g = L.TtaGeom()
    assert L.lib().yre_tta_geometry(h, w, C.byref(g)) == -1
    with pytest.raises(ValueError, match="multiples of 32"):
        tta.geometry(h, w)


def test_descriptors_are_validated_before_any_launch():
    lib = L.lib()
    g = tta.geometry(64, 64)
    ptr = 0x7f0000000000
    good = dict(x_nchw=ptr, B=2, n=2, H=64, W=64, flip=1, rh=g.rh[1], rw=g.rw[1], out_h=g.out_h[1], out_w=g.out_w[1], y=ptr + (1 << 20))
    for bad in (dict(n=3), dict(n=0), dict(x_u8_hwc=ptr), dict(x_nchw=None), dict(rh=65), dict(flip=2), dict(y=ptr + 2)):
        d = L.TtaScaleDesc(**{**good, **bad})
        assert lib.yre_tta_scale_img(C.byref(d), None) == -1, bad
    m = L.TtaMergeDesc()
    for i in range(3):
        m.br[i] = L.TtaMergeBranch(ptr + (i << 24), g.A[i], g.a_begin[i], g.a_end[i], g.scale[i], 64 if i == 1 else 0)
    m.B, m.n, m.nc, m.out = 2, 2, 80, ptr + (4 << 24)
    for field, value in (("n", 3), ("nc", 0), ("nc", 4097), ("out", ptr + 8)):
        old = getattr(m, field)
        setattr(m, field, value)
        assert lib.yre_tta_merge(C.byref(m), None) == -1, field
        setattr(m, field, old)
    for change in (dict(y=ptr + 4), dict(a_end=g.A[0] + 1), dict(a_begin=5, a_end=5), dict(scale=0.0), dict(flip_w=-1)):
        old = L.TtaMergeBranch.from_buffer_copy(m.br[0])
        for k, v in change.items():
            setattr(m.br[0], k, v)
        assert lib.yre_tta_merge(C.byref(m), None) == -1, change
        m.br[0] = old


@pytest.fixture()
def dry():
    engine._ALLOW_CPU_DRY_RUN = True
    yield
    engine._ALLOW_CPU_DRY_RUN = False


@pytest.mark.parametrize("name,Bn,H,W", [("gelan-c", 64, 640, 640), ("gelan-c", 64, 384, 640), ("gelan-c", 16, 1280, 1280),
                                         ("yolov9-c", 16, 640, 640)])
def test_branch_plans_get_a_tcgen05_variant_for_every_conv(dry, name, Bn, H, W):
    g = tta.geometry(H, W)
    m = YOLO.from_yaml(ROOT / "configs/models" / f"{name}.yaml").eval().set_precision("bf16")
    for i in (1, 2):
        p = engine.compile_model(m, torch.empty(Bn, 3, g.out_h[i], g.out_w[i]), main_only=True)
        convs = [a for k, a in p.trace if k == "conv"]
        assert len(convs) > 100
        for a in convs:
            tc_variant(a, 148)                           # asserts that the describe query returns 0
        _, y, _ = p.result
        assert tuple(y.shape) == (Bn, g.A[i], 84)
        print(f"{name} bf16 B{Bn} {g.out_h[i]}x{g.out_w[i]}: act_bytes {p.act_bytes / 2**30:.2f} GiB")


@contextlib.contextmanager
def _host_only_forward(monkeypatch):
    """model_forward's orchestration on dry (host-buffer) plans: the launches are no-ops"""
    monkeypatch.setattr(engine.Plan, "run", lambda self, n=None: None)
    monkeypatch.setattr(torch.cuda, "device", lambda d: contextlib.nullcontext())
    monkeypatch.setattr(tta, "scale_img", lambda x, g, i, out=None, n=None: out)
    monkeypatch.setattr(tta, "merge", lambda ys, g, out=None: torch.zeros(ys[0].shape[0], g.A_tot, ys[0].shape[2]))
    yield


@pytest.mark.parametrize("max_batch", [None, 4])
def test_augment_adds_two_plan_keys_and_branch_0_reuses_the_plain_one(dry, monkeypatch, max_batch):
    m = YOLO.from_yaml(ROOT / "configs/models/gelan-c.yaml").eval().set_precision("fp32")
    m.max_batch = max_batch
    x = torch.zeros(2, 3, 128, 128)
    with _host_only_forward(monkeypatch):
        y_plain, _ = engine.run_forward(m, x, max_batch)
        plain = set(m._plans)
        y, none = tta.forward_augment(m, x, max_batch)
        keys = set(m._plans)
        assert none is None and tuple(y.shape) == (2, 84, tta.geometry(128, 128).A_tot)
        assert plain < keys and len(keys - plain) == 2
        tta.forward_augment(m, x[:1] if max_batch else x, max_batch)       # a second call compiles nothing
        assert set(m._plans) == keys
    g = tta.geometry(128, 128)
    rows = max_batch or 2
    shapes = sorted(k[0] for k in keys - plain)
    assert shapes == sorted((rows, 3, g.out_h[i], g.out_w[i]) for i in (1, 2))
    assert len(m._tta) == 1
    # branch 1 has the input's own shape here (0.83 x 128 pads back to 128): its plan is its own all the same
    assert (g.out_h[1], g.out_w[1]) == (128, 128)


def test_dual_head_runs_every_branch_on_main_only_plans(dry, monkeypatch):
    m = YOLO.from_yaml(ROOT / "configs/models/yolov9-c.yaml").eval().set_precision("fp32")
    x = torch.zeros(1, 3, 64, 96)
    with _host_only_forward(monkeypatch):
        tta.forward_augment(m, x, None)
    assert len(m._plans) == 3 and all(k[5] is True for k in m._plans)     # plan_key's main_only field
    for p in m._plans.values():
        assert p.result[0] == "single"


def _upstream_augment(forward, x):
    """YOLOv5 models/yolo.py _forward_augment / _descale_pred / _clip_augmented on [B, A, no] rows, as upstream has them"""
    img_size = x.shape[-2:]
    s = [1, 0.83, 0.67]
    f = [None, 3, None]
    y = []
    for si, fi in zip(s, f):
        xi = T.scale_img(x.flip(fi) if fi else x, si, gs=32)
        yi = forward(xi).permute(0, 2, 1).contiguous()
        yi[..., :4] /= si
        if fi == 3:
            yi[..., 0] = img_size[1] - yi[..., 0]
        y.append(yi)
    nl = 3
    g = sum(4 ** x for x in range(nl))
    e = 1
    i = (y[0].shape[1] // g) * sum(4 ** x for x in range(e))
    y[0] = y[0][:, :-i]
    i = (y[-1].shape[1] // g) * sum(4 ** (nl - 1 - x) for x in range(e))
    y[-1] = y[-1][:, i:]
    return torch.cat(y, 1), None


def test_oracle_equals_upstream_on_a_gelan_c_forward(gelan_c):
    nodes, nc, sd = gelan_c
    x = G.fractal(2, 128, torch.Generator().manual_seed(8))
    fwd = lambda xi: G.forward(nodes, nc, sd, xi)[0]
    y, none = T.forward_augment(fwd, x)
    y_up, _ = _upstream_augment(fwd, x)
    assert none is None and y.shape == (2, 84, tta.geometry(128, 128).A_tot)
    assert torch.equal(y, y_up.permute(0, 2, 1))
    # the merge of the oracle on its own: windows of the branches in order, x of the mirrored branch reflected
    ys = [fwd(xi) for xi in T.branch_inputs(x)]
    g = tta.geometry(128, 128)
    off = g.a_end[0] - g.a_begin[0]
    mid = y[:, :, off:off + g.A[1]]
    s = torch.tensor(np.float32(0.83))
    assert torch.equal(mid[:, 0], 128 - ys[1][:, 0] / s) and torch.equal(mid[:, 4:], ys[1][:, 4:])


@pytest.mark.parametrize("B,h,w,flip", [(2, 64, 96, False), (2, 64, 96, True), (1, 384, 640, True), (1, 640, 640, False),
                                        (3, 128, 128, True)])
def test_k12_formula_agrees_with_torch_interpolate(B, h, w, flip):
    x = G.fractal(B, h, torch.Generator().manual_seed(h + w), w=w)
    for i in (1, 2):
        ref = T.scale_img(x.flip(3) if flip else x, T.SCALES[i])
        got = T.scale_img_exact(x.numpy(), T.SCALES[i], flip)
        assert got.shape == tuple(ref.shape)
        assert np.abs(got - ref.numpy()).max() <= 1e-6, (i, np.abs(got - ref.numpy()).max())


def test_ctypes_structs_match_the_c_header(tmp_path):
    structs = {"yre_tta_geom": (L.TtaGeom, ["h", "w", "scale", "flip", "rh", "rw", "out_h", "out_w", "A", "a_begin", "a_end",
                                            "A_tot"]),
               "yre_tta_scale_desc": (L.TtaScaleDesc, ["x_nchw", "x_u8_hwc", "B", "n", "H", "W", "flip", "rh", "rw", "out_h",
                                                       "out_w", "y"]),
               "yre_tta_merge_branch": (L.TtaMergeBranch, ["y", "A", "a_begin", "a_end", "scale", "flip_w"]),
               "yre_tta_merge_desc": (L.TtaMergeDesc, ["br", "B", "n", "nc", "out"])}
    lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{ROOT / "include" / "yre.h"}"', "int main(void) {"]
    for name, (_, fields) in structs.items():
        lines.append(f'  printf("{name} %zu\\n", sizeof({name}));')
        for f in fields:
            lines.append(f'  printf("{name}.{f} %zu\\n", offsetof({name}, {f}));')
    lines += ["  return 0;", "}"]
    src = tmp_path / "abi.c"
    src.write_text("\n".join(lines))
    subprocess.run(["gcc", "-o", str(tmp_path / "abi"), str(src)], check=True)
    out = subprocess.run([str(tmp_path / "abi")], check=True, capture_output=True, text=True).stdout
    got = dict(l.split() for l in out.strip().splitlines())
    for name, (ct, fields) in structs.items():
        assert int(got[name]) == C.sizeof(ct), name
        for f in fields:
            assert int(got[f"{name}.{f}"]) == getattr(ct, f).offset, f"{name}.{f}"
