"""Rectangular ("rect") inference without a GPU: the letterbox geometry for a target (new_h, new_w) and a stride, the
tcgen05 kernel selection of non-square full-size plans, and the wiring of a non-square plan against the oracle."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import gelan_ref as G
from oracle import preproc_ref as P
from tests import cpu_plan_exec as X
from tests.conftest import ROOT
from tests.test_cpu_conv_tc_select import tc_variant

from yolo_b200 import YOLO, _lib as L, engine


def rect_geometry(h: int, w: int, new_h: int, new_w: int, stride: int = 0):
    """(new_w, new_h, top, left, out_h, out_w, r, (pad_w, pad_h)): scripts/detect.py:57-71 for a (new_h, new_w) target,
    with YOLOv9's letterbox(auto=True) padding (modulo stride) when stride > 0."""
    r = min(new_h / h, new_w / w)
    nw, nh = int(round(w * r)), int(round(h * r))
    dw, dh = new_w - nw, new_h - nh
    if stride > 0:
        dw, dh = np.mod(dw, stride), np.mod(dh, stride)
    dw, dh = dw / 2, dh / 2
    top, bottom = int(round(dh - 0.1)), int(round(dh + 0.1))
    left, right = int(round(dw - 0.1)), int(round(dw + 0.1))
    return nw, nh, top, left, nh + top + bottom, nw + left + right, r, (int(dw), int(dh))


def letterbox_rect(img: np.ndarray, new_h: int, new_w: int, stride: int = 0, color=(114, 114, 114)):
    """numpy letterbox to a rectangle -> (padded uint8 HWC image, (r, r), (pad_w, pad_h)); the resize is the oracle's
    restatement of cv2.resize(INTER_LINEAR)."""
    h, w = img.shape[:2]
    nw, nh, top, left, oh, ow, r, pad = rect_geometry(h, w, new_h, new_w, stride)
    if (w, h) != (nw, nh):
        img = P.resize_linear_u8(img, nw, nh)
    out = np.empty((oh, ow, 3), np.uint8)
    out[...] = np.asarray(color, np.uint8)
    out[top:top + nh, left:left + nw] = img
    return out, (r, r), pad


def c_geometry(h: int, w: int, new_h: int, new_w: int, stride: int):
    d = L.LetterboxDesc()
    d.h, d.w = h, w
    r, pw, ph = C.c_double(), C.c_int32(), C.c_int32()
    rc = L.lib().yre_letterbox_geometry_rect(C.byref(d), new_h, new_w, stride, C.byref(r), C.byref(pw), C.byref(ph))
    if rc != 0:
        return None
    return d.new_w, d.new_h, d.top, d.left, d.out_h, d.out_w, r.value, (pw.value, ph.value)


GEOMETRY_SIZES = [(1080, 1920), (1920, 1080), (480, 640), (640, 480), (100, 150), (37, 53), (1, 1), (1, 7), (7, 1),
                  (5, 1000), (1000, 5), (999, 1333), (1333, 999), (641, 641), (2160, 3840), (333, 1)]
TARGETS = [(640, 640), (384, 640), (640, 384), (736, 1280), (1280, 1280), (321, 517), (32, 32)]


@pytest.mark.parametrize("stride", [0, 32, 64])
def test_rect_geometry_matches_the_numpy_rule(stride):
    rng = np.random.default_rng(stride)
    sizes = GEOMETRY_SIZES + [(int(h), int(w)) for h, w in rng.integers(1, 4000, (200, 2))]
    checked = 0
    for h, w in sizes:
        for new_h, new_w in TARGETS:
            ref = rect_geometry(h, w, new_h, new_w, stride)
            got = c_geometry(h, w, new_h, new_w, stride)
            if ref[0] <= 0 or ref[1] <= 0:
                assert got is None, (h, w, new_h, new_w)
                continue
            assert got == ref, (h, w, new_h, new_w, stride, got, ref)
            nw, nh, top, left, oh, ow, r, pad = got
            assert top + nh <= oh <= new_h and left + nw <= ow <= new_w
            if stride:
                assert (new_h - oh) % stride == 0 and (new_w - ow) % stride == 0
            checked += 1
    assert checked > 1000


def test_auto_rect_of_a_video_frame():
    """1920x1080 at 640: 640x384 with 12 rows above and below (the FLOP ratio 0.6 of the square letterbox)."""
    assert c_geometry(1080, 1920, 640, 640, 32) == (640, 360, 12, 0, 384, 640, 1 / 3, (0, 12))
    assert c_geometry(1920, 1080, 640, 640, 32) == (360, 640, 0, 12, 640, 384, 1 / 3, (12, 0))
    assert c_geometry(1080, 1920, 640, 640, 64) == (640, 360, 12, 0, 384, 640, 1 / 3, (0, 12))
    assert c_geometry(1080, 1920, 640, 640, 0)[4:6] == (640, 640)


def test_square_target_without_stride_equals_the_square_geometry():
    """(S, S, 0) is yre_letterbox_geometry for every size tests/test_oracle.py checks against the reference's rounding."""
    rng = np.random.default_rng(3)
    sizes = [(480, 640, 640), (481, 641, 640), (1, 1, 640), (5, 1000, 640), (1000, 5, 640), (1281, 1279, 1280)]
    sizes += [(int(h), int(w), 640) for h, w in rng.integers(8, 4000, (300, 2))]
    for h, w, S in sizes:
        d = L.LetterboxDesc(); d.h, d.w, d.new_shape = h, w, S
        rr, pw, ph = C.c_double(), C.c_int32(), C.c_int32()
        rc = L.lib().yre_letterbox_geometry(C.byref(d), C.byref(rr), C.byref(pw), C.byref(ph))
        got = c_geometry(h, w, S, S, 0)
        if rc != 0:
            assert got is None
            continue
        assert got == (d.new_w, d.new_h, d.top, d.left, S, S, rr.value, (pw.value, ph.value)), (h, w, S)
        assert (d.out_h, d.out_w) == (S, S)
        nw, nh, top, left, bottom, right, r, pad = P.letterbox_geometry(h, w, S)
        assert got == (nw, nh, top, left, S, S, r, pad)


def test_rect_geometry_rejects_bad_sizes():
    for args in [(0, 10, 640, 640, 0), (10, 10, 0, 640, 0), (10, 10, 640, -1, 32), (10, 10, 640, 640, -32), (1, 4000, 640, 640, 32)]:
        assert c_geometry(*args) is None, args


@pytest.fixture()
def dry():
    engine._ALLOW_CPU_DRY_RUN = True
    yield
    engine._ALLOW_CPU_DRY_RUN = False


@pytest.mark.parametrize("name,Bn,H,W,main_only", [("gelan-c", 64, 384, 640, False), ("gelan-c", 64, 640, 384, False),
                                                   ("gelan-c", 16, 736, 1280, False), ("yolov9-c", 16, 384, 640, False),
                                                   ("yolov9-c", 16, 384, 640, True)])
def test_non_square_full_size_plans_get_a_tcgen05_variant_for_every_conv(dry, name, Bn, H, W, main_only):
    m = YOLO.from_yaml(ROOT / "configs/models" / f"{name}.yaml").eval().set_precision("bf16")
    m.main_only = main_only
    p = engine.compile_model(m, torch.empty(Bn, 3, H, W))
    convs = [a for k, a in p.trace if k == "conv"]
    assert len(convs) > 100
    for a in convs:
        tc_variant(a, 148)                               # asserts that the describe query returns 0
    # a plan is keyed by (B, H, W): the detection head sees H/s x W/s maps, 5040 anchors at 384x640
    kind, y, _ = p.result
    ys = y if kind == "dual" else [y]
    A = sum((H // s) * (W // s) for s in (8, 16, 32))
    assert all(t.shape[:2] == (Bn, A) for t in ys)


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_gelan_c_non_square_plan_wiring(gelan_c, dry, prec):
    nodes, nc, sd = gelan_c
    m = YOLO.from_yaml(ROOT / "configs/models/gelan-c.yaml")
    m.load_state_dict(sd)
    m.eval().set_precision(prec)
    x = G.fractal(2, 96, torch.Generator().manual_seed(6), w=160)
    cap = {}
    y_ref, raws_ref = G.forward(nodes, nc, sd, x, capture=cap)
    p = engine.compile_model(m, x)
    X.run(p)
    _, y, raws = p.result
    assert y.shape == (2, 12 * 20 + 6 * 10 + 3 * 5, 84)
    tol = 2e-4 if prec == "fp32" else 0.5
    for n, v in p.vals.items():
        if isinstance(v, engine.V):
            ref = cap[n]
            assert X.nchw(X.read(v)).shape == ref.shape, n
            err = (X.nchw(X.read(v)) - ref).abs().max().item()
            assert err <= tol * max(1.0, ref.abs().max().item()), (n, err)
    if prec == "fp32":
        yy = y.permute(0, 2, 1)
        assert (yy[:, :4] - y_ref[:, :4]).abs().max() < 2e-2
        assert (yy[:, 4:] - y_ref[:, 4:]).abs().max() < 2e-4
        for r, q in zip(raws, raws_ref):
            assert (r.t.permute(0, 3, 1, 2) - q).abs().max() < 2e-3


@pytest.mark.parametrize("H,W", [(64, 96), (96, 64)])
def test_yolov9_c_non_square_plan_wiring(yolov9_c, dry, H, W):
    """the dual head's CBFuse resizes between non-square maps"""
    nodes, nc, sd = yolov9_c
    m = YOLO.from_yaml(ROOT / "configs/models/yolov9-c.yaml")
    m.load_state_dict(sd)
    m.eval().set_precision("fp32")
    x = G.fractal(1, H, torch.Generator().manual_seed(5), w=W)
    y_ref, _ = G.forward(nodes, nc, sd, x)
    p = engine.compile_model(m, x)
    X.run(p)
    kind, y, _ = p.result
    assert kind == "dual"
    for got, ref in zip(y, y_ref):
        yy = got.permute(0, 2, 1)
        assert yy.shape == ref.shape
        assert (yy[:, :4] - ref[:, :4]).abs().max() < 2e-2 and (yy[:, 4:] - ref[:, 4:]).abs().max() < 2e-4


def test_batch_must_share_the_destination_extent():
    """checked before anything is launched (the pointers are never dereferenced)"""
    descs = (L.LetterboxDesc * 2)()
    for d, (h, w) in zip(descs, [(1080, 1920), (1920, 1080)]):
        d.src, d.dst, d.h, d.w, d.row_pitch = 0x7f0000000000, 0x7f0010000000, h, w, 3 * w
        assert L.lib().yre_letterbox_geometry_rect(C.byref(d), 640, 640, 32, None, None, None) == 0
    assert (descs[0].out_h, descs[0].out_w, descs[1].out_h, descs[1].out_w) == (384, 640, 640, 384)
    assert L.lib().yre_letterbox_u8_batch(descs, 2, None) == -1
    assert b"share the destination extent" in L.lib().yre_last_error()
