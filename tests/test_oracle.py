"""CPU tests that pin the ORACLE: against fixtures produced by the real reference
(tests/golden/), against the reference's own live known-answer tests (tests/test_heads.py in
the reference checkout) and against torchvision."""
import json
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import gelan_ref as G
from oracle import nms_ref as N
from tests.cases import NMS_CASES, make_pred

GOLD = Path(__file__).parent / "golden"


# ---- known answers the reference's own tests hold (reference tests/test_heads.py) -----------
def test_anchor_known_answers():
    pts, st = G.anchors_and_strides([(80, 80), (40, 40), (20, 20)], [8, 16, 32], torch.float32)
    assert pts.shape == (8400, 2) and st.shape == (8400, 1)            # test_heads.py:42-44
    assert pts[0].tolist() == [0.5, 0.5]                               # test_heads.py:46-49
    assert st[:6400].eq(8).all() and st[6400:8000].eq(16).all() and st[8000:].eq(32).all()  # :51-55


def test_dfl_range_and_known_box():
    w = torch.arange(16.).view(1, 16, 1, 1)
    e = G.dfl_expectation(torch.randn(2, 64, 100, generator=torch.Generator().manual_seed(0)) * 3, w)
    assert e.shape == (2, 4, 100) and e.min() >= 0 and e.max() <= 15   # test_heads.py:19-27
    # ltrb = 1 at anchor (5,5): xyxy (4,4,6,6) (test_heads.py:71-79) == xywh (5,5,2,2); stride 1.
    # A one-hot-at-bin-1 distribution makes the DFL expectation exactly 1.
    raw = torch.full((1, 64 + 2, 11, 11), -1e4)
    raw[:, 1:64:16] = 1e4
    y = G.decode([raw], [1.0], 2, w)
    a = 5 * 11 + 5 - 0  # anchor at x=5.5,y=5.5 -> use exact arithmetic instead:
    assert torch.allclose(y[0, :4, a], torch.tensor([5.5, 5.5, 2.0, 2.0]))


# ---- network forward vs reference-generated fixtures ------------------------------------------
@pytest.mark.parametrize("name,fix", [("gelan-c_128", "gelan_c"), ("gelan-c_640", "gelan_c"), ("yolov9-c_64", "yolov9_c")])
def test_forward_matches_reference_fixture(name, fix, request):
    nodes, nc, sd = request.getfixturevalue(fix)
    gd = np.load(GOLD / f"{name}.npz", allow_pickle=False)
    x = G.fractal(int(gd["batch"]), int(gd["size"]), torch.Generator().manual_seed(int(gd["seed"])))
    cap = {}
    y, raws = G.forward(nodes, nc, sd, x, capture=cap)
    if isinstance(y, list):
        y, raws = y[1], raws[1]
    sa = int(gd["stride_a"])
    # Same torch build => bit-equal here; a different host CPU may pick other conv kernels, so
    # the gate is the reference's own fp32-vs-fp64 floor recorded in the fixture (x4 slack).
    tol_box = max(4 * float(gd["floor_box"]), 1e-3)
    tol_sc = max(4 * float(gd["floor_score"]), 1e-5)
    ysub = y[:, :, ::sa].numpy()
    assert np.abs(ysub[:, :4] - gd["y_sub"][:, :4]).max() <= tol_box
    assert np.abs(ysub[:, 4:] - gd["y_sub"][:, 4:]).max() <= tol_sc
    for n, am in zip(gd["layer_names"], gd["layer_absmean"]):
        assert abs(cap[str(n)].abs().mean().item() - am) <= 1e-4 * max(am, 1e-3), n
    for i, r in enumerate(raws):
        s = max(1, sa // 2)
        assert np.abs(r[:, :, ::s, ::s].numpy() - gd[f"raw{i}_sub"]).max() <= 1e-3
    if sa == 1:   # detections of the reference's NMS on the reference's y
        dets = N.non_max_suppression(torch.from_numpy(gd["y_sub"]).permute(0, 2, 1).contiguous(), 0.25, 0.45)
        for i, d in enumerate(dets):
            assert np.array_equal(d, gd[f"det{i}"])


# ---- NMS ------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(NMS_CASES))
@pytest.mark.parametrize("impl", ["numpy", "c"])
def test_nms_matches_reference_fixture(name, impl):
    gd = np.load(GOLD / "nms_cases.npz")
    c = NMS_CASES[name]
    p = make_pred(c)
    dets, keeps = N.non_max_suppression(p, impl=impl, return_keep=True, **c["kw"])
    for i, (d, k) in enumerate(zip(dets, keeps)):
        assert np.array_equal(d, gd[f"{name}.{i}"]), (name, i)
        assert np.array_equal(p[i, k, 4:].max(1).values.numpy(), d[:, 4])   # keep indices point at the rows


def test_greedy_nms_equals_torchvision():
    tv = pytest.importorskip("torchvision")
    g = torch.Generator().manual_seed(0)
    for quant in (None, 16):
        b = torch.rand(1500, 4, generator=g) * 300
        b[:, 2:] = b[:, :2] + torch.rand(1500, 2, generator=g) * 120
        s = torch.rand(1500, generator=g)
        if quant:
            s = torch.round(s * quant) / quant
        for thr in (0.0, 0.3, 0.45, 0.7):
            assert np.array_equal(tv.ops.nms(b, s, thr).numpy(), N.greedy_nms_numpy(b.numpy(), s.numpy(), thr))


# ---- the reference's parameter schema and detect strides ------------------------------------------
FULL_RES_FIXTURE = {"gelan-c": "gelan-c_128", "yolov9-c": "yolov9-c_64"}      # stored with stride_a = 1


@pytest.mark.parametrize("cfg,fix", [("gelan-c", "gelan_c"), ("yolov9-c", "yolov9_c")])
def test_bit_equal_to_reference(cfg, fix, request):
    """Exact agreement with what the reference itself produced: its state_dict keys in its order (ckpt_keys.json lists
    them in the order of the reference model's state_dict(), make_golden_ckpt.py) and its detect strides (input size over
    the map size of each raw output of its forward at full resolution, make_golden.py)."""
    nodes, nc, _ = request.getfixturevalue(fix)
    ref_keys = [r for _, r in json.loads((GOLD / "ckpt_keys.json").read_text())[cfg]]
    assert ref_keys == list(G.param_schema(nodes, nc).keys())
    gd = np.load(GOLD / f"{FULL_RES_FIXTURE[cfg]}.npz", allow_pickle=False)
    assert int(gd["stride_a"]) == 1
    S, levels = int(gd["size"]), sorted(k for k in gd.files if k.startswith("raw"))
    ref_strides = [S // gd[k].shape[-1] for k in levels]
    assert [S // gd[k].shape[-2] for k in levels] == ref_strides
    assert G.detect_strides(nodes) == ref_strides


# ---- pre/post-processing oracle (SURVEY.md 8f row 1) -------------------------------------------------------
import hashlib  # noqa: E402

from oracle import preproc_ref as P  # noqa: E402
from tests.cases import PREPROC_CASES, preproc_boxes, preproc_image  # noqa: E402

PRE_GOLD = np.load(Path(__file__).resolve().parent / "golden" / "preproc_cases.npz")


@pytest.mark.parametrize("name", list(PREPROC_CASES))
def test_preproc_oracle_matches_reference_fixture(name):
    """oracle letterbox / preprocess / scale_boxes == what the REFERENCE's functions produced (make_golden_preproc.py)."""
    h, w, S, seed = PREPROC_CASES[name]
    img = preproc_image(h, w, seed)
    lb, ratio, pad = P.letterbox(img, S)
    assert lb.shape == (S, S, 3)
    assert hashlib.sha256(lb.tobytes()).digest() == PRE_GOLD[f"{name}/sha"].tobytes()
    assert np.array_equal(lb[[0, S // 3, S - 1]], PRE_GOLD[f"{name}/rows"])
    x, _, _ = P.preprocess(img, S)
    assert hashlib.sha256(x.tobytes()).digest() == PRE_GOLD[f"{name}/x_sha"].tobytes()
    assert ratio[0] == PRE_GOLD[f"{name}/ratio"][0] and tuple(PRE_GOLD[f"{name}/pad"]) == pad
    b = preproc_boxes(S, seed)
    assert np.array_equal(P.scale_boxes(b, (S, S), (h, w), (ratio, pad)), PRE_GOLD[f"{name}/boxes_rp"])
    assert np.array_equal(P.scale_boxes(b, (S, S), (h, w)), PRE_GOLD[f"{name}/boxes_none"])


def test_resize_restatement_matches_cv2_when_available():
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(0)
    for h, w, dw, dh in [(37, 53, 1280, 894), (375, 500, 640, 480), (1079, 1919, 640, 360), (64, 48, 32, 24), (7, 9, 64, 50),
                         (200, 300, 299, 199), (50, 50, 51, 49)]:
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        assert np.array_equal(P.resize_linear_u8(img, dw, dh), cv2.resize(img, (dw, dh), interpolation=cv2.INTER_LINEAR)), (h, w, dw, dh)


def test_letterbox_geometry_c_helper_matches_python_arithmetic():
    """yre_letterbox_geometry (host arithmetic in libyre, no GPU) == the reference's Python rounding for many sizes."""
    import ctypes as C
    import yolo_b200  # noqa: F401
    from yolo_b200 import _lib as L
    rng = np.random.default_rng(3)
    sizes = [(480, 640, 640), (481, 641, 640), (1, 1, 640), (5, 1000, 640), (1000, 5, 640), (1281, 1279, 1280)]
    sizes += [(int(h), int(w), 640) for h, w in rng.integers(8, 4000, (300, 2))]
    for h, w, S in sizes:
        nw, nh, top, left, bottom, right, r, pad = P.letterbox_geometry(h, w, S)
        d = L.LetterboxDesc(); d.h, d.w, d.new_shape = h, w, S
        rr, pw, ph = C.c_double(), C.c_int32(), C.c_int32()
        rc = L.lib().yre_letterbox_geometry(C.byref(d), C.byref(rr), C.byref(pw), C.byref(ph))
        if nw <= 0 or nh <= 0:
            assert rc != 0
            continue
        assert rc == 0, (h, w, S, L.lib().yre_last_error())
        assert (d.new_w, d.new_h, d.top, d.left, rr.value, (pw.value, ph.value)) == (nw, nh, top, left, r, pad), (h, w, S)


# ---- detection-metric oracle (SURVEY.md 8f row 3) -------------------------------------------------------------
from oracle import metrics_ref as MR  # noqa: E402
from tests.cases import METRIC_CASES, metric_case  # noqa: E402

MET_GOLD = np.load(Path(__file__).resolve().parent / "golden" / "metrics_cases.npz")


@pytest.mark.parametrize("name", list(METRIC_CASES))
def test_metrics_oracle_matches_reference_fixture(name):
    """oracle compute_map == the REFERENCE's compute_map, bit for bit in float64 (make_golden_metrics.py)."""
    a = metric_case(name)
    r, r7 = MR.compute_map(*a), MR.compute_map(*a, iou_thresholds=[0.7])
    assert np.array_equal(np.array([r["map50"], r["map75"], r["map"], r7["map"]]), MET_GOLD[name])


def test_metrics_host_aggregation_matches_oracle():
    """The vectorised AP / aggregation used by the product (yolo_b200.metrics._aggregate, host numpy) fed with the ORACLE's
    match flags reproduces the oracle's result bit for bit -- checks the host half of the fast path without a GPU."""
    import yolo_b200  # noqa: F401
    from yolo_b200.metrics import _aggregate
    for name in METRIC_CASES:
        pb, ps, pc, gb, gc, nc = metric_case(name)
        thr = [0.5 + 0.05 * i for i in range(10)]
        tp = np.concatenate([MR.match_image(pb[i], pc[i], gb[i], gc[i], thr) for i in range(len(pb))]) if sum(map(len, pb)) else np.zeros((0, 10), np.uint8)
        off = np.concatenate([[0], np.cumsum([len(x) for x in pb])]).astype(np.int32)
        got = _aggregate(np.concatenate(ps), np.concatenate(pc), tp, off, gc, nc, thr)
        ref = MR.compute_map(pb, ps, pc, gb, gc, nc)
        assert got == ref, name
