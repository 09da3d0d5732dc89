"""Multi-label NMS without a GPU: the three oracle restatements agree bit for bit (tests/nms_ml_oracle.py), multi-label
equals single-label where every anchor has at most one candidate class, the path model drives K7's select kernel down
every way to its sorted candidates (tests/nms_ml_path_cases.py), and the C ABI's arithmetic and refusals."""
import ctypes as C

import numpy as np
import pytest

from oracle import nms_ref as N
from tests import nms_ml_oracle as O
from tests import nms_ml_path_cases as M
from tests import nms_path_cases as P

import yolo_b200  # noqa: F401
from yolo_b200 import _lib

PATHS = ("smem", "sampled", "overflow", "redo")


def _same(a, b):
    (da, ka), (db, kb) = a, b
    return da.shape == db.shape and np.array_equal(da.view(np.uint32), db.view(np.uint32)) and np.array_equal(ka, kb)


# ---- the oracle -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(M.CASES))
def test_c_oracle_equals_numpy_and_torchvision(name):
    """C == numpy restatement == (cls > conf).nonzero() + the reference's offset + torchvision.ops.nms, on every image that
    the O(n * keeps) restatements can afford"""
    pytest.importorskip("torchvision")
    c = M.CASES[name]
    pred = M.pred_of(name).numpy()
    for b in range(pred.shape[0]):
        got = O.nms_image_c(pred[b], multi_label=True, **c.kw)
        if M.paths_of(name)[b].n > 20000:
            continue
        assert _same(got, O.nms_image_numpy(pred[b], multi_label=True, **c.kw)), (name, b)
        assert _same(got, O.nms_image_torch(pred[b], **c.kw)), (name, b)


def test_oracle_cases_cover_the_semantics():
    """several classes of one anchor kept; equal scores across classes of one anchor and across anchors; keeps beyond
    max_det; zero candidates; nc % 4 != 0; a class list with duplicates, absent classes and classes >= nc"""
    def kept(name, b=0):
        pred = M.pred_of(name).numpy()[b]
        return O.nms_image_c(pred, multi_label=True, **M.CASES[name].kw)

    d, k = kept("ml_several_classes")
    assert len(k) > len(set(k.tolist()))                              # one anchor, several rows
    d, k = kept("ml_ties")
    same_anchor_tie = any(np.sum((k == a) & (d[:, 4] == s)) > 1 for a, s in zip(k, d[:, 4]))
    assert same_anchor_tie and len(set(d[:, 4].tolist())) < len(d) // 4
    assert len(kept("ml_empty", 0)[0]) == 0 and len(kept("ml_empty", 1)[0]) > 0
    for md in (300, 1000, 4096):
        assert M.paths_of(f"ml_maxdet{md}")[0].kept == md < M.paths_of(f"ml_maxdet{md}")[0].n
    assert {1, 5, 81} <= {M.pred_of(n).shape[2] - 4 for n in M.CASES}
    cl = M.CASES["ml_classes"].kw["classes"]
    assert len(set(cl)) < len(cl) and max(cl) >= M.pred_of("ml_classes").shape[2] - 4
    d, _ = kept("ml_classes")
    assert set(d[:, 5].astype(int).tolist()) <= set(cl)
    assert (M.pred_of("ml_leaky").numpy()[0, :, 0] < -20).any()       # boxes reaching below -0.5


def test_leaky_boxes_suppress_across_classes():
    """with x1, y1 < -0.5 the class offset does not separate the classes: the reference suppresses across them, which is
    what the leaky case exercises (fewer keeps than with agnostic-free separation)"""
    pred = M.pred_of("ml_leaky").numpy()[0]
    kw = dict(M.CASES["ml_leaky"].kw)
    d, k = O.nms_image_c(pred, multi_label=True, **kw)
    far = pred.copy()
    far[:, 0:2] += 1000.0                                             # same boxes, no negative coordinates
    d2, _ = O.nms_image_c(far, multi_label=True, **kw)
    assert len(d) != len(d2) or not np.array_equal(d[:, 4:], d2[:, 4:])


def test_multi_label_equals_single_label_where_it_must():
    """nc = 1, and inputs with at most one class above the threshold per anchor (the single-label path cases at conf
    0.001 give every other class a score below 9e-4): the keys (score, a * nc + c) sort as (score, a)"""
    rng = np.random.default_rng(0)
    for nc in (1,):
        p = M.sparse_image(3000, nc, 1, per_anchor=1, n_anchors=2500)
        for kw in (dict(conf_thres=0.001, iou_thres=0.45), dict(conf_thres=0.3, iou_thres=0.6, agnostic=True)):
            assert _same(O.nms_image_c(p, multi_label=True, **kw), N.nms_image_c(p, **kw))
    for name in ("nc5", "nc81", "classes_odd", "grid_dup_maxdet513", "band_0.45", "cross_class_below", "overflow_classes"):
        c = P.CASES[name]
        pred = P.pred_of(name).numpy()
        for b in range(pred.shape[0]):
            sc = pred[b, :, 4:]
            assert ((sc > np.float32(c.kw["conf_thres"])).sum(1) <= 1).all(), name
            assert _same(O.nms_image_c(pred[b], multi_label=True, **c.kw), N.nms_image_c(pred[b], **c.kw)), (name, b)
    p = rng.uniform(0, 1, (64, 4 + 1)).astype(np.float32)
    assert _same(O.nms_image_numpy(p, multi_label=True), N.nms_image_numpy(p))


# ---- the path model ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(M.CASES))
def test_model_matches_case_name(name):
    got = tuple(p.path for p in M.paths_of(name))
    assert got == M.CASES[name].expect, (name, M.paths_of(name))


def test_every_path_is_covered():
    found = {p.path for name in M.CASES for p in M.paths_of(name)}
    assert set(PATHS) <= found, f"no determinate multi-label case takes {set(PATHS) - found}"
    assert any(set(PATHS) <= {p.path for p in M.paths_of(n)} for n in M.CASES)


def test_sort_global_features_are_covered():
    """agnostic (prune off), a class filter, fused scale rows, nc = 80 and B > 1 each reach sort_global on its two ways"""
    feats = {path: set() for path in M.SORT_GLOBAL}
    for name, c in M.CASES.items():
        ps = M.paths_of(name)
        for p in ps:
            if p.path in M.SORT_GLOBAL:
                f = feats[p.path]
                f.add("prune" if p.prune else "no_prune")
                f |= {k for k in ("agnostic", "classes") if c.kw.get(k)}
                f |= {"scale"} if c.scale else set()
                f |= {"batch"} if len(ps) > 1 else set()
                f |= {"nc80"} if M.pred_of(name).shape[2] == 84 else set()
    assert {"prune", "scale", "batch", "nc80"} <= feats["overflow"] and {"no_prune", "agnostic"} <= feats["overflow"]
    assert {"prune", "scale", "batch", "nc80", "classes"} <= feats["redo"]


def test_indeterminate_samples_are_reported():
    """above SMEM_KEYS candidates the sample depends on warp order unless every pair is a candidate, A % 32 == 0 and
    stride | 32 * nc"""
    p = M.overflow_image(2048, 8, 1, 4)
    assert M.select_path(p[:2040], conf_thres=0.001).path == "indeterminate"       # A not a multiple of 32
    q = p.copy()
    q[5, 6] = 0.0                                                                    # one pair not a candidate
    assert M.select_path(q, conf_thres=0.001).path == "indeterminate"
    r = M.dense_image(2048, 5, 3)                                                    # n = 10240: stride 3 does not divide 160
    assert M.select_path(r, conf_thres=0.001).path == "indeterminate"
    assert M.select_path(p, conf_thres=0.001).path == "overflow"


def test_model_reads_the_kernel_constants():
    src = P.KNMS.read_text()
    k = P.kernel_constants(src)
    redo, over = M.pred_of("ml_redo")[0].numpy(), M.pred_of("ml_overflow")[0].numpy()
    assert M.select_path(redo, **M.CASES["ml_redo"].kw, consts=k).path == "redo"
    sm = P.kernel_constants(src.replace(f"SMEM_KEYS = {k['SMEM_KEYS']};", "SMEM_KEYS = 16384;"))
    assert M.select_path(over, **M.CASES["ml_overflow"].kw, consts=sm).path == "smem"


# ---- C ABI --------------------------------------------------------------------------------------------------------------
def test_symbols_and_workspace_arithmetic():
    lib = _lib.lib()
    for name in ("yre_nms_multi_label_workspace_bytes", "yre_nms_batched_multi_label", "yre_nms_multi_label_filter_only"):
        assert hasattr(lib, name) and name in _lib.SYMBOLS
    ws = lib.yre_nms_multi_label_workspace_bytes
    assert ws(64, 8400, 80) == 8 * 64 * (1 << 20) + 8 * 64 + 256             # 672 000 pairs -> 2^20 keys: 537 MB
    assert ws(16, 33600, 80) == 8 * 16 * (1 << 22) + 8 * 16 + 256            # 2 688 000 pairs -> 2^22 keys
    assert ws(2, 8400, 1) == 8 * 2 * 16384 + 16 + 256
    assert ws(1, 1 << 24, 64) > 0 and ws(1, (1 << 24) + 1, 64) == 0          # A * nc up to 2^30
    assert ws(0, 10, 10) == ws(1, 0, 10) == ws(1, 10, 0) == 0


def test_refusals_without_gpu():
    lib = _lib.lib()
    assert lib.yre_nms_batched_multi_label(None, None) == -1
    assert lib.yre_nms_multi_label_filter_only(None, None) == -1
    fake = 1 << 20                                                              # never dereferenced: the checks fail first
    d = _lib.NmsDesc(fake, 1, 1 << 25, 33, 0.001, 0.7, 300, None, -1, 0, fake, fake, fake, fake, 1 << 62, None)
    assert lib.yre_nms_batched_multi_label(C.byref(d), None) == -3 and b"multi-label" in lib.yre_last_error()
    assert lib.yre_nms_multi_label_filter_only(C.byref(d), None) == -3
    d.A = 1 << 24
    d.nc = 65                                                                   # 2^30 + 2^24 pairs
    assert lib.yre_nms_batched_multi_label(C.byref(d), None) == -3
    d.nc, d.workspace_bytes = 64, 16                                            # within the limit, workspace too small
    assert lib.yre_nms_batched_multi_label(C.byref(d), None) == -1
