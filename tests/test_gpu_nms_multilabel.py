"""Multi-label K7 (yre_nms_batched_multi_label) bit for bit against the C oracle (tests/nms_ml_oracle.c): counts, all six
columns of every kept row and keep_anchor, on every case of tests/nms_ml_path_cases.py (every way the select kernel gets its
sorted candidates; tests/test_cpu_nms_multilabel.py checks which way each takes), on full-size inputs with every pair a
candidate, on a TTA output and through the Evaluator.  multi_label=False stays the single-label path."""
import ctypes as C
import functools
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import gelan_ref as G
from oracle import metrics_ref as MR
from tests import nms_ml_oracle as O
from tests import nms_ml_path_cases as M

pytestmark = pytest.mark.gpu

import yolo_b200
from yolo_b200 import _lib as L

DEV = "cuda"
ROOT = Path(__file__).resolve().parents[1]


@functools.lru_cache(maxsize=None)
def oracle(name):
    return O.non_max_suppression(M.pred_of(name), return_keep=True, multi_label=True, **M.CASES[name].kw)


def assert_matches(dets, keeps, out, counts, keep, what):
    out, counts, keep = out.cpu().numpy(), counts.cpu().numpy(), keep.cpu().numpy()
    assert counts.tolist() == [len(d) for d in dets], (what, counts.tolist(), [len(d) for d in dets])
    for b, (d, k) in enumerate(zip(dets, keeps)):
        n = len(d)
        bad = np.nonzero((out[b, :n].view(np.uint32) != d.view(np.uint32)).any(1))[0]
        assert len(bad) == 0, f"{what} image {b}: {len(bad)} of {n} rows differ, first at row {bad[0]}"
        assert np.array_equal(keep[b, :n], k), (what, b)


@pytest.mark.parametrize("name", list(M.CASES))
def test_multi_label_bit_exact(name):
    c = M.CASES[name]
    pred = M.pred_of(name).to(DEV)
    out, counts, keep = yolo_b200.nms_raw(pred, **c.kw, multi_label=True)
    assert_matches(*oracle(name), out, counts, keep, name)
    dets = yolo_b200.non_max_suppression(pred, **c.kw, multi_label=True)                   # the sync API agrees
    pend = yolo_b200.non_max_suppression_async(pred, **c.kw, multi_label=True).result()    # and the async one
    for b in range(pred.shape[0]):
        n = int(counts[b])
        assert torch.equal(dets[b], out[b, :n]) and torch.equal(pend[b], out[b, :n])
    sc = M.scale_of(name)
    if sc is None:
        return
    fo, fc, fk = yolo_b200.nms_raw(pred, **c.kw, scale=sc.to(DEV), multi_label=True)
    assert torch.equal(fc, counts) and torch.equal(fk, keep)
    for b in range(pred.shape[0]):
        n = int(counts[b])
        pw, ph, gain, ow, oh = sc[b].tolist()
        ref = out[b, :n].clone()
        yolo_b200.scale_boxes(ref[:, :4], None, (oh, ow), ((gain, gain), (pw, ph)))
        assert torch.equal(fo[b, :n].view(torch.int32), ref.view(torch.int32)), (name, b)


@pytest.mark.parametrize("name", [n for n in M.CASES if any(p.path in M.SORT_GLOBAL for p in M.paths_of(n))])
def test_sort_global_ignores_stale_workspace(name):
    """A zeroed workspace holds keys that sort first (index 0, NaN score): sort_global's ~0 padding must keep them out."""
    c = M.CASES[name]
    lib = L.lib()
    pred = M.pred_of(name).to(DEV)
    Bn, A, ch = pred.shape
    md = c.kw.get("max_det", 300)
    ws = torch.zeros((lib.yre_nms_multi_label_workspace_bytes(Bn, A, ch - 4),), dtype=torch.uint8, device=DEV)
    out = torch.empty((Bn, md, 6), dtype=torch.float32, device=DEV)
    counts = torch.empty((Bn,), dtype=torch.int32, device=DEV)
    keep = torch.empty((Bn, md), dtype=torch.int64, device=DEV)
    cls = c.kw.get("classes")
    cls_t = torch.tensor(cls, dtype=torch.int32, device=DEV) if cls is not None else None
    d = L.NmsDesc(pred.data_ptr(), Bn, A, ch - 4, c.kw["conf_thres"], c.kw["iou_thres"], md,
                  cls_t.data_ptr() if cls_t is not None else None, len(cls) if cls is not None else -1,
                  int(bool(c.kw.get("agnostic"))), out.data_ptr(), counts.data_ptr(), keep.data_ptr(), ws.data_ptr(),
                  ws.numel(), None)
    L.check(lib.yre_nms_batched_multi_label(C.byref(d), torch.cuda.current_stream().cuda_stream), "nms")
    assert_matches(*oracle(name), out, counts, keep, name)


@pytest.mark.parametrize("B,A", [(64, 8400), (16, 33600)])
def test_full_size_every_pair_a_candidate(B, A):
    """64 x 8 400 x 84 and 16 x 33 600 x 84 at conf 0.001 with every class score above it: 672 000 / 2 688 000 candidates
    per image"""
    rng = np.random.default_rng(A)
    S = 640.0 if A == 8400 else 1280.0
    p = np.empty((B, A, 84), np.float32)
    p[..., 0:2] = rng.uniform(0, S, (B, A, 2))
    p[..., 2:4] = rng.uniform(4.0, 200.0, (B, A, 2))
    p[..., 4:] = rng.uniform(0.0015, 1.0, (B, A, 80))
    pred = torch.from_numpy(p).to(DEV)
    out, counts, keep = yolo_b200.nms_raw(pred, 0.001, 0.7, multi_label=True)
    dets, keeps = O.non_max_suppression(p, 0.001, 0.7, return_keep=True, multi_label=True)
    assert_matches(dets, keeps, out, counts, keep, f"{B}x{A}")


def test_default_is_single_label():
    """multi_label=False is the call without the argument, bit for bit, and differs from multi-label where anchors have
    several classes above the threshold"""
    for name in ("ml_several_classes", "ml_overflow", "ml_nc5"):
        c = M.CASES[name]
        pred = M.pred_of(name).to(DEV)
        oa, ca, ka = yolo_b200.nms_raw(pred, **c.kw)
        ob, cb, kb = yolo_b200.nms_raw(pred, **c.kw, multi_label=False)
        assert torch.equal(ca, cb)
        for b, n in enumerate(ca.tolist()):
            assert torch.equal(oa[b, :n].view(torch.int32), ob[b, :n].view(torch.int32)) and torch.equal(ka[b, :n], kb[b, :n])
    name = "ml_several_classes"
    _, _, k_ml = yolo_b200.nms_raw(M.pred_of(name).to(DEV), **M.CASES[name].kw, multi_label=True)
    _, _, k_sl = yolo_b200.nms_raw(M.pred_of(name).to(DEV), **M.CASES[name].kw)
    assert not torch.equal(k_ml, k_sl)


def _gelan():
    from yolo_b200 import YOLO
    nodes, nc = G.load_graph(ROOT / "configs/models/gelan-c.yaml")
    m = YOLO.from_yaml(ROOT / "configs/models/gelan-c.yaml")
    m.load_state_dict(G.calibrated_state_dict(nodes, nc))
    return m, nc


def test_tta_output_through_multi_label():
    m, _ = _gelan()
    m = m.to(DEV).eval().set_precision("bf16")
    x = G.fractal(2, 256, torch.Generator().manual_seed(9)).to(DEV)
    y, _ = m(x, augment=True)
    pred = y.permute(0, 2, 1).contiguous()
    for conf, iou in ((0.001, 0.7), (0.25, 0.45)):
        out, counts, keep = yolo_b200.nms_raw(pred, conf, iou, multi_label=True)
        dets, keeps = O.non_max_suppression(pred.cpu(), conf, iou, return_keep=True, multi_label=True)
        assert sum(len(d) for d in dets) > 0
        assert_matches(dets, keeps, out, counts, keep, f"tta {conf}")


def test_evaluator_multi_label_matches_oracle_map():
    """Evaluator(multi_label=True) == the oracle's compute_map on the oracle's multi-label detections of the same y"""
    from yolo_b200 import Evaluator
    m, nc = _gelan()
    rng = np.random.default_rng(5)
    S, batches = 256, []
    for bi in range(2):
        imgs = G.fractal(3, S, torch.Generator().manual_seed(30 + bi))
        rows = []
        for i in range(3):
            k = int(rng.integers(0, 6))
            cxy, wh = rng.uniform(0.2, 0.8, (k, 2)), rng.uniform(0.05, 0.4, (k, 2))
            rows += [[i, int(rng.integers(0, nc)), *cxy[j], *wh[j]] for j in range(k)]
        batches.append((imgs, torch.tensor(rows, dtype=torch.float32).reshape(-1, 6), None, [(S, S)] * 3))
    got = Evaluator(m, batches, num_classes=nc, conf_thres=0.01, iou_thres=0.6, multi_label=True).evaluate()
    pb, ps, pc, gb, gc = [], [], [], [], []
    m = m.cuda().eval()
    n_multi = 0
    for imgs, targets, _, _ in batches:
        y, _ = m(imgs.cuda())
        dets, keeps = O.non_max_suppression(y.permute(0, 2, 1).contiguous().cpu(), 0.01, 0.6, return_keep=True,
                                            multi_label=True)
        for i in range(imgs.shape[0]):
            d = dets[i]
            n_multi += len(keeps[i]) - len(set(keeps[i].tolist()))
            pb.append(d[:, :4]); ps.append(d[:, 4]); pc.append(d[:, 5].astype(np.int64))
            t = targets[targets[:, 0] == i]
            xywh = t[:, 2:6].clone()
            xywh[:, [0, 2]] *= S; xywh[:, [1, 3]] *= S
            xyxy = torch.zeros_like(xywh)
            xyxy[:, 0] = xywh[:, 0] - xywh[:, 2] / 2; xyxy[:, 1] = xywh[:, 1] - xywh[:, 3] / 2
            xyxy[:, 2] = xywh[:, 0] + xywh[:, 2] / 2; xyxy[:, 3] = xywh[:, 1] + xywh[:, 3] / 2
            gb.append(xyxy.numpy()); gc.append(t[:, 1].long().numpy())
    print(f"evaluator: {n_multi} rows share an anchor with a higher-scored row")
    assert got == MR.compute_map(pb, ps, pc, gb, gc, nc)
