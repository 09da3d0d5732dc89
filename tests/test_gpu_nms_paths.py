"""K7 (k_nms.cu) bit for bit against the C oracle on every way nms_select_kernel gets its sorted candidates: the
shared-memory sort, the sampled top-m, sort_global after an overflow and sort_global after a redo (tests/nms_path_cases.py;
tests/test_cpu_nms_paths.py checks on the CPU which way each case takes).  counts, all six columns of every kept row and
keep_anchor are compared as bits; fused scale rows must equal scale_boxes applied to the unfused rows."""
import ctypes as C
import functools

import numpy as np
import pytest
import torch

from oracle import nms_ref as N
from oracle import preproc_ref as PR
from tests import nms_path_cases as P

pytestmark = pytest.mark.gpu

import yolo_b200
from yolo_b200 import _lib as L

DEV = "cuda"


@functools.lru_cache(maxsize=None)
def oracle(name):
    return N.non_max_suppression(P.pred_of(name), impl="c", return_keep=True, **P.CASES[name].kw)


def assert_matches_oracle(name, out, counts, keep):
    dets, keeps = oracle(name)
    out, counts, keep = out.cpu().numpy(), counts.cpu().numpy(), keep.cpu().numpy()
    assert counts.tolist() == [len(d) for d in dets], (name, counts.tolist(), [len(d) for d in dets])
    for b, (d, k) in enumerate(zip(dets, keeps)):
        n = len(d)
        bad = np.nonzero((out[b, :n].view(np.uint32) != d.view(np.uint32)).any(1))[0]
        assert len(bad) == 0, f"{name} image {b}: {len(bad)} of {n} rows differ, first at row {bad[0]}"
        assert np.array_equal(keep[b, :n], k), (name, b)


@pytest.mark.parametrize("name", list(P.CASES))
def test_nms_path_bit_exact(name):
    c = P.CASES[name]
    pred = P.pred_of(name).to(DEV)
    out, counts, keep = yolo_b200.nms_raw(pred, **c.kw)
    assert_matches_oracle(name, out, counts, keep)
    sc = P.scale_of(name)
    if sc is None:
        return
    sd = sc.to(DEV)
    fo, fc, fk = yolo_b200.nms_raw(pred, **c.kw, scale=sd)
    assert torch.equal(fc, counts) and torch.equal(fk, keep)
    dets, _ = oracle(name)
    for b, d in enumerate(dets):
        n = len(d)
        pw, ph, gain, ow, oh = sc[b].tolist()
        ref = out[b, :n].clone()
        yolo_b200.scale_boxes(ref[:, :4], None, (oh, ow), ((gain, gain), (pw, ph)))
        got = fo[b, :n].cpu().numpy()
        assert np.array_equal(got.view(np.uint32), ref.cpu().numpy().view(np.uint32)), (name, b)
        cpu = PR.scale_boxes(d[:, :4], None, (oh, ow), ((gain, gain), (pw, ph)))
        assert np.array_equal(got[:, :4].view(np.uint32), cpu.view(np.uint32)), (name, b)


@pytest.mark.parametrize("name", [n for n in P.CASES if any(p.path in P.SORT_GLOBAL for p in P.paths_of(n))])
def test_nms_sort_global_ignores_stale_workspace(name):
    """sort_global pads each image's keys to a power of two with ~0: whatever the workspace held before must not reach the
    scan.  A zeroed workspace holds keys that sort first (anchor 0, NaN score)."""
    c = P.CASES[name]
    lib = L.lib()
    pred = P.pred_of(name).to(DEV)
    Bn, A, ch = pred.shape
    md = c.kw.get("max_det", 300)
    ws = torch.zeros((lib.yre_nms_workspace_bytes(Bn, A),), dtype=torch.uint8, device=DEV)
    out = torch.empty((Bn, md, 6), dtype=torch.float32, device=DEV)
    counts = torch.empty((Bn,), dtype=torch.int32, device=DEV)
    keep = torch.empty((Bn, md), dtype=torch.int64, device=DEV)
    cls = c.kw.get("classes")
    cls_t = torch.tensor(cls, dtype=torch.int32, device=DEV) if cls is not None else None
    d = L.NmsDesc(pred.data_ptr(), Bn, A, ch - 4, c.kw["conf_thres"], c.kw["iou_thres"], md,
                  cls_t.data_ptr() if cls_t is not None else None, len(cls) if cls is not None else -1,
                  int(bool(c.kw.get("agnostic"))), out.data_ptr(), counts.data_ptr(), keep.data_ptr(), ws.data_ptr(),
                  ws.numel(), None)
    L.check(lib.yre_nms_batched(C.byref(d), torch.cuda.current_stream().cuda_stream), "nms")
    assert_matches_oracle(name, out, counts, keep)


def test_nms_max_det_range_launches():
    """every max_det check_nms accepts launches (the select kernel's shared memory grows with max_det)"""
    pred = P.pred_of("grid_maxdet4096").to(DEV)
    for md in (3149, 3150, 4095, 4096):
        out, counts, _ = yolo_b200.nms_raw(pred, 0.001, 0.5, max_det=md)
        assert counts.tolist() == [md]
    with pytest.raises(L.YreError):
        yolo_b200.nms_raw(pred, 0.001, 0.5, max_det=4097)
