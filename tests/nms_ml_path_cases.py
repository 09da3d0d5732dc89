"""Seeded multi-label NMS inputs and a CPU model of the way K7's select kernel gets their sorted candidates -- the
multi-label counterpart of tests/nms_path_cases.py, whose constants, Path record and input builders it reuses.

Multi-label keys are (~ordered(score) << 32) | (a * nc + c) for every (anchor a, class c) above the threshold.  The
multi-label filter compacts them with one atomicAdd per warp of 32 anchors and writes each warp's keys in (anchor, class)
order, so the sampled set of top_keys (every stride-th slot, stride = ceil(n / 4096)) depends on the order the warps arrive
in -- except when every pair is a candidate, A is a multiple of 32 and stride divides 32 * nc.  Then every warp's range
starts at a multiple of 32 * nc, a slot's offset inside it is the key's index a * nc + c modulo 32 * nc, and the sampled
keys are exactly those with (a * nc + c) % stride == 0, whatever the warp order.  ``select_path`` reports any other image
above SMEM_KEYS candidates as "indeterminate".  The redo decision uses the C oracle's keep list, as nms_path_cases does.

Every case is (pred [B, A, 4 + nc] fp32, nms keyword arguments, scale rows or None, expected path of every image)."""
from __future__ import annotations

import functools

import numpy as np
import torch

from tests import nms_ml_oracle as O
from tests import nms_path_cases as P
from tests.cases import at_threshold_pred


def select_path(pred, conf_thres=0.25, iou_thres=0.45, max_det=300, classes=None, agnostic=False, consts=None) -> P.Path:
    """The way nms_select_kernel<true> gets its sorted candidates for one image pred [A, 4 + nc]."""
    k = P.kernel_constants() if consts is None else consts
    SMEM, TOP, CHUNK = k["SMEM_KEYS"], k["TOP_TARGET"], k["CHUNK"]
    pred = np.ascontiguousarray(pred, np.float32)
    A, nc = pred.shape[0], pred.shape[1] - 4
    a, c, conf = O._candidates(pred, conf_thres, classes)
    idx = a.astype(np.int64) * nc + c
    n = len(idx)
    keys = P._keys(conf, idx)
    rank = np.empty(n, np.int64)
    rank[np.argsort(keys)] = np.arange(n)
    det, keep = O.nms_image_c(pred, conf_thres, iou_thres, max_det, classes, agnostic, multi_label=True)
    ranks = rank[np.searchsorted(idx, keep * nc + det[:, 5].astype(np.int64))]   # idx is ascending (row-major)

    if n == 0:
        prune = False
    else:
        xywh = pred[a, :4]
        hw, hh = xywh[:, 2] * np.float32(0.5), xywh[:, 3] * np.float32(0.5)
        mc = max((xywh[:, 0] - hw).max(), (xywh[:, 1] - hh).max(), (xywh[:, 0] + hw).max(), (xywh[:, 1] + hh).max())
        scale = np.float32(mc) + np.float32(1)
        prune = not agnostic and iou_thres >= 0 and np.float32(nc) * scale < np.float32(2 ** 22)

    if n <= SMEM:
        path, m = "smem", n
    else:
        stride = -(-n // 4096)
        if not (n == A * nc and A % 32 == 0 and (32 * nc) % stride == 0):
            return P.Path(n, "indeterminate", -1, -1, -1, -1, "no", prune)
        samples = np.sort(keys[idx % stride == 0])
        thr = samples[min(len(samples) - 1, TOP // stride)]
        m = int((keys <= thr).sum())
        if m > SMEM:
            path, m = "overflow", n
        elif m < n and (ranks < m).sum() < max_det:
            path = "redo"
        else:
            path = "sampled"
    kept = len(keep)
    last = int(ranks[-1]) if kept else -1
    if kept == max_det:
        chunks = last // CHUNK + 1
        full_at = "last" if last % CHUNK == CHUNK - 1 or last == n - 1 else "inside"
    else:
        chunks, full_at = -(-n // CHUNK), "no"
    return P.Path(n, path, m, kept, last, chunks, full_at, bool(prune))


# ---- inputs ---------------------------------------------------------------------------------------------------------
def dense_image(A, nc, seed, S=640.0, lo=0.002):
    """every pair a candidate at conf 0.001: scattered boxes, every class score in (lo, 0.99)"""
    rng = np.random.default_rng(seed)
    p = np.zeros((A, 4 + nc), np.float32)
    p[:, 0:2] = rng.uniform(0, S, (A, 2))
    p[:, 2:4] = rng.uniform(4.0, 40.0, (A, 2))
    p[:, 4:] = rng.uniform(lo, 0.99, (A, nc))
    return p


def overflow_image(A, nc, seed, stride):
    """every pair a candidate; the sampled pairs ((a * nc + c) % stride == 0) hold the lowest scores, so the sampled
    threshold lets almost every key through: more than SMEM_KEYS"""
    p = dense_image(A, nc, seed)
    idx = np.arange(A * nc).reshape(A, nc)
    rng = np.random.default_rng(seed + 1)
    p[:, 4:] = np.where(idx % stride == 0, rng.uniform(0.002, 0.1, (A, nc)), rng.uniform(0.2, 0.99, (A, nc)))
    return p


def redo_image(A, nc, seed, top=3200, clusters=12):
    """every pair a candidate; every class of `top` / nc anchors scores high and their boxes form `clusters` identical-box
    clusters (one keep per class each), the rest are scattered with low scores: the best ~TOP_TARGET keys give < 300 keeps"""
    rng = np.random.default_rng(seed)
    p = dense_image(A, nc, seed, S=2000.0, lo=0.002)
    p[:, 4:] = rng.uniform(0.002, 0.4, (A, nc))
    t = rng.permutation(A)[: top // nc]
    cid = np.arange(len(t)) % clusters
    p[t, 0] = 2200.0 + 80.0 * (cid % 4)
    p[t, 1] = 100.0 + 80.0 * (cid // 4)
    p[t, 2:4] = 50.0
    p[t, 4:] = rng.uniform(0.5, 0.99, (len(t), nc))
    return p


def sparse_image(A, nc, seed, per_anchor=3, n_anchors=1000):
    """`n_anchors` anchors with `per_anchor` classes above 0.001 each (several classes of one anchor), the rest below"""
    rng = np.random.default_rng(seed)
    p = dense_image(A, nc, seed)
    p[:, 4:] = rng.uniform(0, 9e-4, (A, nc))
    for a in rng.permutation(A)[:n_anchors]:
        p[a, 4 + rng.permutation(nc)[:per_anchor]] = rng.uniform(0.01, 0.9, per_anchor)
    return p


def ties_image(A, nc, seed):
    """scores on a 1/16 grid: equal scores across classes of one anchor and across anchors; overlapping boxes"""
    rng = np.random.default_rng(seed)
    p = dense_image(A, nc, seed, S=160.0)
    p[:, 2:4] = rng.uniform(20.0, 60.0, (A, 2))
    s = np.round(rng.uniform(0, 1, (A, nc)) * 16) / 16
    p[:, 4:] = np.where(s > 0.5, s, 0.0).astype(np.float32)
    return p


def at_threshold_multi(nc=4):
    """tests/cases.py's pairs whose fp32 IoU equals float32(thr), each row's score also given to a second class"""
    p = at_threshold_pred(nc)[0].numpy().copy()
    for r in range(len(p)):
        c = int(p[r, 4:].argmax())
        p[r, 4 + (c + 1) % nc] = p[r, 4 + c]          # equal scores across two classes of one anchor
    return p


def leaky_image(A, nc, seed):
    """boxes around the origin (x1, y1 < -0.5: the class offset lets them reach into the previous class's block) with three
    classes each above threshold"""
    rng = np.random.default_rng(seed)
    p = np.zeros((A, 4 + nc), np.float32)
    p[:, 0:2] = rng.uniform(-30, 30, (A, 2))
    p[:, 2:4] = rng.uniform(4.0, 60.0, (A, 2))
    p[:, 4:] = rng.uniform(0, 0.2, (A, nc))
    for a in range(A):
        p[a, 4 + rng.permutation(nc)[:3]] = rng.uniform(0.3, 0.9, 3)
    return p


def grid_multi(A, nc, seed, per_anchor=4):
    """disjoint boxes on a grid, `per_anchor` classes each: every candidate is kept, so max_det binds"""
    rng = np.random.default_rng(seed)
    p = P.grid_image(A, nc, seed)
    for a in range(A):
        p[a, 4 + rng.permutation(nc)[:per_anchor]] = rng.uniform(0.02, 0.99, per_anchor)
    return p


def _stack(*imgs):
    return torch.from_numpy(np.stack(imgs)).contiguous()


def _c(build, expect, scale=False, **kw):
    return P.Case(build, dict(conf_thres=kw.pop("conf_thres", 0.001), **kw), tuple(expect), scale)


CASES: dict[str, P.Case] = {
    # ---- the four ways to the sorted list (stride 4 with nc = 8, stride 20 with nc = 80)
    "ml_overflow": _c(lambda: _stack(overflow_image(2048, 8, 1, 4)), ["overflow"], iou_thres=0.6),
    "ml_overflow_nc80": _c(lambda: _stack(overflow_image(1024, 80, 2, 20)), ["overflow"], scale=True, iou_thres=0.7),
    "ml_overflow_agnostic": _c(lambda: _stack(overflow_image(2048, 8, 3, 4)), ["overflow"], iou_thres=0.45, agnostic=True),
    "ml_redo": _c(lambda: _stack(redo_image(2048, 8, 11)), ["redo"], iou_thres=0.6),
    "ml_redo_nc80": _c(lambda: _stack(redo_image(1024, 80, 12, clusters=3)), ["redo"], scale=True, iou_thres=0.7),
    "ml_redo_classes": _c(lambda: _stack(redo_image(2048, 8, 13)), ["redo"], iou_thres=0.6, classes=list(range(8)) + [3, 50]),
    "ml_sampled": _c(lambda: _stack(dense_image(2048, 8, 21)), ["sampled"], iou_thres=0.6),
    "ml_sampled_nc80": _c(lambda: _stack(dense_image(1024, 80, 22)), ["sampled"], iou_thres=0.7),
    "ml_mixed4": _c(lambda: _stack(sparse_image(2048, 8, 31), dense_image(2048, 8, 32), overflow_image(2048, 8, 33, 4),
                                   redo_image(2048, 8, 34)), ["smem", "sampled", "overflow", "redo"], scale=True, iou_thres=0.6),
    # ---- semantics
    "ml_several_classes": _c(lambda: _stack(sparse_image(3000, 80, 41), sparse_image(3000, 80, 42, per_anchor=6, n_anchors=600)),
                             ["smem", "smem"], iou_thres=0.45),
    "ml_ties": _c(lambda: _stack(ties_image(600, 12, 43)), ["smem"], iou_thres=0.5, conf_thres=0.25),
    "ml_at_threshold_0.6": _c(lambda: _stack(at_threshold_multi()), ["smem"], iou_thres=0.6, conf_thres=0.25),
    "ml_at_threshold_0.45": _c(lambda: _stack(at_threshold_multi()), ["smem"], iou_thres=0.45, conf_thres=0.25),
    "ml_classes": _c(lambda: _stack(sparse_image(3000, 80, 44)), ["smem"], iou_thres=0.45, classes=[79, 3, 3, 0, 80, 500]),
    "ml_agnostic": _c(lambda: _stack(sparse_image(3000, 80, 45)), ["smem"], iou_thres=0.45, agnostic=True),
    "ml_leaky": _c(lambda: _stack(leaky_image(500, 6, 46)), ["smem"], iou_thres=0.3, conf_thres=0.25),
    **{f"ml_nc{nc}": _c(lambda nc=nc: _stack(sparse_image(2000, nc, 50 + nc, per_anchor=min(nc, 3))), ["smem"],
                        iou_thres=0.45) for nc in (1, 5, 81)},
    "ml_nc5_overflow": _c(lambda: _stack(overflow_image(4096, 5, 56, 5)), ["overflow"], iou_thres=0.45),
    "ml_empty": _c(lambda: _stack(sparse_image(800, 8, 57, n_anchors=0), sparse_image(800, 8, 58)), ["smem", "smem"],
                   iou_thres=0.45),
    **{f"ml_maxdet{md}": _c(lambda: _stack(grid_multi(1500, 20, 59)), ["smem"], iou_thres=0.5, max_det=md)
       for md in (300, 1000, 4096)},
}

SORT_GLOBAL = P.SORT_GLOBAL


@functools.lru_cache(maxsize=None)
def pred_of(name: str) -> torch.Tensor:
    return CASES[name].build()


def scale_of(name: str) -> torch.Tensor | None:
    c = CASES[name]
    return torch.from_numpy(P._scale_rows(pred_of(name).shape[0], 7)) if c.scale else None


@functools.lru_cache(maxsize=None)
def paths_of(name: str) -> tuple[P.Path, ...]:
    c = CASES[name]
    p = pred_of(name).numpy()
    return tuple(select_path(p[b], **c.kw) for b in range(p.shape[0]))
