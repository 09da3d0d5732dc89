"""Seeded NMS inputs that drive K7's select kernel (k_nms.cu) down each of its ways to the sorted candidate list, and a
CPU model of which way each image takes.

``nms_select_kernel`` gets its sorted candidates in one of four ways:

  smem      n <= SMEM_KEYS: all n keys sorted in shared memory;
  sampled   n > SMEM_KEYS: a threshold read from a sorted sample of <= 4096 keys picks the best m ~ TOP_TARGET keys, and
            the scan reaches max_det keeps inside them (or there is nothing beyond them);
  overflow  more than SMEM_KEYS keys pass the sampled threshold (top_keys returns -1): sort_global sorts all n;
  redo      the best m keys give fewer than max_det keeps and there are more candidates: sort_global sorts all n and the
            scan starts again.

``select_path`` restates top_keys and the redo decision.  Above SMEM_KEYS candidates the sample is read at a stride from
the key list that nms_filter compacts with one atomicAdd per warp, so in general it depends on the order the warps
arrive in.  It does not when every anchor is a candidate, A is a multiple of 32 and stride = ceil(n / 4096) is a power of
two <= 32: then every warp adds 32 keys at a 32-aligned slot in lane order, and the sampled keys are those of the anchors
with a % stride == 0.  Any other image with n > SMEM_KEYS is reported "indeterminate".

The redo decision takes the oracle's keep list (oracle/nms_ref.c).  Greedy NMS is prefix-consistent: the keeps of the best
m candidates are the full list's keeps of rank < m.

Every case is (pred [B, A, 4 + nc] fp32, nms keyword arguments, scale rows or None, expected path of every image)."""
from __future__ import annotations

import functools
import re
from dataclasses import dataclass

import numpy as np
import torch

from tests.conftest import ROOT

KNMS = ROOT / "yolo-re_b200/csrc/k_nms.cu"


def kernel_constants(src: str | None = None) -> dict[str, int]:
    """SMEM_KEYS, TOP_TARGET and CHUNK as k_nms.cu defines them."""
    src = KNMS.read_text() if src is None else src
    out = {}
    for name in ("SMEM_KEYS", "TOP_TARGET", "CHUNK"):
        m = re.search(rf"constexpr int {name} = (\d+);", src)
        assert m, f"{name} not found in k_nms.cu"
        out[name] = int(m.group(1))
    return out


@dataclass
class Path:
    n: int                 # candidates
    path: str              # smem / sampled / overflow / redo / indeterminate
    m: int                 # keys of the first scan (n for smem and overflow)
    kept: int              # boxes kept
    last_rank: int         # rank of the last keep in the sorted candidates (-1: none)
    chunks: int            # CHUNK-candidate chunks of the final scan
    full_at: str           # max_det reached "inside" a chunk, at a chunk's "last" candidate, or "no"
    prune: bool            # the cross-class shortcut is on


def _keys(conf: np.ndarray, anchors: np.ndarray) -> np.ndarray:
    """nms_filter's 64-bit sort keys: (~f2ord(conf)) << 32 | anchor"""
    u = conf.astype(np.float32).view(np.uint32).astype(np.uint64)
    o = np.where(u & 0x80000000, ~u & 0xFFFFFFFF, u | 0x80000000)
    return ((~o & 0xFFFFFFFF) << np.uint64(32)) | anchors.astype(np.uint64)


def _candidates(pred, conf_thres, classes):
    sc = pred[:, 4:]
    cls = sc.argmax(1)
    conf = sc[np.arange(len(pred)), cls]
    mask = conf > np.float32(conf_thres)
    if classes is not None:
        mask &= np.isin(cls, np.asarray(classes))
    a = np.nonzero(mask)[0]
    return a, conf[a], cls[a]


def select_path(pred, conf_thres=0.25, iou_thres=0.45, max_det=300, classes=None, agnostic=False, consts=None) -> Path:
    """The way nms_select_kernel gets its sorted candidates for one image pred [A, 4 + nc]."""
    from oracle import nms_ref as N
    k = kernel_constants() if consts is None else consts
    SMEM, TOP, CHUNK = k["SMEM_KEYS"], k["TOP_TARGET"], k["CHUNK"]
    pred = np.ascontiguousarray(pred, np.float32)
    A, nc = pred.shape[0], pred.shape[1] - 4
    anc, conf, _ = _candidates(pred, conf_thres, classes)
    n = len(anc)
    keys = _keys(conf, anc)
    order = np.argsort(keys)
    rank = np.empty(A, np.int64)
    rank[anc[order]] = np.arange(n)
    _, keep = N.nms_image_c(pred, conf_thres, iou_thres, max_det, classes, agnostic)
    ranks = rank[keep]

    if n == 0:
        prune = False
    else:
        xywh = pred[anc, :4]
        hw, hh = xywh[:, 2] * np.float32(0.5), xywh[:, 3] * np.float32(0.5)
        mc = max((xywh[:, 0] - hw).max(), (xywh[:, 1] - hh).max(), (xywh[:, 0] + hw).max(), (xywh[:, 1] + hh).max())
        scale = np.float32(mc) + np.float32(1)
        prune = not agnostic and iou_thres >= 0 and np.float32(nc) * scale < np.float32(2 ** 22)

    if n <= SMEM:
        path, m = "smem", n
    else:
        stride = -(-n // 4096)
        if not (n == A and A % 32 == 0 and stride & (stride - 1) == 0 and stride <= 32):
            return Path(n, "indeterminate", -1, -1, -1, -1, "no", prune)
        samples = np.sort(keys[anc % stride == 0])
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
    return Path(n, path, m, kept, last, chunks, full_at, bool(prune))


# ---- inputs ---------------------------------------------------------------------------------------------------------
def _spread(rng, A, nc, S=640.0, wh=(4.0, 40.0)):
    """A boxes scattered over an S x S image with one dominant class each, scores in (0.01, 0.4)"""
    p = np.zeros((A, 4 + nc), np.float32)
    p[:, 0:2] = rng.uniform(0, S, (A, 2))
    p[:, 2:4] = rng.uniform(*wh, (A, 2))
    p[:, 4:] = rng.uniform(0, 9e-4, (A, nc))
    p[np.arange(A), 4 + rng.integers(0, nc, A)] = rng.uniform(0.01, 0.4, A)
    return p


def _set_score(p, a, s):
    p[a, 4:] = np.minimum(p[a, 4:], np.float32(9e-4))
    cls = p[a, 4:].argmax(1) if np.ndim(a) else p[a, 4:].argmax()
    p[a, 4 + cls] = s


def overflow_image(A, nc, seed):
    """Every anchor a candidate; the sampled anchors (a % 4 == 0) hold the lowest scores, so the sampled threshold lets
    ~A * 3/4 keys through: more than SMEM_KEYS"""
    rng = np.random.default_rng(seed)
    p = _spread(rng, A, nc)
    a = np.arange(A)
    s = np.where(a % 4 == 0, rng.uniform(0.01, 0.1, A), rng.uniform(0.2, 0.99, A))
    _set_score(p, a, s.astype(np.float32))
    return p


def redo_image(A, nc, seed, top=3000, clusters=100):
    """Every anchor a candidate; the best `top` candidates form `clusters` identical-box clusters (one keep each), the rest
    are scattered: the best ~TOP_TARGET candidates yield far fewer than 300 keeps"""
    rng = np.random.default_rng(seed)
    p = _spread(rng, A, nc, S=2000.0)
    t = rng.permutation(A)[:top]
    cid = np.arange(top) % clusters
    gx, gy = cid % 10, cid // 10
    p[t, 0] = 2200.0 + 80.0 * gx
    p[t, 1] = 100.0 + 80.0 * gy
    p[t, 2:4] = 50.0
    cls = rng.integers(0, nc, clusters)[cid]
    p[t, 4:] = rng.uniform(0, 9e-4, (top, nc))
    p[t, 4 + cls] = rng.uniform(0.5, 0.99, top)
    return p


def sampled_image(A, nc, seed):
    rng = np.random.default_rng(seed)
    return _spread(rng, A, nc)


def sparse_image(A, nc, seed, n=3000):
    """at most n candidates (conf > 0.001): the shared-memory sort"""
    rng = np.random.default_rng(seed)
    p = _spread(rng, A, nc)
    drop = rng.permutation(A)[: A - n]
    p[drop, 4:] = rng.uniform(0, 9e-4, (len(drop), nc))
    return p


def grid_image(A, nc, seed, dup_every=0):
    """A disjoint boxes on a grid (every candidate kept), scores descending with the anchor; with dup_every = d, every d-th
    box repeats its predecessor's box with a lower score (suppressed), so the keeps cross chunk boundaries off-grid"""
    rng = np.random.default_rng(seed)
    p = np.zeros((A, 4 + nc), np.float32)
    side = int(np.ceil(np.sqrt(A)))
    a = np.arange(A)
    p[:, 0] = 10.0 * (a % side) + 5.0
    p[:, 1] = 10.0 * (a // side) + 5.0
    p[:, 2:4] = 8.0
    p[:, 4:] = rng.uniform(0, 9e-4, (A, nc))
    p[a, 4 + rng.integers(0, nc, A)] = np.linspace(0.99, 0.02, A, dtype=np.float32)
    if dup_every:
        d = a[(a % dup_every == dup_every - 1)]
        p[d, 0:4] = p[d - 1, 0:4]
        p[d, 4:] = p[d - 1, 4:] * np.float32(0.999)
    return p


def _iou_xywh(r1, r2):
    """IoU of two xywh rows with the reference's fp32 arithmetic (xywh -> xyxy, then inter / ((a1 + a2) - inter))"""
    bx = []
    for r in (r1, r2):
        hw, hh = r[2] / np.float32(2), r[3] / np.float32(2)
        bx.append((r[0] - hw, r[1] - hh, r[0] + hw, r[1] + hh))
    (a1, b1, c1, d1), (a2, b2, c2, d2) = bx
    w = max(np.float32(0), min(c1, c2) - max(a1, a2))
    h = max(np.float32(0), min(d1, d2) - max(b1, b2))
    inter = w * h
    with np.errstate(invalid="ignore", divide="ignore"):
        return inter / (((c1 - a1) * (d1 - b1) + (c2 - a2) * (d2 - b2)) - inter)


def band_image(thr, seed, n_random=64):
    """Pairs whose fp32 IoU lies at thr (1 +- 2^-k), k = 16..24, from nested boxes with power-of-two extents, and random
    pairs whose second width is tuned ulp by ulp to within 2^-17 of thr.  Each pair sits in its own 128-pixel row, one
    class (offset 0); either box of a pair may score higher."""
    rng = np.random.default_rng(seed)
    pairs = []
    for k in range(16, 25):
        for sgn in (-1, 1):
            t = thr * (1 + sgn * 2.0 ** -k)
            for W in (64.0, 32.0):
                w = np.float32(W * t)
                for hi_first in (True, False):
                    y0 = 128.0 * len(pairs) + W / 2
                    pairs.append(([W / 2, y0, W, W], [w / 2, y0, w, W], hi_first))
    f32 = lambda v: np.asarray(v, np.float32)
    tries = 0
    while len(pairs) < 72 + n_random and tries < 4000:
        tries += 1
        y0 = 128.0 * len(pairs) + 64.0
        wa, ha = rng.uniform(20, 90, 2)
        ra = f32([rng.uniform(0, 40) + wa / 2, y0, wa, ha])
        cxb, cyb, hb = ra[0] + rng.uniform(-10, 10), y0 + rng.uniform(-10, 10), rng.uniform(20, 90)
        rb = lambda wb: f32([cxb, cyb, wb, hb])
        grid = np.linspace(1.0, 2.5 * wa, 400)
        v = np.array([_iou_xywh(ra, rb(g)) for g in grid]) - thr
        cross = np.nonzero(np.sign(v[:-1]) * np.sign(v[1:]) < 0)[0]
        if len(cross) == 0:
            continue
        lo, hi = grid[cross[0]], grid[cross[0] + 1]
        up = v[cross[0] + 1] > 0
        for _ in range(60):
            mid = (lo + hi) / 2
            if (_iou_xywh(ra, rb(mid)) > thr) == up:
                hi = mid
            else:
                lo = mid
        wb = np.float32(lo) + np.float32(rng.integers(-4, 5)) * np.spacing(np.float32(lo))
        if abs(float(_iou_xywh(ra, rb(wb))) / thr - 1) < 2.0 ** -17:
            pairs.append((ra, rb(wb), bool(rng.integers(0, 2))))
    nc = 2
    p = np.zeros((2 * len(pairs), 4 + nc), np.float32)
    for q, (r1, r2, hi_first) in enumerate(pairs):
        s = 0.9 - 1e-4 * q
        p[2 * q, :4], p[2 * q + 1, :4] = r1, r2
        p[2 * q, 4], p[2 * q + 1, 4] = (s, s - 0.05) if hi_first else (s - 0.05, s)
    p[:, 5] = 1e-4
    return p


def band_offsets(pred, thr):
    """IoU / thr - 1 of every consecutive pair of rows of band_image"""
    return np.asarray([float(_iou_xywh(pred[i], pred[i + 1])) / thr - 1 for i in range(0, len(pred) - 1, 2)])


def cross_class_image(maxc, variant, nc=80):
    """For every adjacent class pair (c, c+1), c < nc - 1: a 2 x 2 box of class c in the corner (maxc - 2, maxc) and a
    1 x 1 box of class c+1 whose x1 and y1 are `variant`.  Under the class offsets the corner box ends at (c+1) * scale - 1
    and the other starts near (c+1) * scale + variant: at -0.5 and its neighbours the cross-class shortcut's proof is
    tight, below -1 the boxes overlap and the reference suppresses one of them.  Scores alternate which box of a pair is
    tested against the other."""
    rows = []
    v = np.float32(variant)
    for c in range(nc - 1):
        lo = [np.float32(maxc - 2.0), np.float32(maxc)]
        for (x1, x2), cls, s in ((lo, c, 0.9 - 0.001 * c), ([v, v + np.float32(1)], c + 1, 0.85 - 0.001 * c)):
            if c % 2:
                s = 1.7 - s
            w = x2 - x1
            r = np.zeros(4 + nc, np.float32)
            r[0] = r[1] = x1 + w / np.float32(2)
            r[2] = r[3] = w
            r[4 + cls] = s
            rows.append(r)
    return np.stack(rows)


def neg_thr_image(A, nc, seed):
    """scattered boxes with a few zero-area ones (0 / 0 IoU: never suppressed)"""
    rng = np.random.default_rng(seed)
    p = _spread(rng, A, nc)
    z = rng.permutation(A)[:20]
    p[z, 2] = 0.0
    return p


def _stack(*imgs):
    return torch.from_numpy(np.stack(imgs)).contiguous()


def _scale_rows(B, seed):
    rng = np.random.default_rng(seed)
    g = rng.uniform(0.3, 1.5, B)
    return np.stack([rng.uniform(0, 40, B), rng.uniform(0, 40, B), g, rng.uniform(400, 1920, B), rng.uniform(300, 1080, B)],
                    1).astype(np.float32)


@dataclass
class Case:
    build: object          # () -> pred [B, A, 4 + nc]
    kw: dict
    expect: tuple          # path of every image
    scale: bool = False


def _c(build, expect, scale=False, **kw):
    return Case(build, dict(conf_thres=kw.pop("conf_thres", 0.001), **kw), tuple(expect), scale)


CASES: dict[str, Case] = {
    # ---- sort_global after an overflow of the sampled threshold
    "overflow": _c(lambda: _stack(overflow_image(16384, 80, 1)), ["overflow"], iou_thres=0.6),
    "overflow_npow2_scale": _c(lambda: _stack(overflow_image(14336, 80, 2)), ["overflow"], scale=True, iou_thres=0.6),
    "overflow_agnostic": _c(lambda: _stack(overflow_image(16384, 8, 3)), ["overflow"], iou_thres=0.45, agnostic=True),
    "overflow_classes": _c(lambda: _stack(overflow_image(16384, 5, 4)), ["overflow"], iou_thres=0.5,
                           classes=[4, 0, 1, 1, 2, 3, 3, 7, 200]),
    "overflow_maxdet4096": _c(lambda: _stack(overflow_image(16384, 80, 5)), ["overflow"], iou_thres=0.6, max_det=4096),
    "overflow_prune_off": _c(lambda: _stack(overflow_image(16384, 80, 6) * np.array([80.0] * 4 + [1.0] * 80, np.float32)),
                             ["overflow"], iou_thres=0.6),
    # ---- sort_global after the best m candidates gave fewer than max_det keeps
    "redo": _c(lambda: _stack(redo_image(16384, 80, 11)), ["redo"], iou_thres=0.6),
    "redo_npow2_scale": _c(lambda: _stack(redo_image(14336, 80, 12)), ["redo"], scale=True, iou_thres=0.6),
    "redo_32768": _c(lambda: _stack(redo_image(32768, 80, 13)), ["redo"], iou_thres=0.6),
    "redo_agnostic": _c(lambda: _stack(redo_image(16384, 4, 14)), ["redo"], iou_thres=0.5, agnostic=True),
    "redo_classes": _c(lambda: _stack(redo_image(16384, 5, 15)), ["redo"], iou_thres=0.5, classes=[0, 1, 2, 3, 4, 4, 9]),
    "redo_maxdet3149": _c(lambda: _stack(redo_image(16384, 80, 16)), ["redo"], iou_thres=0.6, max_det=3149),
    "redo_neg_thr": _c(lambda: _stack(neg_thr_image(16384, 80, 17)), ["redo"], iou_thres=-0.1),
    # ---- several paths in one batch: sort_global pads inside its own image's region only
    "mixed4": _c(lambda: _stack(sparse_image(16384, 80, 21), sampled_image(16384, 80, 22), overflow_image(16384, 80, 23),
                                redo_image(16384, 80, 24)), ["smem", "sampled", "overflow", "redo"], scale=True, iou_thres=0.6),
    "mixed3_npow2": _c(lambda: _stack(redo_image(14336, 80, 25), sparse_image(14336, 80, 26), overflow_image(14336, 80, 27)),
                       ["redo", "smem", "overflow"], iou_thres=0.6),
    "mixed2": _c(lambda: _stack(overflow_image(32768, 80, 28), redo_image(32768, 80, 29)), ["overflow", "redo"],
                 iou_thres=0.6),
    "sampled_32768": _c(lambda: _stack(sampled_image(32768, 80, 30)), ["sampled"], iou_thres=0.6),
    # ---- chunk boundaries and max_det
    **{f"grid_maxdet{md}": _c(lambda: _stack(grid_image(8192, 80, 40)), ["smem"], iou_thres=0.5, max_det=md)
       for md in (1, 511, 512, 513, 1024, 3149, 4096)},
    **{f"grid_dup_maxdet{md}": _c(lambda: _stack(grid_image(8192, 7, 41, dup_every=5)), ["smem"], iou_thres=0.5, max_det=md)
       for md in (1, 511, 512, 513, 3149, 4096)},
    "overflow_maxdet512_thr0": _c(lambda: _stack(overflow_image(16384, 80, 42)), ["overflow"], iou_thres=0.0, max_det=512),
    # ---- IoU shortcut band (the division-free test of iou_gt) and thresholds outside its window
    **{f"band_{t}": _c(lambda t=t: _stack(band_image(t, 50)), ["smem"], iou_thres=t, conf_thres=0.25, max_det=4096)
       for t in (0.45, 0.5, 0.6, 0.7)},
    "band_0.6_agnostic": _c(lambda: _stack(band_image(0.6, 51)), ["smem"], iou_thres=0.6, conf_thres=0.25, max_det=4096,
                            agnostic=True),
    "thr_1e-7": _c(lambda: _stack(sampled_image(4096, 80, 52)), ["smem"], iou_thres=1e-7),
    "thr_2": _c(lambda: _stack(sampled_image(4096, 80, 53)), ["smem"], iou_thres=2.0),
    # ---- the cross-class shortcut at nc * scale just below / above 2^22 (prune on / off), one image per x1 / y1 variant
    **{f"cross_class_{nm}": _c(lambda mc=mc: _stack(*[cross_class_image(mc, v) for v in
                                                      (-0.5, np.nextafter(np.float32(-0.5), np.float32(-1)),
                                                       np.nextafter(np.float32(-0.5), np.float32(0)), -0.25, -1.0,
                                                       -1.25, -1.5)]),
                               ["smem"] * 7, iou_thres=thr, conf_thres=0.25)
       for nm, mc, thr in (("below", 52427.0, 1e-7), ("above", 52428.0, 1e-7), ("below_0.001", 52427.75, 0.001),
                           ("above_0.001", 52428.25, 0.001))},
    # ---- negative thresholds
    **{f"neg_thr_{t}{'_agnostic' if ag else ''}": _c(lambda: _stack(neg_thr_image(3000, 80, 60), neg_thr_image(3000, 80, 61)),
                                                     ["smem", "smem"], iou_thres=t, agnostic=ag)
       for t in (-0.1, -0.0) for ag in (False, True)},
    # ---- class counts that take the scalar filter and load paths, class filters
    **{f"nc{nc}": _c(lambda nc=nc: _stack(sparse_image(6000, nc, 70 + nc), sparse_image(6000, nc, 80 + nc)), ["smem", "smem"],
                     iou_thres=0.45) for nc in (1, 5, 81)},
    "nc5_overflow": _c(lambda: _stack(overflow_image(16384, 5, 90)), ["overflow"], iou_thres=0.45),
    "classes_odd": _c(lambda: _stack(sparse_image(6000, 81, 91)), ["smem"], iou_thres=0.45, classes=[80, 3, 3, 0, 81, 500]),
}

SORT_GLOBAL = ("overflow", "redo")


@functools.lru_cache(maxsize=None)
def pred_of(name: str) -> torch.Tensor:
    return CASES[name].build()


def scale_of(name: str) -> torch.Tensor | None:
    c = CASES[name]
    return torch.from_numpy(_scale_rows(pred_of(name).shape[0], 7)) if c.scale else None


@functools.lru_cache(maxsize=None)
def paths_of(name: str) -> tuple[Path, ...]:
    c = CASES[name]
    p = pred_of(name).numpy()
    return tuple(select_path(p[b], **c.kw) for b in range(p.shape[0]))
