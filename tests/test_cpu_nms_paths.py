"""CPU check that tests/nms_path_cases.py drives K7's select kernel down every way to its sorted candidates (shared-memory
sort, sampled top-m, overflow -> sort_global, redo -> sort_global), with the edges each must get right.  The model reads
SMEM_KEYS, TOP_TARGET and CHUNK from k_nms.cu, so it cannot drift from the kernel.  Needs the C oracle, no GPU."""
import numpy as np
import pytest

from tests import nms_path_cases as P

PATHS = ("smem", "sampled", "overflow", "redo")


@pytest.mark.parametrize("name", list(P.CASES))
def test_model_matches_case_name(name):
    """The model's path of every image is the case's, and no image above SMEM_KEYS candidates is indeterminate."""
    got = tuple(p.path for p in P.paths_of(name))
    assert got == P.CASES[name].expect, (name, P.paths_of(name))


def test_every_path_is_covered():
    found = {p.path for name in P.CASES for p in P.paths_of(name)}
    assert set(PATHS) <= found, f"no determinate case takes {set(PATHS) - found}"


def test_sort_global_features_are_covered():
    """prune on and off, agnostic, a class filter, fused scale rows and B > 1 each reach sort_global, on both of its ways"""
    feats = {path: set() for path in P.SORT_GLOBAL}
    for name, c in P.CASES.items():
        ps = P.paths_of(name)
        for p in ps:
            if p.path not in P.SORT_GLOBAL:
                continue
            f = feats[p.path]
            f.add("prune" if p.prune else "no_prune")
            f |= {k for k in ("agnostic", "classes") if c.kw.get(k)}
            f |= {"scale"} if c.scale else set()
            f |= {"batch"} if len(ps) > 1 else set()
            f |= {"npow2"} if p.n & (p.n - 1) else set()
    want = {"prune", "no_prune", "agnostic", "classes", "scale", "batch", "npow2"}
    for path, f in feats.items():
        assert want <= f, f"{path}: no case with {want - f}"


def test_mixed_batch_takes_every_path():
    assert any(set(PATHS) <= {p.path for p in P.paths_of(n)} for n in P.CASES)


def test_max_det_and_chunk_edges():
    """max_det 1, 511, 512, 513, 3149 and 4096 (the largest accepted); keeps crossing chunk boundaries; max_det reached on
    the last candidate of a chunk"""
    mds = {c.kw.get("max_det", 300) for c in P.CASES.values()}
    assert {1, 511, 512, 513, 3149, 4096} <= mds
    ps = {n: P.paths_of(n)[0] for n in P.CASES}
    assert ps["grid_maxdet512"].full_at == "last" and ps["grid_maxdet512"].chunks == 1
    assert ps["grid_maxdet1024"].full_at == "last" and ps["grid_maxdet1024"].chunks == 2
    assert ps["grid_maxdet4096"].full_at == "last" and ps["grid_maxdet4096"].kept == 4096
    assert ps["grid_maxdet513"].full_at == "inside" and ps["grid_maxdet513"].chunks == 2
    assert ps["grid_dup_maxdet4096"].kept == 4096 and ps["grid_dup_maxdet4096"].chunks > 8
    assert any(p.kept >= 3149 and p.path in P.SORT_GLOBAL for p in ps.values())


@pytest.mark.parametrize("thr", [0.45, 0.5, 0.6, 0.7])
def test_iou_band(thr):
    """nested pairs at thr (1 +- 2^-k) for k = 16..20 and closer than 2^-21 on either side (k = 21..24 meet the fp32
    resolution of the ratio), both sides of thr inside the division-free shortcut's 2^-18 margin, and random pairs within
    2^-17"""
    off = P.band_offsets(P.pred_of(f"band_{thr}")[0].numpy(), thr)
    nested, rnd = off[:72], off[72:]
    for sgn in (-1, 1):
        for k in range(16, 21):
            assert np.any(np.abs(sgn * nested - 2.0 ** -k) <= 2.0 ** -k / 4), (thr, sgn, k)
        assert np.any((sgn * nested >= 0) & (np.abs(nested) <= 2.0 ** -21)), (thr, sgn)
    assert len(rnd) >= 64 and np.all(np.abs(rnd) < 2.0 ** -17)
    assert np.any((rnd > 0) & (rnd < 2.0 ** -18)) and np.any((rnd < 0) & (rnd > -2.0 ** -18))


def test_cross_class_limits():
    """nc * scale just below 2^22 has the shortcut on, just above off; leaky pairs (x1, y1 < -1) are suppressed by the
    reference, the pairs at the proof's edge (-0.5 and its neighbours) are not"""
    for name in ("cross_class_below", "cross_class_below_0.001"):
        assert all(p.prune for p in P.paths_of(name))
    for name in ("cross_class_above", "cross_class_above_0.001"):
        assert not any(p.prune for p in P.paths_of(name))
    ps = P.paths_of("cross_class_below")
    assert [p.kept for p in ps[:5]] == [158] * 5 and [p.kept for p in ps[5:]] == [79, 79]


def test_negative_threshold_turns_prune_off():
    assert not any(p.prune for p in P.paths_of("neg_thr_-0.1"))
    assert all(p.prune for p in P.paths_of("neg_thr_-0.0"))
    assert [p.kept for p in P.paths_of("neg_thr_-0.1")] == [1, 1]


def test_scalar_class_paths():
    """class counts that are not multiples of 4 (scalar filter and load) and a class list with duplicates, absent
    classes and classes >= nc"""
    ncs = {P.pred_of(n).shape[2] - 4 for n in P.CASES}
    assert {1, 5, 81} <= ncs
    cl = P.CASES["classes_odd"].kw["classes"]
    assert len(set(cl)) < len(cl) and max(cl) >= P.pred_of("classes_odd").shape[2] - 4


def test_model_reads_the_kernel_constants():
    """The constants come from k_nms.cu, and the expectations move with them: a larger TOP_TARGET takes the redo case's
    scan into the scattered candidates (enough keeps: no redo), a smaller one leaves the overflow case overflowing, and
    SMEM_KEYS = 16384 sorts the 16384-candidate overflow case in shared memory."""
    src = P.KNMS.read_text()
    k = P.kernel_constants(src)
    assert k == P.kernel_constants()
    redo, over = P.pred_of("redo")[0].numpy(), P.pred_of("overflow")[0].numpy()
    kw_r, kw_o = P.CASES["redo"].kw, P.CASES["overflow"].kw
    assert P.select_path(redo, **kw_r, consts=k).path == "redo"
    big = P.kernel_constants(src.replace(f"TOP_TARGET = {k['TOP_TARGET']};", "TOP_TARGET = 6144;"))
    assert big["TOP_TARGET"] == 6144
    assert P.select_path(redo, **kw_r, consts=big).path == "sampled"
    small = P.kernel_constants(src.replace(f"TOP_TARGET = {k['TOP_TARGET']};", "TOP_TARGET = 512;"))
    assert P.select_path(over, **kw_o, consts=small).path == "overflow"
    sm = P.kernel_constants(src.replace(f"SMEM_KEYS = {k['SMEM_KEYS']};", "SMEM_KEYS = 16384;"))
    assert P.select_path(over, **kw_o, consts=sm).path == "smem"
    ch = P.kernel_constants(src.replace(f"CHUNK = {k['CHUNK']};", "CHUNK = 256;"))
    assert P.select_path(P.pred_of("grid_maxdet512")[0].numpy(), **P.CASES["grid_maxdet512"].kw, consts=ch).chunks == 2


def test_indeterminate_samples_are_reported():
    """above SMEM_KEYS candidates, a sample that depends on warp order is not counted toward coverage"""
    p = P.overflow_image(16384, 80, 1)
    assert P.select_path(p[:16005], conf_thres=0.001).path == "indeterminate"        # A not a multiple of 32
    assert P.select_path(p[:10240], conf_thres=0.001).path == "indeterminate"        # stride 3
    q = p.copy()
    q[5, 4:] = 0.0                                                                    # one anchor not a candidate
    assert P.select_path(q, conf_thres=0.001).path == "indeterminate"
