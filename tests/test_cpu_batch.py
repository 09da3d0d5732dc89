"""CPU tests of batch capacity (yre_plan_run_batch): a plan compiled for B images runs any n <= B of them.

The tcgen05 convs keep the tiling chosen for B images and walk only the first ceil(n / tb) image tiles, with a persistent
grid sized for them.  yre_conv_tc_schedule reports that schedule without a device; the walks below restate, in numpy, the
three ways the kernels decode a work item into tiles (include/yre.h, k_conv_tc.cu), and check on every tcgen05 conv of
the full-size benchmark plans, a rectangular plan and the kernel-table cases, for every n in 1..B, that

  * the work items cover every (image tile, y tile, x tile, N tile) of images < n exactly once -- the tiles partition the
    output (tiles_x * tw >= Wo, ...), so every output element of images < n is computed exactly once;
  * an item that reaches no image < n is only ever the odd M tile of a CTA pair or of a halo patch pair;
  * every CTA (pair) of the grid has at least one item, and the grid fits the 148 SMs;

and that at n = B the schedule is the tiling and grid yre_conv_tc_describe reports, i.e. a full run is unchanged."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from tests.conftest import ROOT
from tests.conv_tc_cases import CASES, NUM_SMS, desc as case_desc, describe, tiling
from tests.test_cpu_plan_launch_list import canonical_lines

from yolo_b200 import YOLO, _lib, engine

FULL = {"2": ("gelan-c", 3, 640, 640, 64), "4": ("yolov9-c", 3, 640, 640, 16), "5": ("gelan-c", 3, 1280, 1280, 16),
        "rect": ("gelan-c", 3, 384, 640, 16)}
_KIND = {_lib.TC_GENERIC: "generic", _lib.TC_GENERIC_CTA2: "generic-cta2", _lib.TC_HALO_WS: "halo-ws",
         _lib.TC_HALO_STREAM: "halo-stream"}


@pytest.fixture()
def dry():
    engine._ALLOW_CPU_DRY_RUN = True
    yield
    engine._ALLOW_CPU_DRY_RUN = False


def schedule(d: _lib.ConvDesc, n: int, num_sms: int = NUM_SMS) -> dict:
    s = _lib.TcSchedule()
    code = _lib.lib().yre_conv_tc_schedule(C.byref(d), num_sms, n, C.byref(s))
    assert code == 0, _lib.lib().yre_last_error().decode()
    return {f: getattr(s, f) for f, _ in _lib.TcSchedule._fields_}


def _plan_desc(a: dict) -> _lib.ConvDesc:
    """the descriptor of a conv recorded in Plan.trace, built the way Plan.conv builds it, on the tcgen05 engine"""
    null = engine._null_view()
    return _lib.ConvDesc(a["x"].c(), a["y"].c(), a["res"].c() if a["res"] is not None else null, a["w"].data_ptr(),
                         a["b"].data_ptr(), a["k"], a["stride"], _lib.ACT_SILU if a["silu"] else _lib.ACT_NONE,
                         _lib.ENGINE_TCGEN05, a["xu"].c() if a["xu"] is not None else null)


def _shape_key(d: _lib.ConvDesc) -> tuple:
    """what the schedule depends on (pointers only through res / xu being present)"""
    v = lambda w: (w.dtype, w.layout, w.B, w.H, w.W, w.C_total, w.c_off, w.C) if w.ptr else None
    return (v(d.x), v(d.y), v(d.res), v(d.xu), d.k, d.stride, d.act, d.bias is not None)


def full_plan_descs(config: str) -> list[_lib.ConvDesc]:
    name, cin, H, W, Bn = FULL[config]
    m = YOLO.from_yaml(ROOT / "configs/models" / f"{name}.yaml").eval().set_precision("bf16")
    p = engine.compile_model(m, torch.empty(Bn, cin, H, W))
    uniq = {}
    for k, a in p.trace:
        if k == "conv":
            d = _plan_desc(a)
            uniq.setdefault(_shape_key(d), d)
    return list(uniq.values())


def walk(s: dict, rev: int) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
    """(CTA or CTA pair, M tile, N tile) of every tile the kernel of schedule s computes, in the kernels' own decode"""
    w = np.arange(s["work"])
    if s["kind"] in (_lib.TC_GENERIC, _lib.TC_HALO_WS):
        # TileCur: tile t -> nt = t % tiles_n, m = t / tiles_n (x fastest, image tile outermost); rev reflects every digit
        owner, nt, m = w % s["grid"], w % s["tiles_n"], w // s["tiles_n"]
        if rev:
            xt, r = m % s["tiles_x"], m // s["tiles_x"]
            yt, bt = r % s["tiles_y"], r // s["tiles_y"]
            m = ((s["tiles_b"] - 1 - bt) * s["tiles_y"] + (s["tiles_y"] - 1 - yt)) * s["tiles_x"] + (s["tiles_x"] - 1 - xt)
        return owner, m, nt
    if s["kind"] == _lib.TC_GENERIC_CTA2:
        # cluster c takes units c, c + grid / 2, ...; unit u -> N tile u % tiles_n, M tiles 2 (u / tiles_n) + rank
        owner = np.repeat(w % (s["grid"] // 2), 2)
        nt = np.repeat(w % s["tiles_n"], 2)
        m = (2 * (w // s["tiles_n"])[:, None] + np.arange(2)[None, :]).ravel()
        if rev:
            m = ((s["mtiles"] + 1) & ~1) - 1 - m
        return owner, m, nt
    # halo stream: unit P -> N tile P / upn, patches npair (P % upn) + h
    k = s["npair"]
    owner = np.repeat(w % s["grid"], k)
    nt = np.repeat(w // s["upn"], k)
    m = (k * (w % s["upn"])[:, None] + np.arange(k)[None, :]).ravel()
    if rev:
        m = k * s["upn"] - 1 - m
    return owner, m, nt


def check_schedule(d: _lib.ConvDesc, s: dict, n: int) -> None:
    Ho, Wo, Cout = d.y.H, d.y.W, d.y.C
    assert s["tiles_x"] * s["tw"] >= Wo > (s["tiles_x"] - 1) * s["tw"]
    assert s["tiles_y"] * s["th"] >= Ho > (s["tiles_y"] - 1) * s["th"]
    assert s["tiles_b"] == math.ceil(n / s["tb"]) and s["tiles_n"] * s["block_n"] == Cout
    assert s["mtiles"] == s["tiles_x"] * s["tiles_y"] * s["tiles_b"]
    pair = s["kind"] == _lib.TC_GENERIC_CTA2
    assert 1 <= s["grid"] <= NUM_SMS
    assert (s["grid"] // 2 if pair else s["grid"]) <= s["work"], "a CTA without work"
    if pair:
        assert s["grid"] % 2 == 0
    for rev in (0, 1):
        owner, m, nt = walk(s, rev)
        assert owner.min() == 0 and owner.max() == (s["grid"] // 2 if pair else s["grid"]) - 1
        inside = m < s["mtiles"]
        # an item past the last image tile of the run is only the odd tile of a pair: loads stay in the buffer, stores clip
        assert (~inside).sum() <= (s["tiles_n"] if pair or s["npair"] == 2 else 0), (~inside).sum()
        cnt = np.bincount(m[inside] * s["tiles_n"] + nt[inside], minlength=s["mtiles"] * s["tiles_n"])
        assert cnt.shape[0] == s["mtiles"] * s["tiles_n"] and (cnt == 1).all(), (rev, np.unique(cnt))
        bt = m[inside] // (s["tiles_x"] * s["tiles_y"])
        assert (bt * s["tb"] < n).all()


def _check_all_n(d: _lib.ConvDesc) -> None:
    B = d.y.B
    full = tiling(describe(d))
    for n in range(1, B + 1):
        s = schedule(d, n)
        check_schedule(d, s, n)
        # the tiling never depends on n: it is the one chosen for the whole batch
        assert (s["tb"], s["th"], s["tw"], s["block_n"]) == (full["tb"], full["th"], full["tw"], full["N"])
        assert full["kind"].startswith(_KIND[s["kind"]]) and (full["kind"].endswith("-ybx") == bool(s["ybx"]))
        assert (s["npair"] == 2) == full["pair"]
    # no-change proof: at n = B the grid is the one a full run launches today
    assert schedule(d, B)["grid"] == full["grid"]


@pytest.mark.parametrize("config", sorted(FULL))
def test_full_size_plan_schedules_cover_every_image_prefix(config, dry):
    descs = full_plan_descs(config)
    assert len(descs) > 20
    kinds = set()
    for d in descs:
        kinds.add(schedule(d, d.y.B)["kind"])
        _check_all_n(d)
    assert {_lib.TC_GENERIC, _lib.TC_GENERIC_CTA2, _lib.TC_HALO_STREAM} <= kinds


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_kernel_table_case_schedules_cover_every_image_prefix(case):
    _check_all_n(case_desc(case))


def test_halo_pairs_with_an_odd_image_count_leave_one_patch_out(dry):
    """a ybx tile (8 x 8 pixels of two images) of an odd n reaches image n, and a halo patch pair of an odd patch count
    has one patch past the last: both are walked, neither is counted as covering an image < n"""
    descs = [d for d in full_plan_descs("2") if schedule(d, 64)["kind"] == _lib.TC_HALO_STREAM]
    assert any(schedule(d, 64)["ybx"] for d in descs) and any(schedule(d, 64)["npair"] == 2 for d in descs)
    d = next(d for d in descs if schedule(d, 64)["ybx"])
    s = schedule(d, 7)
    assert s["tb"] == 2 and s["tiles_b"] == 4                # images 0..7: image 7 is computed, its stores clip


def test_tile_cursor_steps_like_the_direct_decode():
    """TileCur (init + carry-propagating step by a constant stride) visits the tiles the division decode names, for the
    per-run tile counts of a partial batch"""
    d = case_desc(CASES[0])
    for n in range(1, d.y.B + 1):
        s = schedule(d, n)
        tn, tx, ty = s["tiles_n"], s["tiles_x"], s["tiles_y"]
        for stride in (s["grid"], 2 * s["grid"], 3 * s["grid"]):
            for t0 in range(min(stride, s["work"])):
                dn, r = stride % tn, stride // tn
                dx, r = r % tx, r // tx
                dy, db = r % ty, r // ty
                nt, r = t0 % tn, t0 // tn
                xt, r = r % tx, r // tx
                yt, bt = r % ty, r // ty
                for t in range(t0, s["work"], stride):
                    assert (nt, xt, yt, bt) == (t % tn, (t // tn) % tx, (t // tn // tx) % ty, t // tn // tx // ty)
                    nt += dn; c = nt >= tn; nt -= tn if c else 0
                    xt += dx + c; c = xt >= tx; xt -= tx if c else 0
                    yt += dy + c; c = yt >= ty; yt -= ty if c else 0
                    bt += db + c


def test_schedule_query_rejects_image_counts_outside_the_batch():
    d = case_desc(CASES[0])
    s = _lib.TcSchedule()
    for n in (0, -1, d.y.B + 1):
        assert _lib.lib().yre_conv_tc_schedule(C.byref(d), NUM_SMS, n, C.byref(s)) == -1
        assert b"images outside" in _lib.lib().yre_last_error()


# ---- plans ------------------------------------------------------------------------------------------------------------
def test_plan_capacity_and_run_batch_errors(dry):
    lib = _lib.lib()
    m = YOLO.from_yaml(ROOT / "configs/models/gelan-c.yaml").eval().set_precision("bf16")
    p = engine.compile_model(m, torch.empty(3, 3, 64, 96), capacity=5)
    assert p.batch == 5 and p.capacity == 5
    for n in (0, -2, 6):
        assert lib.yre_plan_run_batch(p.h, n, None) == -1          # nothing is launched
        assert f"{n} images, the plan holds 1..5".encode() in lib.yre_last_error()
    assert lib.yre_plan_run_batch(None, 1, None) == -1

    # ops recorded for different batches: no capacity, run_batch refuses, run still runs every op for its own batch
    h = C.c_void_p()
    _lib.check(lib.yre_plan_create(C.byref(h)))
    try:
        assert lib.yre_plan_batch_capacity(h) == -1 and b"no ops" in lib.yre_last_error()
        for bn in (2, 3):
            x = _lib.View(0x7f0000000000, _lib.BF16, _lib.NHWC, bn, 4, 4, 8, 0, 8)
            y = _lib.View(0x7f0100000000, _lib.BF16, _lib.NHWC, bn, 8, 8, 8, 0, 8)
            _lib.check(lib.yre_plan_add_upsample2x(h, C.byref(x), C.byref(y)))
        assert lib.yre_plan_batch_capacity(h) == -1 and b"recorded for 3 images" in lib.yre_last_error()
        assert lib.yre_plan_run_batch(h, 1, None) == -1
    finally:
        lib.yre_plan_destroy(h)


@pytest.mark.parametrize("cfg,shape,prec,u8,main_only", [("gelan-c", (3, 3, 640, 640), "bf16", False, False),
                                                          ("gelan-c", (7, 640, 384, 3), "fp16", True, False),
                                                          ("yolov9-c", (1, 3, 384, 640), "fp32", False, True)])
def test_max_batch_changes_the_plan_key_and_nothing_else(dry, cfg, shape, prec, u8, main_only):
    """a model with max_batch = N keys (and compiles) the plan of an n-image input as the plan of N images: the same
    launch list, buffers and outputs as a plan compiled for an N-image input"""
    N = 16
    m = YOLO.from_yaml(ROOT / "configs/models" / f"{cfg}.yaml").eval().set_precision(prec)
    m.main_only = main_only
    x = torch.empty(shape, dtype=torch.uint8 if u8 else torch.float32)
    xN = torch.empty((N,) + shape[1:], dtype=x.dtype)
    assert m.max_batch is None
    key_n, key_N = engine.plan_key(m, x), engine.plan_key(m, xN)
    assert key_n != key_N and key_n[0][0] == shape[0]
    m.max_batch = N
    assert engine.plan_key(m, x) == engine.plan_key(m, xN) == key_N
    assert engine._capacity(m, x) == N
    for bad in (N + 1, 0):
        with pytest.raises(ValueError, match=f"runs 1..{N} images"):
            engine._capacity(m, torch.empty((bad,) + shape[1:]))
    torch.manual_seed(0)
    pN = engine.compile_model(m, xN)
    pc = engine.compile_model(m, x, capacity=N)
    lines_N, lines_c = canonical_lines(pN), canonical_lines(pc)
    # the stem records the image tensor it reads (shape only): the n-image input, re-bound at every forward
    stem = [i for i, (k, _) in enumerate(pc.trace) if k == "stem"]
    assert len(stem) >= 1
    for i, (a, b) in enumerate(zip(lines_N, lines_c)):
        if i in stem:
            assert a.replace(str(tuple(xN.shape)), str(tuple(x.shape))) == b
        else:
            assert a == b, i
    assert len(lines_N) == len(lines_c)
