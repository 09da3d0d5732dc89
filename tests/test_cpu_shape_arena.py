"""CPU tests of shape arenas (model.max_shape): the plans of every input shape up to a maximum take their buffers from one
device byte buffer sized for model.max_batch images of that maximum.

On dry plans (host buffers) and on layout-only plans (engine.arena_bytes), without a GPU:
  * every stride-32 rectangle from 32 x 32 up to the maximum fits the arena, for gelan-c, yolov9-c (dual head and
    main_only) and the test-time-augmentation branch plans, at maxima 640² and 1280² and capacities 64 and 16;
  * the buffers of one arena plan are disjoint windows of the arena, at ARENA_ALIGN-aligned offsets in allocation order;
  * an arena plan records the same launches, variants, views, weights and act_bytes as a plan with buffers of its own;
  * plans that share an arena share one upload of each packed weight;
  * the error paths, and that max_shape = None leaves plan_key unchanged."""
import pytest
import torch

from tests.conftest import ROOT
from tests.test_cpu_plan_launch_list import canonical_lines

from yolo_b200 import YOLO, _lib, engine, tta

CONFIGS = {"gelan-c": ("gelan-c", False), "yolov9-c": ("yolov9-c", False), "yolov9-c_main_only": ("yolov9-c", True)}


@pytest.fixture()
def dry():
    engine._ALLOW_CPU_DRY_RUN = True
    yield
    engine._ALLOW_CPU_DRY_RUN = False


@pytest.fixture(scope="module")
def models():
    return {name: YOLO.from_yaml(ROOT / "configs/models" / f"{name}.yaml").eval() for name in ("gelan-c", "yolov9-c")}


@pytest.fixture(scope="module", autouse=True)
def fold_once():
    """Each module is folded once for the whole module: the layout of a plan does not depend on weight values, and
    thousands of layouts are checked below."""
    memo, fold = {}, engine.Plan.fold

    def memo_fold(self, m):
        if id(m) not in memo:
            memo[id(m)] = fold(self, m)
        return memo[id(m)]

    engine.Plan.fold = memo_fold
    yield
    engine.Plan.fold = fold


def layout_end(model, H, W, cap, main_only) -> int:
    """bytes of the arena layout of a plan for cap images of H x W (what it needs of an arena)"""
    x = torch.empty((), dtype=torch.float32).expand(cap, 3, H, W)
    return engine.compile_model(model, x, cap, main_only, layout_only=True).arena_end


def rectangles(M: int):
    return [(h, w) for h in range(32, M + 1, 32) for w in range(32, M + 1, 32)]


@pytest.mark.parametrize("cap", [64, 16])
@pytest.mark.parametrize("M", [640, 1280])
@pytest.mark.parametrize("config", sorted(CONFIGS))
def test_every_rectangle_fits_the_arena(models, config, M, cap):
    name, main_only = CONFIGS[config]
    m = models[name]
    size = engine.arena_bytes(m, 3, M, M, cap, main_only)
    assert size % engine.ARENA_ALIGN == 0
    worst = max((layout_end(m, h, w, cap, main_only), h, w) for h, w in rectangles(M))
    # the arena is the layout of the largest plan, and no smaller rectangle needs more
    assert worst[0] <= size, worst
    assert layout_end(m, M, M, cap, main_only) == size


@pytest.mark.parametrize("cap", [64, 16])
@pytest.mark.parametrize("M", [640, 1280])
def test_every_tta_branch_plan_fits_its_arena(models, M, cap):
    """the branch-i plans of every stride-32 input up to M x M fit the arena sized for the branch-i input of M x M"""
    m = models["gelan-c"]
    gmax = tta.geometry(M, M)
    for i in (1, 2):
        size = engine.arena_bytes(m, 3, gmax.out_h[i], gmax.out_w[i], cap)
        shapes = {(tta.geometry(h, w).out_h[i], tta.geometry(h, w).out_w[i]) for h, w in rectangles(M)}
        assert all(bh <= gmax.out_h[i] and bw <= gmax.out_w[i] for bh, bw in shapes)
        worst = max((layout_end(m, bh, bw, cap, None), bh, bw) for bh, bw in shapes)
        assert worst[0] <= size, (i, worst)


def _arena_plan(m, x, cap, main_only, M, wcache=None):
    arena = torch.empty(engine.arena_bytes(m, 3, M, M, cap, main_only), dtype=torch.uint8)
    return engine.compile_model(m, x, cap, main_only, arena=arena, wcache={} if wcache is None else wcache), arena


def _weights(p: engine.Plan) -> set[int]:
    return {id(a[k]) for kind, a in p.trace if kind in ("conv", "stem") for k in ("w", "b")}


def _buffers(p: engine.Plan) -> list[torch.Tensor]:
    """the activation buffers and static outputs a plan allocated"""
    return [t for t in p.keep if id(t) not in _weights(p)]


def _check_disjoint(p: engine.Plan, arena: torch.Tensor) -> int:
    """every buffer of p is a window of the arena at an aligned offset, after the previous one; returns their count"""
    base, end, n = arena.data_ptr(), arena.data_ptr(), 0
    for t in p.keep:
        if t.untyped_storage().data_ptr() != base:
            continue                               # a weight or bias (not in the arena)
        lo, hi = t.data_ptr(), t.data_ptr() + t.numel() * t.element_size()
        assert t.is_contiguous() and (lo - base) % engine.ARENA_ALIGN == 0
        assert end <= lo and hi <= base + arena.numel(), (lo - base, hi - base, end - base)
        end, n = hi, n + 1
    return n


@pytest.mark.parametrize("M,cap,shapes", [(640, 64, [(640, 640), (384, 640), (640, 384), (32, 32), (608, 96)]),
                                          (1280, 16, [(1280, 1280), (736, 1280), (1280, 224), (512, 672)])])
@pytest.mark.parametrize("config", sorted(CONFIGS))
def test_arena_plans_are_the_plans_without_an_arena(dry, models, config, M, cap, shapes):
    """same trace, op table, variants, launch count, views, weights and act_bytes; every buffer a disjoint window"""
    name, main_only = CONFIGS[config]
    m = models[name].set_precision("bf16")
    for h, w in shapes:
        x = torch.empty(cap, 3, h, w)
        own = engine.compile_model(m, x, cap, main_only)
        p, arena = _arena_plan(m, x, cap, main_only, M)
        assert canonical_lines(p) == canonical_lines(own)
        assert p.op_variants() == own.op_variants() and p.num_launches == own.num_launches
        assert p.act_bytes == own.act_bytes
        # the activations and y: every buffer of the plan is in the arena, none overlaps another
        assert _check_disjoint(p, arena) == len(_buffers(p)) == len(_buffers(own))


def test_uint8_and_fp32_inputs_share_an_arena_layout(models):
    m = models["gelan-c"]
    a = engine.compile_model(m, torch.empty((), dtype=torch.uint8).expand(16, 384, 640, 3), 16, layout_only=True)
    b = engine.compile_model(m, torch.empty((), dtype=torch.float32).expand(16, 3, 384, 640), 16, layout_only=True)
    assert a.arena_end == b.arena_end


def test_plans_of_one_arena_upload_each_weight_once(dry, models):
    m = models["gelan-c"].set_precision("bf16")
    wcache: dict = {}
    p1, _ = _arena_plan(m, torch.empty(64, 3, 640, 640), 64, None, 640, wcache)
    keys1 = set(wcache)
    p2, _ = _arena_plan(m, torch.empty(64, 3, 64, 96), 64, None, 640, wcache)
    new = set(wcache) - keys1
    # the 640² plan runs the first box and class convs of the two large levels apart, the 64 x 96 plan merges them into
    # one GEMM: those two merged weights are the only new uploads, every other weight is the 640² plan's tensor
    assert sorted(new) == [("conv", f"layers.detect.box_convs.{i}.0", f"layers.detect.cls_convs.{i}.0", torch.bfloat16)
                           for i in (0, 1)]
    assert len(_weights(p2) - _weights(p1)) == 2 * len(new)
    for key, (w, b) in wcache.items():
        assert key[-1] == w.dtype == (torch.float32 if key[0] == "stem" else torch.bfloat16) and b.dtype == torch.float32


def test_a_plan_that_does_not_fit_raises_naming_the_shape(dry, models):
    m = models["gelan-c"].set_precision("bf16")
    arena = torch.empty(engine.arena_bytes(m, 3, 384, 640, 16), dtype=torch.uint8)
    with pytest.raises(_lib.YreError, match="16 x 640 x 640"):
        engine.compile_model(m, torch.empty(16, 3, 640, 640), 16, arena=arena, wcache={})


def test_max_shape_errors():
    m = YOLO.from_yaml(ROOT / "configs/models/gelan-c.yaml").eval()
    x = torch.empty(2, 3, 384, 640)
    assert engine._max_shape(m, x) is None
    m.max_shape = (640, 640)
    with pytest.raises(ValueError, match="max_shape.*max_batch"):
        engine._max_shape(m, x)
    m.max_batch = 16
    assert engine._max_shape(m, x) == (640, 640)
    assert engine._max_shape(m, torch.empty(2, 640, 640, 3, dtype=torch.uint8)) == (640, 640)
    for big in (torch.empty(2, 3, 672, 640), torch.empty(2, 3, 640, 672), torch.empty(2, 640, 672, 3, dtype=torch.uint8)):
        with pytest.raises(ValueError, match="up to 640 x 640"):
            engine._max_shape(m, big)
    for bad in ((640,), (0, 640), (640, -32)):
        m.max_shape = bad
        with pytest.raises(ValueError, match="height, width"):
            engine._max_shape(m, x)


def test_max_shape_none_leaves_the_plan_key():
    m = YOLO.from_yaml(ROOT / "configs/models/gelan-c.yaml").eval()
    x = torch.empty(7, 3, 384, 640)
    assert m.max_shape is None
    assert engine.plan_key(m, x) == ((7, 3, 384, 640), torch.float32, None, "bf16", True, False)
    m.max_batch = 16
    assert engine.plan_key(m, x) == ((16, 3, 384, 640), torch.float32, None, "bf16", True, False)
    m.max_shape = (640, 640)
    assert engine.plan_key(m, x) == ((16, 3, 384, 640), torch.float32, None, "bf16", True, False, ("max_shape", (640, 640)))


def test_act_bytes_without_an_arena_is_the_parents(dry, models):
    """the buffers of a plan without an arena are those of the parent commit's alloc (gelan-c, 64 x 640², bf16)"""
    p = engine.compile_model(models["gelan-c"].set_precision("bf16"), torch.empty(64, 3, 640, 640))
    assert p.act_bytes == 11064115200
