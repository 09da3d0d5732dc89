"""GPU tests of shape arenas: with model.max_shape = (672, 672) and model.max_batch = 32, the plans of 640², 640x384,
384x640, 512x672 and 672x672 inputs take their buffers from one arena.

  * same arithmetic: y, every raw logit map and the NMS output of an arena plan are bit-identical to those of a plan with
    buffers of its own and the same max_batch (bf16, fp16, fp32, uint8 frames; n in {1, 7, 32}).  The shapes run
    interleaved, so every run starts on an arena another shape has just written, and the arena is filled with NaN
    before each shape's first run: no kernel reads a cell it did not write in that run;
  * CUDA-graph replays of the arena plans match their eager runs;
  * test-time augmentation with max_shape matches it without;
  * what the forwards allocate is the arena and one upload of the weights, bounded from the plans' act_bytes;
  * the Evaluator scores rectangular batches (x by W, y by H) and square batches exactly as before."""
import pytest
import torch

from oracle import gelan_ref as G
from tests.conftest import ROOT

pytestmark = pytest.mark.gpu

from yolo_b200 import Evaluator, YOLO, compute_map, non_max_suppression

DEV = "cuda"
CAP = 32
NS = (1, 7, 32)
MAX = (672, 672)
SHAPES = [(640, 640), (640, 384), (384, 640), (512, 672), (672, 672)]


def build(sd, prec, max_shape=None, cap=CAP):
    m = YOLO.from_yaml(ROOT / "configs/models/gelan-c.yaml")
    m.load_state_dict(sd, strict=True)
    m = m.to(DEV).eval().set_precision(prec)
    m.max_batch, m.max_shape = cap, max_shape
    return m


def images(h, w, u8=False, seed=5, n=CAP):
    x = G.fractal(n, h, torch.Generator().manual_seed(seed + h + 7 * w), w=w)
    if u8:      # BGR frames [B,H,W,3]
        return (x.flip(1) * 255).round().to(torch.uint8).permute(0, 2, 3, 1).contiguous().to(DEV)
    return x.to(DEV)


def flat(out):
    if isinstance(out, torch.Tensor):
        return [out]
    return [t for o in out for t in flat(o)]


def same_bits(a: torch.Tensor, b: torch.Tensor) -> bool:
    assert a.dtype == b.dtype == torch.float32 and a.shape == b.shape, (a.shape, b.shape)
    return torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def dets(y):
    return non_max_suppression(y.permute(0, 2, 1), 0.001, 0.7, multi_label=True)


def results(m, x):
    """(every output tensor cloned, NMS rows) of a forward"""
    out = m(x)
    return [t.clone() for t in flat(out)], [d.clone() for d in dets(out[0])]


def assert_same(a, b, what):
    (ta, da), (tb, db) = a, b
    assert len(ta) == len(tb) and len(da) == len(db)
    for i, (u, v) in enumerate(zip(ta, tb)):
        assert same_bits(u, v), f"{what}: output {i} differs"
    for i, (u, v) in enumerate(zip(da, db)):
        assert same_bits(u, v), f"{what}: NMS rows of image {i} differ"


def nan_fill(m):
    for a in m._arenas.values():
        a.fill_(0xFF)          # all-ones bytes: NaN in bf16, fp16 and fp32


@pytest.mark.parametrize("prec,u8", [("bf16", False), ("fp16", False), ("fp32", False), ("bf16", True)])
def test_arena_plans_match_plans_with_their_own_buffers(gelan_c, prec, u8):
    _, _, sd = gelan_c
    own, arena = build(sd, prec), build(sd, prec, MAX)
    arena.fresh_outputs = False                     # static outputs: y and the raw maps live in the arena as well
    xs = {s: images(*s, u8=u8) for s in SHAPES}
    ref = {(s, n): results(own, xs[s][:n]) for n in NS for s in SHAPES}
    seen = set()
    for n in NS:
        for s in SHAPES:                             # interleaved: the previous shape has just written the arena
            if s not in seen:
                if not arena._arenas:
                    arena(xs[s][:n])                 # the first forward allocates the arena
                nan_fill(arena)
                seen.add(s)
            assert_same(results(arena, xs[s][:n]), ref[(s, n)], f"{prec}{' u8' if u8 else ''} {s} n={n}")
    assert len(arena._arenas) == 1 and len(arena._plans) == len(SHAPES)
    # the plans are the same launch lists: same variants and tilings
    for key, p in arena._plans.items():
        q = own._plans[key[:-1]]
        assert p.op_variants() == q.op_variants() and p.num_launches == q.num_launches and p.act_bytes == q.act_bytes
    # a cell none of a run's kernels writes stays NaN only where no output reads it: the first run after a NaN fill
    # above matched bit for bit, so every cell an output depends on was written in that run


def test_cuda_graph_replays_match_eager_runs(gelan_c):
    _, _, sd = gelan_c
    eager, graph = build(sd, "bf16", MAX), build(sd, "bf16", MAX)
    eager.fresh_outputs = graph.fresh_outputs = False
    graph.use_cuda_graph = True
    xs = {s: images(*s) for s in SHAPES}
    for rnd in range(2):
        for n in (7, CAP):
            for s in SHAPES:
                assert_same(results(graph, xs[s][:n]), results(eager, xs[s][:n]), f"graph {s} n={n} round {rnd}")


def test_tta_with_max_shape_matches_tta_without(gelan_c):
    _, _, sd = gelan_c
    own, arena = build(sd, "bf16", cap=8), build(sd, "bf16", MAX, cap=8)
    arena.fresh_outputs = False
    for rnd in range(2):
        for s in ((640, 640), (384, 640), (672, 512)):
            x = images(*s, n=8)[:7]
            a = arena(x, augment=True)[0].clone()
            b = own(x, augment=True)[0]
            assert same_bits(a, b), (s, rnd)
    assert len(arena._arenas) == 3                   # branch 0 (the plain plans') and one per scaled branch


def test_memory_is_one_arena_and_one_upload_of_the_weights(gelan_c):
    _, _, sd = gelan_c
    xs = {s: images(*s) for s in SHAPES}
    torch.cuda.synchronize()
    grow = {}
    for arm in ("own", "arena"):
        m = build(sd, "bf16", MAX if arm == "arena" else None)
        m.fresh_outputs = False
        base = torch.cuda.memory_allocated()
        for s in SHAPES:
            m(xs[s])
        torch.cuda.synchronize()
        grow[arm] = torch.cuda.memory_allocated() - base
        plans = list(m._plans.values())
        if arm == "arena":
            (arena,) = m._arenas.values()
            (_, wcache), = m._arena_weights.values()
            # the caching allocator hands out multiples of 512 B
            wbytes = sum(-(-t.numel() * t.element_size() // 512) * 512 for wb in wcache.values() for t in wb)
            # the arena is the layout of the 672² plan: its activations, y, and less than ARENA_ALIGN per buffer
            big = m._plans[max(m._plans, key=lambda k: k[0][2] * k[0][3])]
            nbuf = sum(1 for t in big.keep if t.untyped_storage().data_ptr() == arena.data_ptr())
            ybytes = big.result[1].numel() * 4
            assert big.act_bytes + ybytes <= arena.numel() < big.act_bytes + ybytes + 512 * nbuf
            assert all(p.act_bytes <= big.act_bytes for p in plans)
            # what the five forwards allocated: the arena and one upload of the weights, no output and no other buffer.
            # The slack is the caching allocator's: a block of the large pool is not split when less than 1 MiB of it
            # would remain, and counts whole (1.9 MiB here on one B200); a plan's own buffers would be gigabytes
            print(f"arena {arena.numel()} B, shared weights {wbytes} B, allocated {grow['arena']} B")
            assert arena.numel() + wbytes <= grow["arena"] <= arena.numel() + wbytes + 4 * 2**20 + 65536 * len(plans)
        else:
            assert grow["own"] >= sum(p.act_bytes for p in plans)
        del m, plans
        torch.cuda.empty_cache()
    print(f"allocated by 5 shapes at capacity {CAP}: own buffers {grow['own'] / 2**30:.2f} GiB, "
          f"arena {grow['arena'] / 2**30:.2f} GiB")
    assert grow["arena"] < grow["own"] / 2


def _targets_from(dets_list, H, W, k=4):
    """normalised (image, class, cx, cy, w, h) of the first k detections of every image (so the model scores above 0)"""
    rows = []
    for i, d in enumerate(dets_list):
        d = d[:k].float()
        cx, cy = (d[:, 0] + d[:, 2]) / 2 / W, (d[:, 1] + d[:, 3]) / 2 / H
        w, h = (d[:, 2] - d[:, 0]) / W, (d[:, 3] - d[:, 1]) / H
        rows.append(torch.stack([torch.full_like(cx, i), d[:, 5], cx, cy, w, h], 1))
    return torch.cat(rows).cpu()


def _loader(m, shapes, n=4):
    out = []
    for s in shapes:
        x = images(*s, n=n)
        out.append((x, _targets_from(dets_eval(m, x), *s), None, None))
    return out


def dets_eval(m, x):
    return non_max_suppression(m(x)[0].permute(0, 2, 1).contiguous(), conf_thres=0.001, iou_thres=0.6)


def _gt(targets, bsz, sx, sy):
    """the reference's ground-truth arithmetic (evaluator.py:139-141) with x scaled by sx and y by sy"""
    gtb, gtc = [], []
    for i in range(bsz):
        t = targets[targets[:, 0] == i].to(DEV)
        xywh = t[:, 2:6].float() * torch.tensor([sx, sy, sx, sy], dtype=torch.float32, device=DEV)
        gtb.append(torch.stack([xywh[:, 0] - xywh[:, 2] / 2, xywh[:, 1] - xywh[:, 3] / 2,
                                xywh[:, 0] + xywh[:, 2] / 2, xywh[:, 1] + xywh[:, 3] / 2], 1))
        gtc.append(t[:, 1].long())
    return gtb, gtc


def _square_gt(targets, bsz, img_size):
    """the parent's square-only arithmetic, verbatim: * img_size"""
    gtb, gtc = [], []
    for i in range(bsz):
        t = targets[targets[:, 0] == i].to(DEV)
        xywh = t[:, 2:6].float() * img_size
        xyxy = torch.zeros_like(xywh)
        xyxy[:, 0] = xywh[:, 0] - xywh[:, 2] / 2
        xyxy[:, 1] = xywh[:, 1] - xywh[:, 3] / 2
        xyxy[:, 2] = xywh[:, 0] + xywh[:, 2] / 2
        xyxy[:, 3] = xywh[:, 1] + xywh[:, 3] / 2
        gtb.append(xyxy)
        gtc.append(t[:, 1].long())
    return gtb, gtc


def _expected_map(m, loader, gt_fn):
    pb, ps, pc, gb, gc = [], [], [], [], []
    for x, targets, _, _ in loader:
        for d in dets_eval(m, x):
            pb.append(d[:, :4]), ps.append(d[:, 4]), pc.append(d[:, 5].long())
        b, c = gt_fn(targets, x)
        gb += b
        gc += c
    return compute_map(pb, ps, pc, gb, gc, 80)


def test_evaluator_scores_rectangular_batches(gelan_c):
    _, _, sd = gelan_c
    m = build(sd, "bf16", (640, 640), cap=4)
    mixed = _loader(m, [(640, 640), (384, 640), (640, 384), (320, 320)])
    got = Evaluator(m, mixed).evaluate()
    want = _expected_map(m, mixed, lambda t, x: _gt(t, x.shape[0], x.shape[3], x.shape[2]))
    assert got == want and got["map50"] > 0
    # a rectangular batch scaled by its height alone (the old arithmetic) scores differently
    wrong = _expected_map(m, mixed, lambda t, x: _gt(t, x.shape[0], x.shape[2], x.shape[2]))
    assert wrong != want

    square = _loader(m, [(640, 640), (320, 320)])
    got = Evaluator(m, square).evaluate()
    assert got == _expected_map(m, square, lambda t, x: _square_gt(t, x.shape[0], x.shape[2]))
