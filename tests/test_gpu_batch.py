"""GPU tests of batch capacity: a model with max_batch = 16 compiles one plan for 16 images and runs every forward of
n <= 16 images on it (yre_plan_run_batch).

  * same arithmetic: y, every raw logit map and the NMS output of n images are bit-identical to rows [:n] of the
    16-image run of the same plan on a batch that starts with those n images (all three precisions, a dual head and its
    main_only plan, a rectangular plan, uint8 frames);
  * no write beyond n: with every image >= n of every plan-owned buffer filled with a NaN sentinel, a run of n images
    leaves every sentinel in place and still computes the same n results -- so no image's output depends on another
    image's data either;
  * CUDA graphs keyed by (input buffer, n) replay what the eager runs compute;
  * one plan serves n = 1..16, and what a forward allocates is its outputs."""
import pytest
import torch

from oracle import gelan_ref as G
from tests.conftest import ROOT

pytestmark = pytest.mark.gpu

from yolo_b200 import YOLO, engine, non_max_suppression

DEV = "cuda"
CAP = 16
NS = (1, 7, 8, 9, 15, 16)


def build(cfg, sd, prec, main_only=False):
    m = YOLO.from_yaml(ROOT / "configs/models" / f"{cfg}.yaml")
    m.load_state_dict(sd, strict=True)
    m = m.to(DEV).eval().set_precision(prec)
    m.main_only = main_only
    m.max_batch = CAP
    return m


def images(h=640, w=640, u8=False, seed=5):
    x = G.fractal(CAP, h, torch.Generator().manual_seed(seed), w=w)
    if u8:      # BGR frames [B,H,W,3]
        return (x.flip(1) * 255).round().to(torch.uint8).permute(0, 2, 3, 1).contiguous().to(DEV)
    return x.to(DEV)


def flat(out):
    """every tensor of a forward's value (y, raws; both heads of a dual head), in order"""
    if isinstance(out, torch.Tensor):
        return [out]
    return [t for o in out for t in flat(o)]


def ys(out):
    y = out[0]
    return y if isinstance(y, list) else [y]


def same_bits(a: torch.Tensor, b: torch.Tensor) -> bool:
    assert a.dtype == b.dtype == torch.float32 and a.shape == b.shape, (a.shape, b.shape)
    return torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def dets(y):
    return non_max_suppression(y.permute(0, 2, 1), 0.25, 0.45)


CONFIGS = {
    "bf16": dict(cfg="gelan-c", prec="bf16"),
    "fp16": dict(cfg="gelan-c", prec="fp16"),
    "fp32": dict(cfg="gelan-c", prec="fp32"),
    "dual": dict(cfg="yolov9-c", prec="bf16"),
    "main_only": dict(cfg="yolov9-c", prec="bf16", main_only=True),
    "rect640x384": dict(cfg="gelan-c", prec="bf16", h=640, w=384),
    "u8": dict(cfg="gelan-c", prec="bf16", u8=True),
}


def _model_and_images(request, name):
    c = CONFIGS[name]
    nodes, nc, sd = request.getfixturevalue("gelan_c" if c["cfg"] == "gelan-c" else "yolov9_c")
    m = build(c["cfg"], sd, c["prec"], c.get("main_only", False))
    return m, images(c.get("h", 640), c.get("w", 640), c.get("u8", False))


@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_first_n_images_match_the_capacity_run(request, name):
    m, x = _model_and_images(request, name)
    full = [t.clone() for t in flat(m(x))]
    full_dets = [dets(y) for y in ys(m(x))]
    assert len(m._plans) == 1 and next(iter(m._plans.values())).capacity == CAP
    for n in NS:
        out = m(x[:n])
        got = flat(out)
        assert len(got) == len(full)
        for i, (g, f) in enumerate(zip(got, full)):
            assert g.shape[0] == n and same_bits(g, f[:n]), (n, i)
        for y, fd in zip(ys(out), full_dets):
            d = dets(y)
            assert len(d) == n and all(torch.equal(a, b) for a, b in zip(d, fd[:n])), n
    assert len(m._plans) == 1


def _plan_buffers(p: engine.Plan) -> list[tuple[torch.Tensor, bool]]:
    """(tensor, parity-plane layout) of every buffer the plan owns that holds images: the activation windows of its
    launch list and its outputs"""
    acts: dict[int, tuple[torch.Tensor, bool]] = {}

    def visit(o):
        if isinstance(o, engine.V):
            acts[id(o.t)] = (o.t, o.layout == engine.L.PHASE4)
        elif isinstance(o, engine.VCat):
            visit(o.up), visit(o.rest)
        elif isinstance(o, (list, tuple)):
            for e in o:
                visit(e)

    for kind, a in p.trace:
        for k, v in a.items():
            if k == "y" and kind == "decode":
                acts[id(v)] = (v, False)
            elif k != "x" or kind != "stem":          # the stem's x is the caller's image tensor
                visit(v)
    keep = {id(t) for t in p.keep}
    assert set(acts) <= keep
    return list(acts.values())


def _rows(t: torch.Tensor, phase4: bool, n: int) -> torch.Tensor:
    return t[:, n:] if phase4 else t[n:]


@pytest.mark.parametrize("name", ["bf16", "fp16", "fp32", "dual", "u8"])
def test_no_buffer_row_past_n_is_written(request, name):
    m, x = _model_and_images(request, name)
    m.fresh_outputs = False                               # outputs are plan buffers too
    full = [t.clone() for t in flat(m(x))]
    p = next(iter(m._plans.values()))
    bufs = _plan_buffers(p)
    assert sum(ph for _, ph in bufs) >= 1 and len(bufs) > 20
    for n in (1, 7, 9, 15):
        for t, ph in bufs:
            _rows(t, ph, n).fill_(float("nan"))
        got = flat(m(x[:n]))
        torch.cuda.synchronize()
        for i, (t, ph) in enumerate(bufs):
            assert torch.isnan(_rows(t, ph, n)).all(), (n, i, tuple(t.shape))
        for i, (g, f) in enumerate(zip(got, full)):
            assert g.shape[0] == n and same_bits(g, f[:n]), (n, i)


def test_cuda_graphs_per_input_buffer_and_image_count(gelan_c):
    nodes, nc, sd = gelan_c
    m = build("gelan-c", sd, "bf16")
    m.fresh_outputs = False
    x = images()
    eager = {n: [t.clone() for t in flat(m(x[:n]))] for n in (CAP, 3)}
    m.use_cuda_graph = True
    for n in (CAP, 3, CAP, 3):
        got = flat(m(x[:n]))
        assert all(g.shape[0] == n and same_bits(g, e) for g, e in zip(got, eager[n])), n
    p = next(iter(m._plans.values()))
    assert len(m._plans) == 1 and set(p.graphs) == {(x.data_ptr(), CAP), (x.data_ptr(), 3)}


def test_one_plan_serves_every_batch_size(gelan_c):
    nodes, nc, sd = gelan_c
    m = build("gelan-c", sd, "bf16")
    x = images()
    out = m(x[:1])
    del out
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    for n in range(1, CAP + 1):
        out = m(x[:n])
        torch.cuda.synchronize()
        storages = {t.untyped_storage().data_ptr(): t.untyped_storage().nbytes() for t in flat(out)}
        out_bytes = sum(-(-b // 512) * 512 for b in storages.values())
        assert all(t.shape[0] == n for t in flat(out))
        assert torch.cuda.memory_allocated() - base <= out_bytes, (n, torch.cuda.memory_allocated() - base, out_bytes)
        del out
    assert len(m._plans) == 1
    with pytest.raises(ValueError, match=f"runs 1..{CAP} images"):
        m(images()[:0])
    x17 = torch.cat([x, x[:1]])
    with pytest.raises(ValueError, match=f"runs 1..{CAP} images"):
        m(x17)
