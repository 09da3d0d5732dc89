"""Test-time augmentation on the GPU: model(x, augment=True).

  * K12 (yre_tta_scale_img) equals K12's fp32 formula (oracle/tta_ref.py scale_img_exact) bit for bit and torch's
    F.interpolate + F.pad within 1e-6, for the mirrored and the plain branch, square and rectangular, n < B; uint8 frames
    give the same images as the fp32 tensor preprocess() makes of them;
  * K13 (yre_tta_merge) equals a torch restatement bit for bit;
  * the fp32 engine matches the oracle's TTA within the repo's 1e-4 gate, and NMS on the merged y is bit-exact against the
    C reference (detections and kept anchors);
  * bf16 / fp16: the merged y is bit-identical to the restatement over plain forwards of the three branch inputs;
  * CUDA-graph replay, batch capacity, the dual head and Evaluator(augment=True)."""
import numpy as np
import pytest
import torch

from oracle import gelan_ref as G
from oracle import nms_ref as N
from oracle import tta_ref as T
from tests.conftest import ROOT

pytestmark = pytest.mark.gpu

import yolo_b200
from yolo_b200 import YOLO, Evaluator, nms_raw, preprocess, tta

DEV = "cuda"


def _model(name, sd, prec, **attrs):
    m = YOLO.from_yaml(ROOT / "configs/models" / f"{name}.yaml")
    m.load_state_dict(sd, strict=True)
    m = m.to(DEV).eval().set_precision(prec)
    for k, v in attrs.items():
        setattr(m, k, v)
    return m


def same_bits(a: torch.Tensor, b: torch.Tensor) -> bool:
    assert a.dtype == b.dtype == torch.float32 and a.shape == b.shape, (a.shape, b.shape)
    return torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def restate(ys: list[torch.Tensor], g) -> torch.Tensor:
    """descale + clip + concat of [n, A_i, 4+nc] rows in torch (fp32 division on the CPU, where it is IEEE division)"""
    parts = []
    for i, y in enumerate(ys):
        p = y[:, g.a_begin[i]:g.a_end[i]].cpu().clone()
        p[..., :4] = p[..., :4] / torch.tensor(g.scale[i], dtype=torch.float32)
        if g.flip[i]:
            p[..., 0] = g.w - p[..., 0]
        parts.append(p)
    return torch.cat(parts, 1)


# ---- K12 -----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,n,h,w", [(3, 3, 128, 128), (4, 2, 384, 640), (2, 1, 640, 384), (1, 1, 64, 96), (2, 2, 640, 640)])
def test_k12_is_bit_exact_and_agrees_with_torch(B, n, h, w):
    x = G.fractal(B, h, torch.Generator().manual_seed(h * w + B), w=w)
    xd = x.to(DEV)
    g = tta.geometry(h, w)
    for i in (1, 2):
        flip = bool(g.flip[i])
        out = torch.full((B, 3, g.out_h[i], g.out_w[i]), float("nan"), device=DEV)
        tta.scale_img(xd, g, i, out=out, n=n)
        got = out[:n].cpu().numpy()
        ref = T.scale_img_exact(x[:n].numpy(), T.SCALES[i], flip)
        assert np.array_equal(got.view(np.int32), ref.view(np.int32)), (i, np.abs(got - ref).max())
        assert torch.isnan(out[n:]).all()                                # no image >= n written
        tref = T.scale_img(xd[:n].flip(3) if flip else xd[:n], T.SCALES[i])
        assert (out[:n] - tref).abs().max().item() <= 1e-6, i
        tcpu = T.scale_img(x[:n].flip(3) if flip else x[:n], T.SCALES[i])
        assert np.abs(got - tcpu.numpy()).max() <= 1e-6, i


@pytest.mark.parametrize("h,w", [(384, 640), (128, 128)])
def test_k12_from_uint8_frames_equals_the_preprocessed_tensor(h, w):
    rng = np.random.default_rng(h + w)
    frames = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for _ in range(3)]
    xf, _, _ = preprocess(frames, (h, w))                                 # fp32 RGB / 255: what model(x) would get
    xu, _, _ = preprocess(frames, (h, w), dtype=torch.uint8)
    g = tta.geometry(h, w)
    for i in (1, 2):
        assert same_bits(tta.scale_img(xu, g, i), tta.scale_img(xf, g, i)), i


# ---- K13 -----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nc", [80, 3])
@pytest.mark.parametrize("B,h,w", [(1, 128, 128), (7, 384, 640), (64, 640, 640)])
def test_k13_equals_the_torch_restatement(nc, B, h, w):
    g = tta.geometry(h, w)
    gen = torch.Generator(device=DEV).manual_seed(B + nc)
    ys = [torch.rand((B, g.A[i], 4 + nc), generator=gen, device=DEV) * 900 - 100 for i in range(3)]
    ref = restate(ys, g)
    out = tta.merge(ys, g)
    assert tuple(out.shape) == (B, g.A_tot, 4 + nc) and same_bits(out.cpu(), ref)
    # n < B: the first n images, nothing past them
    n = max(1, B // 2)
    big = torch.full((B, g.A_tot, 4 + nc), float("nan"), device=DEV)
    tta.merge([y[:n] for y in ys], g, out=big)
    assert same_bits(big[:n].cpu(), ref[:n]) and torch.isnan(big[n:]).all()


# ---- the path --------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("H,W,batch", [(128, 128, 2), (192, 320, 1)])
def test_fp32_tta_vs_oracle_and_nms(gelan_c, H, W, batch):
    nodes, nc, sd = gelan_c
    x = G.fractal(batch, H, torch.Generator().manual_seed(H + W + 1), w=W)
    y_ref, _ = T.forward_augment(lambda xi: G.forward(nodes, nc, sd, xi)[0], x)
    sd64 = {k: (v.double() if v.is_floating_point() else v) for k, v in sd.items()}
    y64, _ = T.forward_augment(lambda xi: G.forward(nodes, nc, sd64, xi)[0], x.double())
    floor_box = (y_ref[:, :4].double() - y64[:, :4]).abs().max().item()
    floor_sc = (y_ref[:, 4:].double() - y64[:, 4:]).abs().max().item()
    y, none = _model("gelan-c", sd, "fp32")(x.to(DEV), augment=True)
    assert none is None and y.shape == y_ref.shape == (batch, 84, tta.geometry(H, W).A_tot)
    dbox = (y[:, :4].cpu().double() - y64[:, :4]).abs().max().item()
    dsc = (y[:, 4:].cpu().double() - y64[:, 4:]).abs().max().item()
    print(f"TTA {H}x{W} B{batch}: ours-vs-fp64 |dbox|={dbox:.3e}px |dscore|={dsc:.3e}; oracle floor {floor_box:.3e}px {floor_sc:.3e}")
    assert dbox <= max(1e-4 * max(H, W), 3 * floor_box) and dsc <= max(1e-4, 3 * floor_sc)
    pred = y.permute(0, 2, 1).contiguous()
    out, counts, keep = nms_raw(pred, 0.25, 0.45)
    dets, keeps = N.non_max_suppression(pred.cpu(), 0.25, 0.45, return_keep=True)
    assert sum(len(d) for d in dets) > 0
    for i, (d, k) in enumerate(zip(dets, keeps)):
        c = int(counts[i])
        assert c == len(d) and np.array_equal(out[i, :c].cpu().numpy(), d) and np.array_equal(keep[i, :c].cpu().numpy(), k)


@pytest.mark.parametrize("prec", ["bf16", "fp16"])
def test_16bit_tta_is_the_merge_of_plain_forwards(gelan_c, prec):
    nodes, nc, sd = gelan_c
    m = _model("gelan-c", sd, prec)
    xd = G.fractal(3, 384, torch.Generator().manual_seed(17), w=640).to(DEV)
    g = tta.geometry(384, 640)
    xs = [xd] + [tta.scale_img(xd, g, i) for i in (1, 2)]
    ys = [m(xi)[0].permute(0, 2, 1).contiguous() for xi in xs]         # plain forwards of the branch inputs
    y, _ = m(xd, augment=True)
    assert same_bits(y.permute(0, 2, 1).cpu(), restate(ys, g))
    assert same_bits(y[:, :, :g.a_end[0]], m(xd)[0][:, :, :g.a_end[0]])  # branch 0: the plain forward of x (s = 1)
    assert len(m._plans) == 5                                           # x, the two scaled inputs, the two branch plans


def test_cuda_graph_replay_equals_eager(gelan_c):
    nodes, nc, sd = gelan_c
    m = _model("gelan-c", sd, "bf16")
    xd = G.fractal(4, 384, torch.Generator().manual_seed(23), w=640).to(DEV)
    eager = m(xd, augment=True)[0].clone()
    m.fresh_outputs, m.use_cuda_graph = False, True
    for _ in range(3):
        y, _ = m(xd, augment=True)
        assert same_bits(y, eager)
    assert len(m._plans) == 3 and all(len(p.graphs) == 1 for p in m._plans.values())


def test_capacity_runs_the_first_n_images(gelan_c):
    nodes, nc, sd = gelan_c
    m = _model("gelan-c", sd, "bf16", max_batch=16)
    xd = G.fractal(16, 320, torch.Generator().manual_seed(29), w=384).to(DEV)
    full = m(xd, augment=True)[0].clone()
    for n in (1, 7, 16):
        y, _ = m(xd[:n], augment=True)
        assert y.shape[0] == n and same_bits(y, full[:n]), n
    m.fresh_outputs = False
    for n in (7, 1):
        y, _ = m(xd[:n], augment=True)
        assert y.shape[0] == n and same_bits(y, full[:n]), n
    assert len(m._plans) == 3 and len(m._tta) == 1
    with pytest.raises(ValueError, match="runs 1..16 images"):
        m(torch.cat([xd, xd[:1]]), augment=True)


def test_non_multiples_of_32_are_rejected(gelan_c):
    nodes, nc, sd = gelan_c
    m = _model("gelan-c", sd, "bf16")
    with pytest.raises(ValueError, match="multiples of 32"):
        m(torch.zeros(1, 3, 100, 128, device=DEV), augment=True)
    assert not m._plans


def test_dual_head_tta_equals_its_main_only_tta(yolov9_c):
    nodes, nc, sd = yolov9_c
    xd = G.fractal(2, 256, torch.Generator().manual_seed(31), w=384).to(DEV)
    ya, none = _model("yolov9-c", sd, "bf16")(xd, augment=True)
    yb, _ = _model("yolov9-c", sd, "bf16", main_only=True)(xd, augment=True)
    assert none is None and isinstance(ya, torch.Tensor) and same_bits(ya, yb)


def test_evaluator_with_augment(gelan_c):
    from oracle import metrics_ref as MR
    nodes, nc, sd = gelan_c
    m = _model("gelan-c", sd, "bf16")
    rng = np.random.default_rng(7)
    S, batches = 256, []
    for bi in range(2):
        imgs = G.fractal(3, S, torch.Generator().manual_seed(40 + bi))
        rows = []
        for i in range(3):
            k = int(rng.integers(1, 6))
            cxy, wh = rng.uniform(0.2, 0.8, (k, 2)), rng.uniform(0.05, 0.4, (k, 2))
            rows += [[i, int(rng.integers(0, nc)), *cxy[j], *wh[j]] for j in range(k)]
        batches.append((imgs, torch.tensor(rows, dtype=torch.float32).reshape(-1, 6), None, [(S, S)] * 3))
    got = Evaluator(m, batches, num_classes=nc, conf_thres=0.25, iou_thres=0.45, augment=True).evaluate()
    pb, ps, pc, gb, gc = [], [], [], [], []
    for imgs, targets, _, _ in batches:
        y, _ = m(imgs.to(DEV), augment=True)
        dets = yolo_b200.non_max_suppression(y.permute(0, 2, 1).contiguous(), 0.25, 0.45)
        for i in range(imgs.shape[0]):
            d = dets[i].cpu().numpy()
            pb.append(d[:, :4]); ps.append(d[:, 4]); pc.append(d[:, 5].astype(np.int64))
            t = targets[targets[:, 0] == i]
            xywh = t[:, 2:6].clone()
            xywh[:, [0, 2]] *= S; xywh[:, [1, 3]] *= S
            xyxy = torch.zeros_like(xywh)
            xyxy[:, 0] = xywh[:, 0] - xywh[:, 2] / 2; xyxy[:, 1] = xywh[:, 1] - xywh[:, 3] / 2
            xyxy[:, 2] = xywh[:, 0] + xywh[:, 2] / 2; xyxy[:, 3] = xywh[:, 1] + xywh[:, 3] / 2
            gb.append(xyxy.numpy()); gc.append(t[:, 1].long().numpy())
    assert sum(len(p) for p in pb) > 0
    assert got == MR.compute_map(pb, ps, pc, gb, gc, nc)
