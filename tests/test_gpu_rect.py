"""Rectangular ("rect") inference on the GPU: the letterbox kernel writing an out_h x out_w destination, the whole path at
non-square sizes against the oracle, every launch of non-square full-size plans teacher-forced, and the path identities
(uint8 frames, fused box scaling, CUDA graphs, batch order) off the diagonal."""
import time

import numpy as np
import pytest
import torch

from oracle import gelan_ref as G
from oracle import nms_ref as N
from oracle import preproc_ref as P
from tests import teacher_force as TF
from tests.conftest import ROOT
from tests.test_cpu_conv_tc_select import tc_variant
from tests.test_cpu_rect import letterbox_rect, rect_geometry

pytestmark = pytest.mark.gpu

import yolo_b200
from yolo_b200 import YOLO, letterbox, nms_raw, preprocess, scale_boxes, scale_rows
from yolo_b200 import engine as E

DEV = "cuda"


def _image(h, w, seed):
    return np.random.default_rng(seed).integers(0, 256, (h, w, 3), dtype=np.uint8)


def _chw(lb: np.ndarray) -> np.ndarray:
    return np.ascontiguousarray(lb[:, :, ::-1].transpose(2, 0, 1)).astype(np.float32) / np.float32(255.0)


# ---- K8: letterbox to a rectangle ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("h,w,new_shape,auto,stride", [(1080, 1920, 640, True, 32), (1920, 1080, 640, True, 32),
                                                       (480, 640, 640, True, 64), (333, 517, (384, 640), False, 32),
                                                       (100, 37, (200, 96), False, 32), (360, 640, 640, True, 32),
                                                       (25, 41, (320, 192), True, 32), (1, 1, (64, 32), False, 32)])
def test_letterbox_to_a_rectangle_is_bit_exact(h, w, new_shape, auto, stride):
    img = _image(h, w, h * w)
    nh_, nw_ = (new_shape, new_shape) if isinstance(new_shape, int) else new_shape
    ref, ref_ratio, ref_pad = letterbox_rect(img, nh_, nw_, stride if auto else 0)
    lb, ratio, pad = letterbox(img, new_shape, auto=auto, stride=stride)
    assert lb.shape == ref.shape and np.array_equal(lb, ref)
    assert ratio == ref_ratio and pad == ref_pad
    x, ratios, pads = preprocess(img, new_shape, auto=auto, stride=stride)
    assert ratios == [ref_ratio] and pads == [ref_pad]
    assert np.array_equal(x[0].cpu().numpy(), _chw(ref))


@pytest.mark.parametrize("dtype", [torch.float32, torch.uint8])
def test_mixed_size_batch_into_one_rectangle(dtype):
    """40 images of different sizes and orientations (two launches of 32 + 8) share one rectangle: the per-axis maximum
    of their own smallest stride-32 rectangles; an image whose rectangle is smaller is letterboxed into the shared one."""
    rng = np.random.default_rng(9)
    sizes = [(int(h), int(w)) for h, w in rng.integers(40, 900, (38, 2))] + [(1080, 1920), (300, 301)]
    imgs = [_image(h, w, i) for i, (h, w) in enumerate(sizes)]
    own = [rect_geometry(h, w, 320, 320, 32) for h, w in sizes]
    H, W = max(g[4] for g in own), max(g[5] for g in own)
    x, ratios, pads = preprocess(imgs, 320, dtype=dtype, auto=True)
    assert tuple(x.shape) == ((40, 3, H, W) if dtype == torch.float32 else (40, H, W, 3))
    got = x.cpu().numpy()
    for i, img in enumerate(imgs):
        stride = 32 if own[i][4:6] == (H, W) else 0
        ref, r, pad = letterbox_rect(img, *((320, 320) if stride else (H, W)), stride)
        assert ref.shape[:2] == (H, W)
        assert (ratios[i], pads[i]) == (r, pad), i
        assert np.array_equal(got[i], _chw(ref) if dtype == torch.float32 else ref), i
    # on the device, the batch equals the images letterboxed one by one
    xd, _, _ = preprocess([torch.from_numpy(i).to(DEV) for i in imgs], 320, dtype=dtype, auto=True)
    assert torch.equal(xd, x)


def test_square_letterbox_is_unchanged():
    """auto=False with an int, and the (S, S) pair, give today's square output: the oracle, which is pinned to the
    reference's own letterbox."""
    imgs = [_image(h, w, h) for h, w in ((480, 640), (333, 500), (640, 480), (1280, 1280), (17, 901))]
    x, ratios, pads = preprocess(imgs, 640)
    x2, ratios2, pads2 = preprocess(imgs, (640, 640))
    assert torch.equal(x, x2) and ratios == ratios2 and pads == pads2
    for i, img in enumerate(imgs):
        ref, r, pad = P.preprocess(img, 640)
        assert np.array_equal(x[i].cpu().numpy(), ref) and ratios[i] == r and pads[i] == pad
        lb, r1, p1 = letterbox(img, 640)
        assert np.array_equal(lb, P.letterbox(img, 640)[0]) and (r1, p1) == (r, pad)


# ---- whole path at non-square sizes against the oracle ---------------------------------------------------------------------
def _model(name, sd, prec):
    m = YOLO.from_yaml(ROOT / "configs/models" / f"{name}.yaml")
    m.load_state_dict(sd, strict=True)
    return m.to(DEV).eval().set_precision(prec)


@pytest.mark.parametrize("H,W,batch", [(192, 320, 2), (320, 192, 1), (224, 416, 1)])
def test_fp32_end_to_end_vs_oracle_and_nms_non_square(gelan_c, H, W, batch):
    """the gates of test_fp32_end_to_end_vs_oracle_and_nms with max(H, W) as the size; 224x416 has odd ADown outputs
    (7x13 at stride 32)"""
    nodes, nc, sd = gelan_c
    x = G.fractal(batch, H, torch.Generator().manual_seed(H + W), w=W)
    y_ref, _ = G.forward(nodes, nc, sd, x)
    sd64 = {k: (v.double() if v.is_floating_point() else v) for k, v in sd.items()}
    y64, _ = G.forward(nodes, nc, sd64, x.double())
    floor_box = (y_ref[:, :4].double() - y64[:, :4]).abs().max().item()
    floor_sc = (y_ref[:, 4:].double() - y64[:, 4:]).abs().max().item()
    y, raws = _model("gelan-c", sd, "fp32")(x.to(DEV))
    A = sum((H // s) * (W // s) for s in (8, 16, 32))
    assert y.shape == (batch, 84, A) and [tuple(r.shape) for r in raws] == [(batch, 144, H // s, W // s) for s in (8, 16, 32)]
    dbox = (y[:, :4].cpu().double() - y64[:, :4]).abs().max().item()
    dsc = (y[:, 4:].cpu().double() - y64[:, 4:]).abs().max().item()
    print(f"{H}x{W} B{batch}: ours-vs-fp64 |dbox|={dbox:.3e}px |dscore|={dsc:.3e}; reference floor {floor_box:.3e}px {floor_sc:.3e}")
    assert dbox <= max(1e-4 * max(H, W), 3 * floor_box) and dsc <= max(1e-4, 3 * floor_sc)
    pred = y.permute(0, 2, 1).contiguous()
    dets = yolo_b200.non_max_suppression(pred, 0.25, 0.45)
    ref = N.non_max_suppression(pred.cpu(), 0.25, 0.45)
    for a, b in zip(dets, ref):
        assert np.array_equal(a.cpu().numpy(), b)


# ---- every launch of non-square full-size plans, teacher-forced per element (tests/teacher_force.py) ------------------------
def _rect_inputs(Bn, H, W, seed):
    """eight distinct multi-octave images repeated with a brightness ramp (bench_data.make_inputs, non-square)"""
    base = G.fractal(min(Bn, 8), H, torch.Generator().manual_seed(seed), w=W)
    x = base.repeat(-(-Bn // base.shape[0]), 1, 1, 1)[:Bn].clone()
    return x * torch.linspace(0.85, 1.0, Bn).view(-1, 1, 1, 1)


@pytest.mark.parametrize("prec", ["bf16", "fp16"])
@pytest.mark.parametrize("name,Bn,H,W", [("gelan-c", 64, 384, 640), ("yolov9-c", 16, 384, 640)])
def test_every_launch_of_a_non_square_plan_teacher_forced(name, Bn, H, W, prec, request):
    nodes, nc, sd = request.getfixturevalue("gelan_c" if name == "gelan-c" else "yolov9_c")
    model = _model(name, sd, prec)
    x = _rect_inputs(Bn, H, W, seed=7).to(DEV)
    sms = torch.cuda.get_device_properties(x.device).multi_processor_count
    with torch.cuda.device(x.device):
        p = E.compile_model(model, x)
        names, variants = [n for n, _ in p.op_table()], p.op_variants()
        assert "conv_ffma" not in names
        for i, (kind, a) in enumerate(p.trace):
            if kind == "conv":
                assert tc_variant(a, sms) == variants[i], (i, p.op_descriptions()[i])
        t0 = time.perf_counter()
        worst = TF.teacher_force(p, label=f"{name} {prec} {Bn}x{H}x{W} ")
        t1 = time.perf_counter()
        TF.run_reproduces(p)
        print(f"{name} {prec} {Bn}x{H}x{W}: {len(names)} launches checked per element in {t1 - t0:.1f} s, worst err / bound "
              f"per kernel family: {TF.report(worst)}; the back-to-back run reproduces every buffer")


# ---- path identities --------------------------------------------------------------------------------------------------------
def _frames(n, h, w, seed):
    x = G.fractal(n, h, torch.Generator().manual_seed(seed), w=w)
    return [(f.permute(1, 2, 0).flip(-1) * 255.0).round().clamp(0, 255).to(torch.uint8).contiguous().numpy() for f in x]


@pytest.mark.parametrize("prec", ["bf16", "fp16"])
def test_rect_path_identities(gelan_c, prec):
    """1080x1920 frames letterboxed to 640x384 (auto): uint8 frames through the fused stem == the fp32 tensor path;
    NMS with fused scale rows == scale_boxes afterwards; CUDA-graph replay == eager; a batch permutation permutes y."""
    nodes, nc, sd = gelan_c
    frames = _frames(6, 1080, 1920, 21)
    xu, ratios, pads = preprocess(frames, 640, dtype=torch.uint8, auto=True)
    xf, ratios_f, pads_f = preprocess(frames, 640, auto=True)
    assert tuple(xu.shape) == (6, 384, 640, 3) and ratios == ratios_f and pads == pads_f == [(0, 12)] * 6
    m = _model("gelan-c", sd, prec)
    y_f, raws_f = m(xf)
    y_u, raws_u = m(xu)
    assert y_f.shape == (6, 84, 5040)
    assert torch.equal(y_f, y_u) and all(torch.equal(a, b) for a, b in zip(raws_f, raws_u))
    pred = y_u.permute(0, 2, 1).contiguous()
    origs = [f.shape[:2] for f in frames]
    out0, cnt0, keep0 = nms_raw(pred, 0.25, 0.45)
    out1, cnt1, keep1 = nms_raw(pred, 0.25, 0.45, scale=scale_rows(ratios, pads, origs, device=DEV))
    assert torch.equal(cnt0, cnt1) and int(cnt0.sum()) > 0
    for i in range(6):
        n = int(cnt0[i])
        assert torch.equal(keep0[i, :n], keep1[i, :n])
        ref = out0[i, :n].clone()
        scale_boxes(ref[:, :4], xu.shape[1:3], origs[i], (ratios[i], pads[i]))
        assert torch.equal(ref, out1[i, :n])
        ref2 = out0[i, :n].clone()                         # the reference's own non-square ratio_pad=None formula
        scale_boxes(ref2[:, :4], xu.shape[1:3], origs[i])
        assert torch.equal(ref2, out1[i, :n])
    m.fresh_outputs, m.use_cuda_graph = False, True
    y_g, _ = m(xu)
    y_g2, _ = m(xu)
    assert torch.equal(y_g, y_u) and torch.equal(y_g2, y_u)
    m.fresh_outputs, m.use_cuda_graph = True, False
    perm = torch.tensor([3, 0, 5, 1, 4, 2], device=DEV)
    y_p, raws_p = m(xu[perm].contiguous())
    assert torch.equal(y_p, y_u[perm]) and all(torch.equal(a, b[perm]) for a, b in zip(raws_p, raws_u))


def test_boxes_map_back_to_the_original_frame():
    """a box drawn in a 1080x1920 frame, letterboxed to 384x640 and mapped back by scale_boxes, lands where it was"""
    _, (r, _), pad = letterbox(_image(1080, 1920, 1), 640, auto=True)
    orig = torch.tensor([[100.0, 50.0, 1800.0, 1000.0], [0.0, 0.0, 1920.0, 1080.0]])
    lb = orig * r + torch.tensor([pad[0], pad[1], pad[0], pad[1]], dtype=torch.float32)
    back = scale_boxes(lb.to(DEV).contiguous(), (384, 640), (1080, 1920), ((r, r), pad)).cpu()
    assert (back - orig).abs().max().item() < 1e-3
