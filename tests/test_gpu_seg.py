"""GPU tests of instance segmentation: gelan-c-seg's forward (prototype branch, mask towers, K6 with mask coefficients)
and K15 (masks from the kept detections).

  * fp32 engine: y, mc and proto against the oracle's fp64 forward, within smoke()'s oracle gate;
  * bf16 and fp16: every launch of the seg plan teacher-forced per element (tests/teacher_force.py) at 64 x 640² and
    64 x 384 x 640; y and the raw maps bit-identical to gelan-c's plan with the same weights; mc bit-identical to a
    gather of the mask-tower outputs;
  * K15 against the numpy restatement (oracle/seg_ref.py) in each mode, outside the derived band: counts of 0, some and
    max_det, boxes outside the image and degenerate ones, multi-label rows sharing an anchor, native mode with mixed
    frame sizes from fused-scale NMS; rows at or after counts[b] and guard bytes around the planes keep their 0xAB fill;
  * batch capacity, shape arenas filled with NaN before each shape's first run and CUDA-graph replay reproduce eager
    full runs bit for bit; augment=True raises."""
import ctypes

import numpy as np
import pytest
import torch

from bench_data import make_inputs
from oracle import gelan_ref as G
from oracle import seg_ref as S
from tests import teacher_force as TF
from tests.conftest import ROOT

from yolo_b200 import YOLO, _lib as L, masks_raw, nms_raw, process_mask, process_mask_native
from yolo_b200 import engine as E

pytestmark = pytest.mark.gpu
DEV = "cuda"
SEG = ROOT / "configs/models/gelan-c-seg.yaml"


@pytest.fixture(scope="module")
def seg_sd():
    nodes, nc, nm, npr = S.load_graph(SEG)
    return nodes, nc, S.calibrated_state_dict(nodes, nc, nm, npr)


def _x(Bn, H, W, seed):
    """seeded bench images cropped to H x W"""
    return make_inputs(Bn, max(H, W), seed=seed)[:, :, :H, :W].contiguous().to(DEV)


def _model(sd, prec, cfg=SEG, strict=True):
    m = YOLO.from_yaml(cfg)
    keys = set(m.state_dict())
    m.load_state_dict({k: v for k, v in sd.items() if k in keys}, strict=strict)
    return m.to(DEV).eval().set_precision(prec)


def test_fp32_engine_against_the_oracle(seg_sd):
    nodes, nc, sd = seg_sd
    x = G.fractal(2, 128, torch.Generator().manual_seed(11))
    y32, (_, mc32, p32) = S.forward(nodes, nc, sd, x)
    y64, (_, mc64, p64) = S.forward(nodes, nc, {k: (v.double() if v.is_floating_point() else v) for k, v in sd.items()}, x.double())
    m = _model(sd, "fp32")
    y, (raws, mc, proto) = m(x.to(DEV))
    torch.cuda.synchronize()
    assert tuple(mc.shape) == (2, 32, y.shape[2]) and tuple(proto.shape) == (2, 32, 32, 32)
    for got, ref32, ref64, scale in ((y[:, :4], y32[:, :4], y64[:, :4], 128), (y[:, 4:], y32[:, 4:], y64[:, 4:], 1),
                                     (mc, mc32, mc64, 1), (proto, p32, p64, 1)):
        floor = (ref32 - ref64).abs().max().item()
        d = (got.cpu().double() - ref64).abs().max().item()
        assert d <= max(1e-4 * scale, 3 * floor), (d, floor)
    assert mc64.std() > 0.3 and 0.05 < (p64 > 0.1).double().mean() < 0.95       # the calibration gives live masks


@pytest.mark.parametrize("shape", [(64, 640, 640), (64, 384, 640)])
@pytest.mark.parametrize("prec", ["bf16", "fp16"])
def test_every_new_launch_teacher_forced_and_detection_bit_identical(seg_sd, shape, prec):
    _, _, sd = seg_sd
    Bn, H, W = shape
    x = _x(Bn, H, W, 5)
    seg, det = _model(sd, prec), _model(sd, prec, ROOT / "configs/models/gelan-c.yaml")
    with torch.cuda.device(x.device):
        p = E.compile_model(seg, x)
        names = [n for n, _ in p.op_table()]
        assert "conv_ffma" not in names and names[-1] == "dfl_decode_masks"
        worst = TF.teacher_force(p, label=f"seg {prec} ")
        TF.run_reproduces(p)
        print(f"seg {prec} {shape}: {TF.report(worst)}")
        # mc is the gather of the mask towers' outputs at every anchor, bit for bit
        a = p.trace[-1][1]
        ref = torch.cat([v.t.reshape(Bn, -1, 32) for v in a["masks"]], 1)
        assert torch.equal(a["mc"], ref)
        # y and the raw maps are those of gelan-c's plan with the same weights
        seg.fresh_outputs = det.fresh_outputs = True
        ys, (rs, _, _) = seg(x)
        yd, rd = det(x)
        torch.cuda.synchronize()
        assert torch.equal(ys, yd) and all(torch.equal(u, v) for u, v in zip(rs, rd))


# ---- K15 against its restatement --------------------------------------------------------------------------------------------
G0 = 4096          # guard bytes either side of the masks


def _k15(proto, mc, out, counts, keep, mode, in_hw=(0, 0), scale=None, out_hw=None):
    """K15 through the C ABI into a buffer with 0xAB guards: (masks uint8 [B, max_det, oh, ow], the whole buffer)"""
    Bn, mh, mw, nm = proto.shape
    max_det = out.shape[1]
    oh, ow = out_hw
    n = Bn * max_det * oh * ow
    buf = torch.full((n + 2 * G0,), 0xAB, dtype=torch.uint8, device=DEV)
    masks = buf[G0:G0 + n].view(Bn, max_det, oh, ow)
    d = L.MaskDesc(proto.data_ptr(), Bn, Bn, mh, mw, nm, nm, mc.data_ptr(), mc.shape[1], out.data_ptr(), counts.data_ptr(),
                   keep.data_ptr(), max_det, S_MODES[mode], in_hw[0], in_hw[1], scale.data_ptr() if scale is not None else None,
                   masks.data_ptr(), oh, ow)
    L.check(L.lib().yre_seg_masks(ctypes.byref(d), torch.cuda.current_stream().cuda_stream), "seg_masks")
    torch.cuda.synchronize()
    return masks.cpu(), buf.cpu()


S_MODES = {"proto": L.MASK_PROTO, "input": L.MASK_INPUT, "native": L.MASK_NATIVE}


def _check(masks, buf, proto, mc, out, counts, keep, mode, shapes, frames=None):
    """every written row against the restatement outside the band; untouched bytes keep 0xAB"""
    assert (buf[:G0] == 0xAB).all() and (buf[-G0:] == 0xAB).all()
    pn, mcn, on, kn = proto.cpu().numpy(), mc.cpu().numpy(), out.cpu().numpy(), keep.cpu().numpy()
    inside = total = 0
    for b in range(masks.shape[0]):
        c = int(counts[b])
        assert (masks[b, c:] == 0xAB).all(), "a row at or after counts[b] was written"
        if c == 0:
            continue
        got = masks[b, :c].numpy()
        shape = shapes if frames is None else frames[b]
        if frames is not None:
            h0, w0 = frames[b]
            assert (got[:, h0:] == 0xAB).all() and (got[:, :, w0:] == 0xAB).all(), "bytes outside the native window"
            got = got[:, :h0, :w0]
        assert set(np.unique(got)) <= {0, 1}
        coef = mcn[b, kn[b, :c]]
        probs = S.k15_probs(pn[b], coef, on[b, :c, :4], mode, shape)
        band = S.k15_band(pn[b], coef, mode, shape)
        out_band = np.abs(probs.astype(np.float64) - 0.5) > band
        bad = out_band & ((probs > 0.5) != (got == 1))
        assert not bad.any(), f"image {b}: {bad.sum()} pixels differ outside the band"
        inside += (~out_band).sum()
        total += got.size
    assert inside <= 1e-3 * max(total, 1)


def _inputs(g, Bn, mh, mw, A, max_det, counts, H, W):
    proto = (torch.rand((Bn, mh, mw, 32), generator=g) * 1.3 - 0.28).to(DEV)
    mc = (torch.randn((Bn, A, 32), generator=g) * 0.6).to(DEV)
    xy = torch.rand((Bn, max_det, 2), generator=g) * torch.tensor([W, H]) * 1.1 - 0.05 * torch.tensor([W, H])
    wh = torch.rand((Bn, max_det, 2), generator=g) * torch.tensor([W, H]) * 0.6
    out = torch.cat([xy, xy + wh, torch.rand((Bn, max_det, 2), generator=g)], 2)
    out[:, 0, :4] = torch.tensor([-30.0, -20.0, W + 40.0, H + 9.0])             # beyond the image
    out[:, 1, :4] = torch.tensor([50.0, 40.0, 50.0, 90.0])                      # degenerate
    out[:, 2, :4] = torch.tensor([W - 3.5, 2.25, W + 1.0, 17.75])               # on the right edge
    keep = torch.randint(0, A, (Bn, max_det), generator=g)
    keep[:, 4] = keep[:, 3]                                                      # rows sharing an anchor (multi-label)
    return proto, mc, out.to(DEV), torch.tensor(counts, dtype=torch.int32, device=DEV), keep.to(DEV)


@pytest.mark.parametrize("mode, H, W", [("proto", 640, 640), ("input", 640, 640), ("input", 384, 640), ("proto", 96, 160)])
def test_k15_against_the_restatement(mode, H, W):
    g = torch.Generator().manual_seed(H + W + len(mode))
    mh, mw, max_det = H // 4, W // 4, 24
    counts = [0, 7, max_det, 13]
    proto, mc, out, cnt, keep = _inputs(g, 4, mh, mw, 500, max_det, counts, H, W)
    oh, ow = (mh, mw) if mode == "proto" else (H, W)
    masks, buf = _k15(proto, mc, out, cnt, keep, mode, (H, W), out_hw=(oh, ow))
    _check(masks, buf, proto, mc, out, cnt, keep, mode, (H, W))
    # the Python entry point computes the same bytes
    r = masks_raw(proto.permute(0, 3, 1, 2), mc.permute(0, 2, 1), out, cnt, keep, mode, shape=(H, W)).cpu()
    for b, c in enumerate(counts):
        assert torch.equal(r[b, :c], masks[b, :c].bool())


def test_k15_native_with_mixed_frames():
    g = torch.Generator().manual_seed(3)
    frames = [(480, 640), (1080, 1920), (500, 375), (37, 53), (480, 720)]
    max_det, mh, mw = 16, 160, 160
    counts = [16, 5, 9, 16, 11]
    oh, ow = max(f[0] for f in frames), max(f[1] for f in frames)
    proto, mc, out, cnt, keep = _inputs(g, len(frames), mh, mw, 400, max_det, counts, 640, 640)
    scale = torch.tensor([[0.0, 0.0, 1.0, w, h] for h, w in frames], dtype=torch.float32, device=DEV)
    for b, (h, w) in enumerate(frames):                                      # boxes in frame pixels
        out[b, :, :4] *= torch.tensor([w / 640, h / 640, w / 640, h / 640], device=DEV)
    masks, buf = _k15(proto, mc, out, cnt, keep, "native", scale=scale, out_hw=(oh, ow))
    _check(masks, buf, proto, mc, out, cnt, keep, "native", None, frames)
    r = masks_raw(proto.permute(0, 3, 1, 2), mc.permute(0, 2, 1), out, cnt, keep, "native", scale=scale).cpu()
    assert tuple(r.shape[2:]) == (oh, ow)
    for b, ((h, w), c) in enumerate(zip(frames, counts)):
        assert torch.equal(r[b, :c, :h, :w], masks[b, :c, :h, :w].bool())


def test_per_image_functions_match_upstream_outside_the_band():
    g = torch.Generator().manual_seed(9)
    protos = torch.rand((32, 96, 160), generator=g) * 1.3 - 0.28
    mc = torch.randn((6, 32), generator=g) * 0.6
    boxes = torch.tensor([[10.0, 20.0, 300.0, 200.0], [-5.0, -5.0, 700.0, 400.0], [100.5, 50.25, 100.5, 80.0],
                          [600.0, 300.0, 640.0, 384.0], [0.0, 0.0, 33.3, 44.4], [200.0, 100.0, 520.0, 370.0]])
    ph, mcn = protos.permute(1, 2, 0).numpy(), mc.numpy()
    for up in (False, True):
        got = process_mask(protos.to(DEV), mc.to(DEV), boxes.to(DEV), (384, 640), upsample=up).cpu().numpy()
        ref = S.process_mask_probs(protos, mc, boxes, (384, 640), up).double().numpy()
        band = S.k15_band(ph, mcn, "input" if up else "proto", (384, 640))
        assert got.dtype == np.bool_ and not (((ref > 0.5) != got) & (np.abs(ref - 0.5) > band)).any()
    for frame in ((480, 720), (500, 375)):          # 375: an odd width, so every store is a byte store
        fb = boxes * torch.tensor([frame[1] / 640, frame[0] / 384] * 2)
        got = process_mask_native(protos.to(DEV), mc.to(DEV), fb.to(DEV), frame).cpu().numpy()
        ref = S.process_mask_native_probs(protos, mc, fb, frame).double().numpy()
        band = S.k15_band(ph, mcn, "native", frame)
        assert got.shape == (6,) + frame and not (((ref > 0.5) != got) & (np.abs(ref - 0.5) > band)).any()
    assert process_mask(protos.to(DEV), mc[:0].to(DEV), boxes[:0].to(DEV), (384, 640), True).shape == (0, 384, 640)


def test_end_to_end_multi_label_masks(seg_sd):
    """forward -> multi-label NMS -> K15: rows sharing an anchor take the same coefficients"""
    _, _, sd = seg_sd
    m = _model(sd, "bf16")
    x = make_inputs(4, 640, seed=2).to(DEV)
    y, (_, mc, proto) = m(x)
    out, counts, keep = nms_raw(y.permute(0, 2, 1), 0.001, 0.7, max_det=300, multi_label=True)
    masks, buf = _k15(proto.permute(0, 2, 3, 1).contiguous(), mc.permute(0, 2, 1).contiguous(), out, counts, keep, "proto",
                      (640, 640), out_hw=(160, 160))
    k = keep.cpu()
    assert any(len(set(k[b, :int(counts[b])].tolist())) < int(counts[b]) for b in range(4)), "no shared anchors"
    _check(masks, buf, proto.permute(0, 2, 3, 1).contiguous(), mc.permute(0, 2, 1).contiguous(), out, counts, keep, "proto",
           (640, 640))


def test_end_to_end_native_masks_from_fused_scale_nms(seg_sd):
    """frames letterboxed into 640², NMS with the scale rows (boxes in frame pixels) -> K15 native mode.  The largest
    frame is 500 x 375: planes of an odd width and at odd offsets take the byte-store and unaligned zero-fill paths."""
    _, _, sd = seg_sd
    m = _model(sd, "bf16")
    frames = [(500, 375), (281, 375), (375, 333), (375, 375)]
    rows = []
    for h, w in frames:
        gain = min(640 / h, 640 / w)
        rows.append([(640 - w * gain) / 2, (640 - h * gain) / 2, gain, w, h])
    scale = torch.tensor(rows, dtype=torch.float32, device=DEV)
    x = make_inputs(len(frames), 640, seed=4).to(DEV)
    y, (_, mc, proto) = m(x)
    out, counts, keep = nms_raw(y.permute(0, 2, 1), 0.25, 0.45, max_det=64, scale=scale)
    assert int(counts.min()) > 0
    p_hwc, m_an = proto.permute(0, 2, 3, 1).contiguous(), mc.permute(0, 2, 1).contiguous()
    masks, buf = _k15(p_hwc, m_an, out, counts, keep, "native", scale=scale, out_hw=(500, 375))
    _check(masks, buf, p_hwc, m_an, out, counts, keep, "native", None, frames)
    r = masks_raw(proto, mc, out, counts, keep, "native", scale=scale).cpu()      # shape read from scale
    assert tuple(r.shape[2:]) == (500, 375)
    for b, ((h, w), c) in enumerate(zip(frames, counts.tolist())):
        assert torch.equal(r[b, :c, :h, :w], masks[b, :c, :h, :w].bool())
        assert masks[b, :c].sum() > 0


# ---- engine modes -------------------------------------------------------------------------------------------------------------
def _flat(o):
    y, (raws, mc, proto) = o
    return [y, mc, proto, *raws]


def test_capacity_arena_and_graph_replay_reproduce_eager_runs(seg_sd):
    _, _, sd = seg_sd
    xs = {(H, W): _x(16, H, W, H + W) for H, W in ((640, 640), (384, 640), (256, 320))}
    m = _model(sd, "bf16")
    ref = {k: [t.clone() for t in _flat(m(x))] for k, x in xs.items()}         # eager full runs of 16 images
    torch.cuda.synchronize()

    m.max_batch = 16                                             # batch capacity: the first 7 images of the full run
    for k, x in xs.items():
        got = _flat(m(x[:7]))
        assert all(torch.equal(a, b[:7]) for a, b in zip(got, ref[k])), k
    m.max_shape = (640, 640)                                    # shape arena, NaN-filled before each shape's first run
    E._arena(m, xs[640, 640], 16, None, None, (640, 640))       # allocated now, so that the first run reads NaN too
    assert len(m._arenas) == 1
    for k, x in xs.items():
        for arena in m._arenas.values():
            arena.fill_(0xFF)
        got = _flat(m(x))
        assert all(torch.equal(a, b) for a, b in zip(got, ref[k])), k
    assert len(m._arenas) == 1                                  # every shape ran on the arena that was filled
    m.fresh_outputs, m.use_cuda_graph = False, True             # CUDA-graph replay on static outputs
    for _ in range(2):
        for k, x in xs.items():
            got = _flat(m(x))
            assert all(torch.equal(a, b) for a, b in zip(got, ref[k])), k
    with pytest.raises(ValueError, match="segmentation"):
        m(xs[640, 640], augment=True)
