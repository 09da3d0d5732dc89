"""K14 on the GPU: 4:2:0 YUV frames (NV12, NV21, I420, YV12; BT.601 and BT.709) letterboxed bit-exactly as K8 letterboxes
the oracle's conversion, which is pinned to cv2.cvtColor on every (Y, U, V) triple (tests/test_cpu_yuv.py).  Covers both
output modes, every resize mode (bilinear up and down, exact 2x area, copy), a 2 x 2 frame, a two-launch mixed-size
batch, pitched planes in separate allocations, guard bands around `out`, and detections end to end against the BGR
path on the same frames."""
import numpy as np
import pytest
import torch

from oracle import gelan_ref as G
from oracle import yuv_ref as Y
from tests.conftest import ROOT
from tests.test_cpu_rect import letterbox_rect, rect_geometry

pytestmark = pytest.mark.gpu

from yolo_b200 import YOLO, letterbox, non_max_suppression_async, preprocess, scale_rows

DEV = "cuda"
MATRICES = ("bt601", "bt709")


def yuv_frame(h, w, fmt, seed):
    """cv2-layout (h * 3/2) x w frame of random planes"""
    rng = np.random.default_rng(seed)
    y = rng.integers(0, 256, (h, w), dtype=np.uint8)
    u, v = (rng.integers(0, 256, (h // 2, w // 2), dtype=np.uint8) for _ in range(2))
    return Y.to_frame(y, u, v, fmt)


def _chw(lb: np.ndarray) -> np.ndarray:
    return np.ascontiguousarray(lb[:, :, ::-1].transpose(2, 0, 1)).astype(np.float32) / np.float32(255.0)


# (h, w, new_shape, auto): bilinear down (square and auto rect), bilinear up, exact 2x area, copy, a 2 x 2 frame
GEOMETRIES = [(1080, 1920, 640, False), (1080, 1920, 640, True), (240, 320, 640, False), (1280, 1280, 640, False),
              (384, 640, 640, True), (2, 2, 64, False)]


@pytest.mark.parametrize("matrix", MATRICES)
@pytest.mark.parametrize("fmt", Y.FORMATS)
@pytest.mark.parametrize("h,w,S,auto", GEOMETRIES)
def test_k14_equals_k8_on_the_converted_frame(h, w, S, auto, fmt, matrix):
    frame = yuv_frame(h, w, fmt, h * w + len(fmt))
    ref, ref_ratio, ref_pad = letterbox_rect(Y.yuv420_to_bgr(frame, fmt, matrix), S, S, 32 if auto else 0)
    lb, ratio, pad = letterbox(frame, S, auto=auto, fmt=fmt, yuv_matrix=matrix)      # numpy in, numpy out
    assert isinstance(lb, np.ndarray) and lb.shape == ref.shape and np.array_equal(lb, ref)
    assert ratio == ref_ratio and pad == ref_pad
    dev = torch.from_numpy(frame).to(DEV)
    x, ratios, pads = preprocess(dev, S, auto=auto, fmt=fmt, yuv_matrix=matrix)
    assert ratios == [ref_ratio] and pads == [ref_pad]
    assert np.array_equal(x[0].cpu().numpy(), _chw(ref))
    xu, _, _ = preprocess(dev, S, auto=auto, fmt=fmt, yuv_matrix=matrix, dtype=torch.uint8)
    assert np.array_equal(xu[0].cpu().numpy(), ref)


@pytest.mark.parametrize("dtype", [torch.float32, torch.uint8])
@pytest.mark.parametrize("fmt", Y.FORMATS)
def test_mixed_size_batch_of_40_frames(fmt, dtype):
    """two launches (32 + 8); every frame letterboxed into the batch's shared rectangle as the BGR path does it"""
    rng = np.random.default_rng(40)
    sizes = [(2 * int(h), 2 * int(w)) for h, w in rng.integers(20, 450, (38, 2))] + [(1080, 1920), (300, 302)]
    frames = [yuv_frame(h, w, fmt, i) for i, (h, w) in enumerate(sizes)]
    matrix = "bt709" if fmt in ("nv21", "yv12") else "bt601"
    x, ratios, pads = preprocess(frames, 320, dtype=dtype, auto=True, fmt=fmt, yuv_matrix=matrix)
    bgr = [Y.yuv420_to_bgr(f, fmt, matrix) for f in frames]
    xr, ratios_r, pads_r = preprocess(bgr, 320, dtype=dtype, auto=True)
    assert x.shape == xr.shape and torch.equal(x, xr) and ratios == ratios_r and pads == pads_r
    own = [rect_geometry(h, w, 320, 320, 32) for h, w in sizes]
    H, W = max(g[4] for g in own), max(g[5] for g in own)
    got = x.cpu().numpy()
    for i in (0, 38, 39):
        stride = 32 if own[i][4:6] == (H, W) else 0
        ref, _, _ = letterbox_rect(bgr[i], *((320, 320) if stride else (H, W)), stride)
        assert np.array_equal(got[i], _chw(ref) if dtype == torch.float32 else ref), i


def _pitched(a: np.ndarray, pitch: int) -> torch.Tensor:
    """a copied into its own device allocation with rows `pitch` bytes apart; the padding bytes are 0xFF"""
    buf = torch.full((a.shape[0], pitch), 0xFF, dtype=torch.uint8, device=DEV)
    buf[:, :a.shape[1]] = torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    return buf[:, :a.shape[1]]


@pytest.mark.parametrize("matrix", MATRICES)
@pytest.mark.parametrize("fmt", Y.FORMATS)
def test_pitched_planes_in_separate_allocations(fmt, matrix):
    """decoder surfaces: every plane in its own allocation with a pitch above its row, the pitch padding 0xFF; and
    for NV12 / NV21 one pitched (h * 3/2) x w surface"""
    h, w = 720, 1280
    frame = yuv_frame(h, w, fmt, 77)
    yp, up, vp = Y.split_planes(frame, fmt)
    nv = fmt in ("nv12", "nv21")
    if nv:
        planes = (_pitched(yp, 1536), _pitched(frame[h:], 1408))
    else:
        planes = (_pitched(yp, 1536), _pitched(up, 768), _pitched(vp, 768))
    assert planes[0].stride(0) == 1536 and planes[1].stride(0) > planes[1].shape[1]
    ref, _, _ = letterbox_rect(Y.yuv420_to_bgr(frame, fmt, matrix), 640, 640, 32)
    for dtype in (torch.float32, torch.uint8):
        x, _, _ = preprocess(planes, 640, dtype=dtype, auto=True, fmt=fmt, yuv_matrix=matrix)
        assert np.array_equal(x[0].cpu().numpy(), _chw(ref) if dtype == torch.float32 else ref)
    lb, _, _ = letterbox(planes, 640, auto=True, fmt=fmt, yuv_matrix=matrix)
    assert lb.is_cuda and np.array_equal(lb.cpu().numpy(), ref)
    if nv:
        surface = _pitched(frame, 2048)
        lb, _, _ = letterbox(surface, 640, auto=True, fmt=fmt, yuv_matrix=matrix)
        assert np.array_equal(lb.cpu().numpy(), ref)
    # the output does not change when the padding changes from 0xFF to 0x00
    x1, _, _ = preprocess(planes, 640, dtype=torch.uint8, auto=True, fmt=fmt, yuv_matrix=matrix)
    for p in planes:
        p.as_strided((p.shape[0], p.stride(0) - p.shape[1]), (p.stride(0), 1), p.storage_offset() + p.shape[1]).fill_(0)
    x0, _, _ = preprocess(planes, 640, dtype=torch.uint8, auto=True, fmt=fmt, yuv_matrix=matrix)
    assert torch.equal(x0, x1)


@pytest.mark.parametrize("dtype", [torch.float32, torch.uint8])
def test_guard_bands_around_out_stay_untouched(dtype):
    frames = [yuv_frame(1080, 1920, "nv12", s) for s in (1, 2, 3)]
    shape = (3, 3, 384, 640) if dtype == torch.float32 else (3, 384, 640, 3)
    n, g = int(np.prod(shape)), 4096
    buf = torch.full((n + 2 * g,), 77, dtype=dtype, device=DEV)
    out = buf[g:g + n].view(shape)
    x, _, _ = preprocess(frames, 640, out=out, dtype=dtype, auto=True, fmt="nv12")
    assert x.data_ptr() == out.data_ptr()
    assert bool((buf[:g] == 77).all()) and bool((buf[g + n:] == 77).all())
    ref, _, _ = preprocess([Y.yuv420_to_bgr(f, "nv12") for f in frames], 640, dtype=dtype, auto=True)
    assert torch.equal(out, ref)


def test_rejections_reach_python():
    with pytest.raises(ValueError):
        preprocess(np.zeros((7, 4), np.uint8), 64, fmt="nv12")                    # not (h * 3/2) x w
    with pytest.raises(Exception, match="even"):
        preprocess(np.zeros((6, 5), np.uint8), 64, fmt="nv12")                    # odd width
    f = torch.zeros((6, 8), dtype=torch.uint8, device=DEV)
    with pytest.raises(ValueError, match="contiguous"):
        preprocess(torch.zeros((6, 16), dtype=torch.uint8, device=DEV)[:, :8], 64, fmt="i420")
    with pytest.raises(ValueError):
        preprocess((f[:4], f[:2, :2]), 64, fmt="i420")                           # (y, u) without v
    with pytest.raises(ValueError):
        preprocess((f[:4], f[:2, :4]), 64, fmt="nv12", yuv_matrix="bt2020")


# ---- end to end ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("arena", [False, True])
def test_nv12_detections_equal_the_bgr_path(gelan_c, arena):
    """preprocess(nv12, dtype=uint8, auto=True) -> model -> non_max_suppression_async(scale=...) gives the detections of
    the same frames converted on the host and fed through the BGR path (bf16; with and without max_batch/max_shape)"""
    nodes, nc, sd = gelan_c
    x = G.fractal(4, 1080, torch.Generator().manual_seed(31), w=1920)
    frames = [Y.to_frame(*Y.encode_bt601((f.permute(1, 2, 0).flip(-1) * 255).round().clamp(0, 255).to(torch.uint8).numpy()),
                         "nv12") for f in x]
    bgr = [Y.yuv420_to_bgr(f, "nv12") for f in frames]
    try:
        import cv2
        assert all(np.array_equal(b, cv2.cvtColor(f, cv2.COLOR_YUV2BGR_NV12)) for b, f in zip(bgr, frames))
    except ImportError:
        pass
    m = YOLO.from_yaml(ROOT / "configs/models/gelan-c.yaml")
    m.load_state_dict(sd, strict=True)
    m = m.to(DEV).eval().set_precision("bf16")
    if arena:
        m.max_batch, m.max_shape = 8, (640, 640)
    origs = [(1080, 1920)] * 4
    runs = []
    for src, fmt in ((frames, "nv12"), (bgr, "bgr")):
        xu, ratios, pads = preprocess(src, 640, dtype=torch.uint8, auto=True, fmt=fmt)
        assert tuple(xu.shape) == (4, 384, 640, 3)
        y, _ = m(xu)
        pred = y.permute(0, 2, 1).contiguous()
        dets = non_max_suppression_async(pred, 0.25, 0.45, scale=scale_rows(ratios, pads, origs, device=DEV)).result()
        runs.append((xu, [d.clone() for d in dets]))
    (xa, da), (xb, db) = runs
    assert torch.equal(xa, xb)
    assert sum(len(d) for d in da) > 0
    for a, b in zip(da, db):
        assert torch.equal(a, b)
