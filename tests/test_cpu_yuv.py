"""4:2:0 YUV frame input (K14) without a GPU: the oracle's conversion against cv2.cvtColor on every (Y, U, V) triple,
BT.709 against its float formula, the letterbox of a converted frame against cv2, the plane descriptor's layout against
the C header, and every host-side rejection of yre_letterbox_yuv420_batch (all checked before anything is launched)."""
import ctypes as C
import subprocess

import numpy as np
import pytest

from oracle import preproc_ref as P
from oracle import yuv_ref as Y
from tests.conftest import ROOT

from yolo_b200 import _lib as L
from yolo_b200 import letterbox, preprocess

CV2_FLAG = {"nv12": "COLOR_YUV2BGR_NV12", "nv21": "COLOR_YUV2BGR_NV21", "i420": "COLOR_YUV2BGR_I420", "yv12": "COLOR_YUV2BGR_YV12"}


def exhaustive_frame(f: int):
    """Frame f of 64 (512 x 512 luma): 2 x 2 block b has (U, V) = (b >> 8, b & 255) and lumas 4 f .. 4 f + 3, so the 64
    frames hold each of the 2^24 (Y, U, V) triples exactly once."""
    b = np.arange(256 * 256).reshape(256, 256)
    u, v = (b >> 8).astype(np.uint8), (b & 255).astype(np.uint8)
    y = np.empty((512, 512), np.uint8)
    for k, (dy, dx) in enumerate(((0, 0), (0, 1), (1, 0), (1, 1))):
        y[dy::2, dx::2] = 4 * f + k
    return y, u, v


@pytest.mark.parametrize("fmt", Y.FORMATS)
def test_restatement_equals_cv2_on_every_yuv_triple(fmt):
    cv2 = pytest.importorskip("cv2")
    seen = np.zeros(1 << 24, bool)
    for f in range(64):
        y, u, v = exhaustive_frame(f)
        frame = Y.to_frame(y, u, v, fmt)
        got = Y.yuv420_to_bgr(frame, fmt)
        assert np.array_equal(got, cv2.cvtColor(frame, getattr(cv2, CV2_FLAG[fmt]))), (fmt, f)
        up = lambda c: np.repeat(np.repeat(c, 2, 0), 2, 1).astype(np.int64)
        seen[(y.astype(np.int64) << 16) | (up(u) << 8) | up(v)] = True
    assert seen.all()


@pytest.mark.parametrize("matrix", ["bt601", "bt709"])
def test_fixed_point_stays_within_one_of_the_float_formula(matrix):
    cy, cvr, cvg, cug, cub = Y.FLOAT_COEFFS[matrix]
    worst = 0
    for f in range(64):
        y, u, v = exhaustive_frame(f)
        got = Y.yuv420_to_bgr((y, u, v), "i420", matrix).astype(np.int64)
        up = lambda c: np.repeat(np.repeat(c, 2, 0), 2, 1).astype(np.float64) - 128
        yy, uu, vv = np.maximum(y.astype(np.float64) - 16, 0) * cy, up(u), up(v)
        ref = np.stack([yy + cub * uu, yy + cvg * vv + cug * uu, yy + cvr * vv], -1)
        ref = np.clip(np.floor(ref + 0.5), 0, 255)
        worst = max(worst, int(np.abs(got - ref).max()))
    assert worst <= 1


def test_plane_forms_agree():
    """cv2's single array and the tuple of planes describe the same frame in each format"""
    rng = np.random.default_rng(5)
    y = rng.integers(0, 256, (6, 10), dtype=np.uint8)
    u, v = (rng.integers(0, 256, (3, 5), dtype=np.uint8) for _ in range(2))
    ref = Y.convert(y, np.repeat(np.repeat(u, 2, 0), 2, 1), np.repeat(np.repeat(v, 2, 0), 2, 1))
    for fmt in Y.FORMATS:
        frame = Y.to_frame(y, u, v, fmt)
        planes = (y, frame[6:]) if fmt in ("nv12", "nv21") else (y, u, v)
        assert np.array_equal(Y.yuv420_to_bgr(frame, fmt), ref) and np.array_equal(Y.yuv420_to_bgr(planes, fmt), ref), fmt


@pytest.mark.parametrize("h,w,S", [(1080, 1920, 640), (240, 320, 640), (1280, 1280, 640), (480, 640, 640), (2, 2, 64)])
def test_letterbox_of_a_converted_frame_equals_cv2(h, w, S):
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(h + w)
    frame = rng.integers(0, 256, (h * 3 // 2, w), dtype=np.uint8)
    bgr = Y.yuv420_to_bgr(frame, "nv12")
    got, ratio, pad = P.letterbox(bgr, S)
    nw, nh, top, left, bottom, right, r, _ = P.letterbox_geometry(h, w, S)
    resized = cv2.resize(bgr, (nw, nh), interpolation=cv2.INTER_LINEAR) if (nw, nh) != (w, h) else bgr
    ref = cv2.copyMakeBorder(resized, top, bottom, left, right, cv2.BORDER_CONSTANT, value=(114, 114, 114))
    assert np.array_equal(got, ref)


def test_plane_descriptor_matches_the_c_header(tmp_path):
    fields = ["luma", "luma_pitch", "chroma", "chroma_pitch", "format", "matrix"]
    lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{ROOT / "include" / "yre.h"}"', "int main(void) {",
             '  printf("size %zu\\n", sizeof(yre_yuv420_planes));']
    lines += [f'  printf("{f} %zu\\n", offsetof(yre_yuv420_planes, {f}));' for f in fields]
    lines += ["  return 0;", "}"]
    (tmp_path / "abi.c").write_text("\n".join(lines))
    subprocess.run(["gcc", "-o", str(tmp_path / "abi"), str(tmp_path / "abi.c")], check=True)
    out = subprocess.run([str(tmp_path / "abi")], check=True, capture_output=True, text=True).stdout
    got = {k: int(v) for k, v in (l.split() for l in out.strip().splitlines())}
    assert got["size"] == C.sizeof(L.Yuv420Planes)
    for f in fields:
        assert got[f] == getattr(L.Yuv420Planes, f).offset, f
    assert got["size"] == 48                   # pointers and pitches 8 bytes, enums 4 (x86-64 and aarch64 alike)


# ---- host-side rejections: the pointers are never dereferenced ------------------------------------------------------
BASE, DST = 0x7f0000000000, 0x7f0010000000


def _descs(n, h=1080, w=1920):
    d = (L.LetterboxDesc * n)()
    for i in range(n):
        d[i].h, d[i].w, d[i].dst = h, w, DST + i * (1 << 24)
        assert L.lib().yre_letterbox_geometry_rect(C.byref(d[i]), 640, 640, 32, None, None, None) == 0
    return d


def _planes(n, fmt=L.YUV_NV12, w=1920, pitch=2048):
    p = (L.Yuv420Planes * n)()
    nv = fmt in (L.YUV_NV12, L.YUV_NV21)
    for i in range(n):
        p[i].luma, p[i].luma_pitch = BASE + i * (1 << 24), pitch
        p[i].chroma[0] = BASE + i * (1 << 24) + (1 << 22)
        p[i].chroma[1] = None if nv else BASE + i * (1 << 24) + (1 << 23)
        p[i].chroma_pitch = pitch if nv else pitch // 2
        p[i].format, p[i].matrix = fmt, L.YUV_BT601
    return p


def _rejects(d, p, n, what: bytes):
    assert L.lib().yre_letterbox_yuv420_batch(d, p, n, None) == -1
    assert what in L.lib().yre_last_error(), L.lib().yre_last_error()


@pytest.mark.parametrize("fmt", [L.YUV_NV12, L.YUV_NV21, L.YUV_I420, L.YUV_YV12])
def test_host_side_rejections(fmt):
    nv = fmt in (L.YUV_NV12, L.YUV_NV21)
    # odd luma extents (the geometry itself is fine)
    for h, w in [(1081, 1920), (1080, 1919), (1, 2), (2, 1)]:
        _rejects(_descs(1, h, w), _planes(1, fmt), 1, b"even")
    # pitches shorter than their rows; the exact row length is accepted up to the launch
    for field, value in [("luma_pitch", 1918), ("chroma_pitch", 1918 if nv else 958)]:
        p = _planes(1, fmt)
        setattr(p[0], field, value)
        _rejects(_descs(1), p, 1, b"pitch")
    # unknown enums
    p = _planes(1, fmt); p[0].format = 4
    _rejects(_descs(1), p, 1, b"bad format")
    p = _planes(1, fmt); p[0].matrix = 2
    _rejects(_descs(1), p, 1, b"bad matrix")
    p = _planes(1, fmt); p[0].matrix = -1
    _rejects(_descs(1), p, 1, b"bad matrix")
    # null planes (and a second chroma plane where the format has one)
    for k in ("luma", 0, 1):
        p = _planes(1, fmt)
        if k == "luma":
            p[0].luma = None
        elif k == 0:
            p[0].chroma[0] = None
        else:
            p[0].chroma[1] = BASE if nv else None
        _rejects(_descs(1), p, 1, b"null plane")
    # the letterbox descriptor's own source fields must stay empty
    d = _descs(1); d[0].src = BASE
    _rejects(d, _planes(1, fmt), 1, b"src and row_pitch")
    d = _descs(1); d[0].row_pitch = 5760
    _rejects(d, _planes(1, fmt), 1, b"src and row_pitch")
    _rejects(_descs(1), None, 1, b"null planes")


def test_a_bad_frame_anywhere_in_the_batch_fails_before_the_first_launch():
    """40 frames take two launches; a bad 40th frame is reported without launching the first 32 (on a machine without
    a GPU a launch would fail with a CUDA error instead)."""
    d, p = _descs(40), _planes(40)
    p[39].matrix = 7
    _rejects(d, p, 40, b"bad matrix")
    d = _descs(40)
    d[39].out_mode = L.LB_U8_HWC
    _rejects(d, _planes(40), 40, b"share the destination extent")


def test_python_rejects_unknown_format_and_matrix_before_touching_the_device():
    frame = np.zeros((6, 4), np.uint8)
    with pytest.raises(ValueError, match="fmt"):
        preprocess(frame, 64, fmt="rgb")
    with pytest.raises(ValueError, match="yuv_matrix"):
        letterbox(frame, 64, fmt="nv12", yuv_matrix="bt2020")
