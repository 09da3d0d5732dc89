"""TEST INFRASTRUCTURE ONLY (see oracle/__init__.py): CPU restatement of 4:2:0 YUV -> BGR, the conversion K14 performs
before the letterbox of oracle/preproc_ref.py.

OpenCV's `cv2.cvtColor(frame, COLOR_YUV2BGR_{NV12,NV21,I420,YV12})` (opencv-python 4.13.0) is BT.601 limited range in
20-bit fixed point with nearest chroma: every 2 x 2 luma block uses one (U, V) sample.  Its constants are
round(c * 2^20) of the 3-decimal coefficients; per pixel

  uu = U - 128, vv = V - 128, y = max(0, Y - 16) * CY
  B = sat((y + 2^19 + CUB uu) >> 20)
  G = sat((y + 2^19 + CVG vv + CUG uu) >> 20)
  R = sat((y + 2^19 + CVR vv) >> 20)

BT.709 (HD video) uses the same scheme on the BT.709 limited-range coefficients; cv2 has no such code, so this
restatement is its definition.  Pinned against cv2 on all 2^24 (Y, U, V) triples in tests/test_cpu_yuv.py.

A frame is cv2's single array, (h * 3/2) x w uint8, or a tuple of planes: (y, uv) for NV12 / NV21 (uv: h/2 x w,
interleaved) and (y, u, v) for I420 / YV12 (u, v: h/2 x w/2).
"""
from __future__ import annotations

import numpy as np

FORMATS = ("nv12", "nv21", "i420", "yv12")

# (1.164, R from V, G from V, G from U, B from U) * 2^20, rounded
COEFFS = {"bt601": (1220542, 1673527, -852492, -409993, 2116026),      # 1.164, 1.596, -0.813, -0.391, 2.018
          "bt709": (1220542, 1880097, -558891, -223347, 2214593)}      # 1.164, 1.793, -0.533, -0.213, 2.112
FLOAT_COEFFS = {"bt601": (1.164, 1.596, -0.813, -0.391, 2.018), "bt709": (1.164, 1.793, -0.533, -0.213, 2.112)}


def split_planes(frame_or_planes, fmt: str):
    """(y [h, w], u [h/2, w/2], v [h/2, w/2]) of a frame in either form."""
    if fmt not in FORMATS:
        raise ValueError(f"unknown 4:2:0 format {fmt!r}")
    nv = fmt in ("nv12", "nv21")
    if isinstance(frame_or_planes, tuple):
        y = np.asarray(frame_or_planes[0])
        if nv:
            uv = np.asarray(frame_or_planes[1]).reshape(y.shape[0] // 2, y.shape[1] // 2, 2)
            c0, c1 = uv[..., 0], uv[..., 1]
            return (y, c0, c1) if fmt == "nv12" else (y, c1, c0)
        return y, np.asarray(frame_or_planes[1]), np.asarray(frame_or_planes[2])
    f = np.asarray(frame_or_planes)
    h, w = f.shape[0] * 2 // 3, f.shape[1]
    if f.shape[0] % 3 or h % 2 or w % 2:
        raise ValueError(f"a 4:2:0 frame is (h * 3/2) x w with even h and w, got {f.shape}")
    y = f[:h]
    if nv:
        uv = f[h:].reshape(h // 2, w // 2, 2)
        c0, c1 = uv[..., 0], uv[..., 1]
        return (y, c0, c1) if fmt == "nv12" else (y, c1, c0)
    chroma = f[h:].reshape(-1)
    c0 = chroma[:(h // 2) * (w // 2)].reshape(h // 2, w // 2)
    c1 = chroma[(h // 2) * (w // 2):].reshape(h // 2, w // 2)
    return (y, c0, c1) if fmt == "i420" else (y, c1, c0)


def convert(y: np.ndarray, u: np.ndarray, v: np.ndarray, matrix: str = "bt601") -> np.ndarray:
    """uint8 (..., 3) BGR of per-pixel Y, U, V arrays of one shape (the fixed-point formula above)."""
    cy, cvr, cvg, cug, cub = COEFFS[matrix]
    uu = u.astype(np.int64) - 128
    vv = v.astype(np.int64) - 128
    yy = np.maximum(y.astype(np.int64) - 16, 0) * cy + (1 << 19)
    sat = lambda t: np.clip(t >> 20, 0, 255).astype(np.uint8)
    return np.stack([sat(yy + cub * uu), sat(yy + cvg * vv + cug * uu), sat(yy + cvr * vv)], -1)


def yuv420_to_bgr(frame_or_planes, fmt: str, matrix: str = "bt601") -> np.ndarray:
    """uint8 h x w x 3 BGR: cv2.cvtColor(frame, COLOR_YUV2BGR_<fmt>) for "bt601"; the same scheme for "bt709"."""
    y, u, v = split_planes(frame_or_planes, fmt)
    up = lambda c: np.repeat(np.repeat(c, 2, 0), 2, 1)
    return convert(y, up(u), up(v), matrix)


def to_frame(y: np.ndarray, u: np.ndarray, v: np.ndarray, fmt: str) -> np.ndarray:
    """cv2's single (h * 3/2) x w array of the planes y [h, w], u, v [h/2, w/2]."""
    h, w = y.shape
    if fmt in ("nv12", "nv21"):
        c = np.stack([u, v] if fmt == "nv12" else [v, u], -1).reshape(h // 2, w)
    else:
        c = np.concatenate([u.reshape(-1), v.reshape(-1)] if fmt == "i420" else [v.reshape(-1), u.reshape(-1)]).reshape(h // 2, w)
    return np.concatenate([y, c], 0)


def encode_bt601(bgr: np.ndarray):
    """(y [h, w], u, v [h/2, w/2]) limited-range BT.601 planes of a uint8 BGR frame with even h, w, chroma averaged over
    each 2 x 2 block.  Only a source of natural-looking synthetic frames: decoding is what the letterbox checks."""
    b, g, r = (bgr[..., i].astype(np.float64) for i in range(3))
    y = 16 + 0.257 * r + 0.504 * g + 0.098 * b
    u = 128 - 0.148 * r - 0.291 * g + 0.439 * b
    v = 128 + 0.439 * r - 0.368 * g - 0.071 * b
    sub = lambda c: c.reshape(c.shape[0] // 2, 2, c.shape[1] // 2, 2).mean((1, 3))
    q = lambda c: np.clip(np.rint(c), 0, 255).astype(np.uint8)
    return q(y), q(sub(u)), q(sub(v))
