"""Test-time augmentation -- the definition the B200 path (yolo_b200.tta, K12 / K13) is checked against.

Upstream's `model(x, augment=True)`: YOLOv5 models/yolo.py `_forward_augment`, `_descale_pred`, `_clip_augmented` and
utils/torch_utils.py `scale_img`; ultralytics v8 runs the same code on the [B, no, A] layout used here.  The reference
(yolo-re) has no TTA, so this restatement is the specification:

  for (s, flip) in (1, none), (0.83, left-right), (0.67, none):
      xi = scale_img(x.flip(3) if flip else x, s)          # bilinear resize to (int(h s), int(w s)), pad 0.447 to
                                                           # (ceil(h s / 32) 32, ceil(w s / 32) 32) right and bottom
      yi = forward(xi)                                     # decoded y [B, 4+nc, Ai]: xywh in xi's pixels, class scores
      yi[:, :4] /= s (fp32);  flipped: x = w - x           # w: the ORIGINAL input width
  drop the last A0 // 21 anchors of branch 0 (P5) and the first 16 (A2 // 21) of branch 2 (P3); concat along anchors.

`scale_img_exact` restates K12's fp32 bilinear formula operation by operation (numpy fp32, one rounding per operation):
that is K12's bit-exact contract, and torch's F.interpolate agrees with it to within 1e-6.
"""
from __future__ import annotations

import math

import numpy as np
import torch
import torch.nn.functional as F

GS = 32                                    # max stride of the model: branch inputs are padded to multiples of it
SCALES = (1.0, 0.83, 0.67)
FLIPS = (None, 3, None)                    # upstream's flip codes: 3 = the width axis (left-right)
STRIDES = (8, 16, 32)
PAD = 0.447


def scale_img(img: torch.Tensor, ratio: float = 1.0, gs: int = GS) -> torch.Tensor:
    """utils/torch_utils.py scale_img (same_shape=False)"""
    if ratio == 1.0:
        return img
    h, w = img.shape[2:]
    s = (int(h * ratio), int(w * ratio))
    img = F.interpolate(img, size=s, mode="bilinear", align_corners=False)
    h, w = (math.ceil(x * ratio / gs) * gs for x in (h, w))
    return F.pad(img, [0, w - s[1], 0, h - s[0]], value=PAD)


def branch_shapes(h: int, w: int) -> list[tuple[tuple[int, int], tuple[int, int]]]:
    """((resized h, w), (padded h, w)) of every branch, with scale_img's arithmetic"""
    out = []
    for s in SCALES:
        if s == 1.0:
            out.append(((h, w), (h, w)))
        else:
            out.append(((int(h * s), int(w * s)), (math.ceil(h * s / GS) * GS, math.ceil(w * s / GS) * GS)))
    return out


def descale_pred(p: torch.Tensor, flip, scale: float, img_size) -> torch.Tensor:
    """_descale_pred on [B, no, A]: boxes / scale in fp32, x = w - x when the width axis was flipped"""
    p = p.clone()
    p[:, :4] /= scale
    if flip == 3:
        p[:, 0] = img_size[1] - p[:, 0]
    return p


def clip_augmented(y: list[torch.Tensor], nl: int = 3) -> list[torch.Tensor]:
    """_clip_augmented on [B, no, A]: the first branch loses its largest-stride level, the last one its smallest"""
    g = sum(4 ** x for x in range(nl))
    e = 1
    i = (y[0].shape[-1] // g) * sum(4 ** x for x in range(e))
    y[0] = y[0][..., :-i]
    i = (y[-1].shape[-1] // g) * sum(4 ** (nl - 1 - x) for x in range(e))
    y[-1] = y[-1][..., i:]
    return y


def windows(h: int, w: int) -> list[tuple[int, int, int]]:
    """(A_i, a_begin, a_end): the anchors of each branch's y and the window clip_augmented keeps"""
    out = []
    for _, (oh, ow) in branch_shapes(h, w):
        out.append([sum((oh // s) * (ow // s) for s in STRIDES), 0, 0])
        out[-1][2] = out[-1][0]
    out[0][2] -= out[0][0] // 21
    out[-1][1] = 16 * (out[-1][0] // 21)
    return [tuple(o) for o in out]


def branch_inputs(x: torch.Tensor) -> list[torch.Tensor]:
    """the three branch inputs of x [B, 3, h, w]"""
    return [scale_img(x.flip(f) if f else x, s) for s, f in zip(SCALES, FLIPS)]


def merge(ys: list[torch.Tensor], img_size) -> torch.Tensor:
    """descale + clip + concat of the branches' y [B, no, Ai]"""
    ys = [descale_pred(y, f, s, img_size) for y, s, f in zip(ys, SCALES, FLIPS)]
    return torch.cat(clip_augmented(ys), -1)


def forward_augment(forward, x: torch.Tensor):
    """_forward_augment: forward(xi) -> y [B, no, Ai]; returns (y [B, no, A_tot], None)"""
    return merge([forward(xi) for xi in branch_inputs(x)], x.shape[-2:]), None


def _coeff(n_out: int, n_in: int):
    scale = np.float32(n_in) / np.float32(n_out)
    d = np.arange(n_out, dtype=np.float32)
    src = scale * (d + np.float32(0.5)) - np.float32(0.5)
    src = np.maximum(src, np.float32(0))
    i0 = src.astype(np.int64)
    i1 = i0 + (i0 < n_in - 1)
    l1 = src - i0.astype(np.float32)
    return i0, i1, np.float32(1) - l1, l1


def scale_img_exact(img: np.ndarray, ratio: float, flip: bool, gs: int = GS) -> np.ndarray:
    """K12's arithmetic on fp32 [B, 3, h, w] (numpy fp32, every operation rounded once, no contraction)"""
    img = np.ascontiguousarray(img[..., ::-1] if flip else img, dtype=np.float32)
    h, w = img.shape[2:]
    (rh, rw), (oh, ow) = branch_shapes(h, w)[SCALES.index(ratio)]
    y0, y1, h0, h1 = _coeff(rh, h)
    x0, x1, w0, w1 = _coeff(rw, w)
    v00, v01 = img[:, :, y0][..., x0], img[:, :, y0][..., x1]
    v10, v11 = img[:, :, y1][..., x0], img[:, :, y1][..., x1]
    top = w0 * v00 + w1 * v01
    bot = w0 * v10 + w1 * v11
    res = h0[:, None] * top + h1[:, None] * bot
    out = np.full(img.shape[:2] + (oh, ow), np.float32(PAD), dtype=np.float32)
    out[:, :, :rh, :rw] = res
    return out
