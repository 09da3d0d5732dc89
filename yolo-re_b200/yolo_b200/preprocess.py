"""Device-side mirror of the steps either side of the detection path (SURVEY.md 8f row 1).

    letterbox(img, new_shape=640, color=(114, 114, 114))        reference scripts/detect.py:40-71 (+ auto, stride:
                                                                YOLOv9's rectangular letterbox)
    preprocess(imgs, new_shape=640)                             reference scripts/detect.py:223-227 (letterbox,
                                                                BGR->RGB, HWC->CHW, .float()/255, batched)
    scale_boxes(boxes, img_shape, orig_shape, ratio_pad=None)   reference scripts/detect.py:74-109

Same names, argument meaning and return values as the reference; the arithmetic runs in libyre's K8/K9 kernels
(bit-exact with cv2.resize(INTER_LINEAR) on uint8 and with torch's fp32 box arithmetic).  Images are uint8 HWC BGR,
either numpy arrays (copied to the current CUDA device) or CUDA uint8 tensors.  There is no CPU path.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib as L


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _to_device_u8(img) -> torch.Tensor:
    if isinstance(img, np.ndarray):
        if img.dtype != np.uint8:
            raise TypeError(f"letterbox: expected a uint8 image, got {img.dtype}")
        img = torch.from_numpy(np.ascontiguousarray(img)).cuda(non_blocking=True)
    if not (isinstance(img, torch.Tensor) and img.is_cuda and img.dtype == torch.uint8):
        raise L.YreError("letterbox: image must be a uint8 numpy array or a CUDA uint8 tensor (no CPU path)")
    if img.dim() != 3 or img.shape[2] != 3:
        raise ValueError(f"letterbox: expected an HxWx3 image, got {tuple(img.shape)}")
    if img.stride(2) != 1 or img.stride(1) != 3:
        img = img.contiguous()
    return img


def _desc(img: torch.Tensor, new_shape, color, stride: int = 0) -> tuple[L.LetterboxDesc, float, tuple[int, int]]:
    new_h, new_w = (new_shape, new_shape) if isinstance(new_shape, (int, np.integer)) else new_shape
    d = L.LetterboxDesc()
    d.src, d.h, d.w, d.row_pitch = img.data_ptr(), img.shape[0], img.shape[1], img.stride(0)
    d.color[0], d.color[1], d.color[2] = int(color[0]), int(color[1]), int(color[2])
    r, pw, ph = C.c_double(), C.c_int32(), C.c_int32()
    L.check(L.lib().yre_letterbox_geometry_rect(C.byref(d), int(new_h), int(new_w), int(stride), C.byref(r), C.byref(pw),
                                                C.byref(ph)), "letterbox_geometry_rect")
    return d, r.value, (pw.value, ph.value)


def letterbox(img, new_shape: int | tuple[int, int] = 640, color: tuple[int, int, int] = (114, 114, 114), auto: bool = False,
              stride: int = 32):
    """Resize and pad to ``new_shape`` (an int S for S x S, or an (h, w) pair): returns (uint8 HWC image, (r, r),
    (pad_w, pad_h)) like the reference.  ``auto=True`` keeps only the padding modulo ``stride`` on each axis, the
    smallest stride-multiple rectangle (YOLOv9's ``letterbox(auto=True)``; 1920x1080 -> 640x384 at 640).  A numpy input
    gives a numpy result, a CUDA tensor stays on the device."""
    was_numpy = isinstance(img, np.ndarray)
    src = _to_device_u8(img)
    d, r, pad = _desc(src, new_shape, color, stride if auto else 0)
    out = torch.empty((d.out_h, d.out_w, 3), dtype=torch.uint8, device=src.device)
    d.out_mode, d.dst = L.LB_U8_HWC, out.data_ptr()
    L.check(L.lib().yre_letterbox_u8(C.byref(d), _stream()), "letterbox_u8")
    return (out.cpu().numpy() if was_numpy else out), (r, r), pad


def preprocess(imgs, new_shape: int | tuple[int, int] = 640, color: tuple[int, int, int] = (114, 114, 114),
               out: torch.Tensor | None = None, dtype: torch.dtype = torch.float32, auto: bool = False, stride: int = 32):
    """Fused letterbox + BGR->RGB + HWC->CHW + /255 for a list of images (or one image).

    Returns (x [B, 3, H, W] fp32 on the device, ratios [(r, r)], pads [(pad_w, pad_h)]) -- x is the tensor the
    reference builds at scripts/detect.py:223-227, ready for ``model(x)``.  H x W is ``new_shape`` (an int S for S x S,
    or an (h, w) pair).

    ``auto=True`` makes a rectangular batch: every image's smallest stride-multiple rectangle is found as
    ``letterbox(auto=True)`` finds it, the batch takes the per-axis maximum of those, and an image whose own rectangle
    is smaller is letterboxed into the batch's (the reference's rect batches do the same).  Each image is centred;
    its ratio and padding are reported per image.

    ``dtype=torch.uint8`` stops after the letterbox and returns the frames as one uint8 [B, H, W, 3] BGR batch;
    ``model(x_u8)`` then fuses BGR->RGB / HWC->CHW / /255 into its first convolution, so the fp32 image tensor is
    never written (4x less traffic on both sides of it).  Detections are identical either way."""
    if isinstance(imgs, (np.ndarray, torch.Tensor)) and imgs.ndim == 3:
        imgs = [imgs]
    srcs = [_to_device_u8(i) for i in imgs]
    dev = srcs[0].device
    if dtype not in (torch.float32, torch.uint8):
        raise ValueError("preprocess: dtype must be torch.float32 or torch.uint8")
    geo = [_desc(src, new_shape, color, stride if auto else 0) for src in srcs]
    H, W = max(g[0].out_h for g in geo), max(g[0].out_w for g in geo)
    geo = [g if (g[0].out_h, g[0].out_w) == (H, W) else _desc(src, (H, W), color) for g, src in zip(geo, srcs)]
    shape = (len(srcs), 3, H, W) if dtype == torch.float32 else (len(srcs), H, W, 3)
    if out is None:
        out = torch.empty(shape, dtype=dtype, device=dev)
    if tuple(out.shape) != shape or out.dtype != dtype or not out.is_contiguous() or not out.is_cuda:
        raise ValueError(f"preprocess: `out` must be a contiguous CUDA {dtype} tensor of shape {shape}")
    ratios, pads = [], []
    descs = (L.LetterboxDesc * len(srcs))()
    for i, (d, r, pad) in enumerate(geo):
        d.out_mode, d.dst = (L.LB_F32_CHW if dtype == torch.float32 else L.LB_U8_HWC), out[i].data_ptr()
        descs[i] = d
        ratios.append((r, r)); pads.append(pad)
    L.check(L.lib().yre_letterbox_u8_batch(descs, len(srcs), _stream()), "letterbox_u8_batch")
    return out, ratios, pads


def scale_rows(ratios, pads, orig_shapes, device=None) -> torch.Tensor:
    """fp32 [B, 5] rows (pad_w, pad_h, gain, orig_w, orig_h) for ``nms_raw(..., scale=...)`` /
    ``non_max_suppression_async(..., scale=...)``: the ``ratio_pad`` form of scale_boxes (scripts/detect.py:100-101)
    for every image of a batch, so the box rescale/clip runs inside the NMS output pass."""
    rows = [[float(p[0]), float(p[1]), float(r[0]), float(o[1]), float(o[0])] for r, p, o in zip(ratios, pads, orig_shapes)]
    t = torch.tensor(rows, dtype=torch.float32)
    return t.to(device, non_blocking=True) if device is not None else t


def scale_boxes(boxes: torch.Tensor, img_shape, orig_shape, ratio_pad=None) -> torch.Tensor:
    """Boxes (xyxy, model-input pixels) -> original-image pixels, clipped; IN PLACE like the reference, any row
    stride (``detections[:, :4]`` works)."""
    if ratio_pad is None:
        gain = min(img_shape[0] / orig_shape[0], img_shape[1] / orig_shape[1])
        pad = ((img_shape[1] - orig_shape[1] * gain) / 2, (img_shape[0] - orig_shape[0] * gain) / 2)
    else:
        gain, pad = ratio_pad[0][0], ratio_pad[1]
    if not (boxes.is_cuda and boxes.dtype == torch.float32):
        raise L.YreError("scale_boxes: boxes must be a CUDA fp32 tensor (no CPU path)")
    if boxes.dim() != 2 or boxes.shape[1] < 4 or (boxes.shape[0] > 1 and boxes.stride(1) != 1):
        raise ValueError(f"scale_boxes: expected [n, >=4] rows with unit column stride, got {tuple(boxes.shape)}")
    n = boxes.shape[0]
    stride = boxes.stride(0) if n > 1 else max(4, boxes.shape[1])
    L.check(L.lib().yre_scale_boxes(boxes.data_ptr(), n, stride, float(pad[0]), float(pad[1]), float(gain),
                                    float(orig_shape[1]), float(orig_shape[0]), _stream()), "scale_boxes")
    return boxes
