"""Instance-segmentation masks on the GPU (K15): upstream YOLOv9's ``process_mask``, ``process_mask_native`` and
``crop_mask`` (utils/segment/general.py) for the kept detections of a whole batch, in one launch after NMS.

``masks_raw`` takes what a segmentation model's forward and ``nms_raw`` return, without a host synchronisation:

    y, (raws, mc, proto) = model(x)                        # gelan-c-seg
    out, counts, keep = nms_raw(y.permute(0, 2, 1), 0.25, 0.45)
    masks = masks_raw(proto, mc, out, counts, keep, "input", shape=x.shape[2:])   # [B, max_det, H, W] bool

Rows ``j >= counts[b]`` of the result are not written (they hold whatever the allocation held).  ``process_mask`` and
``process_mask_native`` keep upstream's per-image signatures.  Masks are bool, where upstream leaves float 0. / 1.
(INTEGRATION.md section 4)."""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib as L

MODES = {"proto": L.MASK_PROTO, "input": L.MASK_INPUT, "native": L.MASK_NATIVE}


def _nhwc(proto: torch.Tensor) -> torch.Tensor:
    """proto [B, nm, mh, mw] as an NHWC-contiguous tensor (the forward's own proto already is one: no copy)"""
    t = proto.permute(0, 2, 3, 1)
    return t if t.is_contiguous() else t.contiguous()


def masks_raw(proto: torch.Tensor, mc: torch.Tensor, out: torch.Tensor, counts: torch.Tensor, keep: torch.Tensor,
              mode: str = "input", shape=None, scale: torch.Tensor | None = None) -> torch.Tensor:
    """Runs K15 and returns the padded device masks ``[B, max_det, H, W]`` (bool) without a host synchronisation.

    proto: fp32 ``[B, nm, mh, mw]``; mc: fp32 ``[B, nm, A]`` (both as the forward returns them); out, counts, keep: what
    ``nms_raw`` returns.  mode:
      * ``"proto"``: ``process_mask(upsample=False)``, ``mh x mw`` masks; ``shape`` = the network input ``(h, w)``;
      * ``"input"``: ``process_mask(upsample=True)``, masks of the network input ``shape = (h, w)``;
      * ``"native"``: ``process_mask_native`` on boxes in frame pixels (``nms_raw(..., scale=scale)``); ``scale`` is that
        fp32 ``[B, 5]`` tensor (pad_w, pad_h, gain, orig_w, orig_h).  Image b's mask is the ``[:orig_h, :orig_w]`` window
        of planes ``shape = (H, W)`` large enough for every frame (None: the largest frame, read with one host sync)."""
    if mode not in MODES:
        raise ValueError(f"mode must be one of {sorted(MODES)} (got {mode!r})")
    for t in (proto, mc, out, counts, keep):
        if not t.is_cuda:
            raise L.YreError("the yolo-re B200 path runs on CUDA tensors only (there is no CPU fallback)")
    if proto.dim() != 4 or mc.dim() != 3 or out.dim() != 3 or out.shape[2] != 6:
        raise ValueError("expected proto [B, nm, mh, mw], mc [B, nm, A] and NMS rows [B, max_det, 6]")
    Bn, nm, mh, mw = proto.shape
    max_det = out.shape[1]
    if mc.shape[:2] != (Bn, nm) or out.shape[0] != Bn or tuple(counts.shape) != (Bn,) or tuple(keep.shape) != (Bn, max_det):
        raise ValueError("proto, mc and the NMS outputs disagree on the batch, the mask count or max_det")
    if proto.dtype != torch.float32 or mc.dtype != torch.float32 or out.dtype != torch.float32 or \
            counts.dtype != torch.int32 or keep.dtype != torch.int64:
        raise ValueError("proto, mc and out must be fp32, counts int32 and keep int64 (as the forward and nms_raw return them)")
    p = _nhwc(proto)
    m = mc.permute(0, 2, 1)
    m = m if m.is_contiguous() else m.contiguous()
    out, counts, keep = out.contiguous(), counts.contiguous(), keep.contiguous()
    in_h = in_w = 0
    if mode == "native":
        if scale is None or not (scale.is_cuda and scale.dtype == torch.float32 and tuple(scale.shape) == (Bn, 5)):
            raise ValueError("native mode needs scale, the fp32 CUDA tensor [B, 5] given to nms_raw")
        scale = scale.contiguous()
        if shape is None:
            shape = tuple(int(v) for v in scale[:, [4, 3]].amax(0).tolist())
        oh, ow = int(shape[0]), int(shape[1])
    else:
        if shape is None:
            raise ValueError(f"mode {mode!r} needs shape, the network input (h, w)")
        in_h, in_w = int(shape[0]), int(shape[1])
        oh, ow = (mh, mw) if mode == "proto" else (in_h, in_w)
    masks = torch.empty((Bn, max_det, max(oh, 0), max(ow, 0)), dtype=torch.bool, device=proto.device)
    if Bn == 0 or max_det == 0:
        return masks
    d = L.MaskDesc(p.data_ptr(), Bn, Bn, mh, mw, nm, p.stride(2), m.data_ptr(), m.shape[1], out.data_ptr(), counts.data_ptr(),
                   keep.data_ptr(), max_det, MODES[mode], in_h, in_w, scale.data_ptr() if mode == "native" else None,
                   masks.data_ptr(), oh, ow)
    with torch.cuda.device(proto.device):
        L.check(L.lib().yre_seg_masks(C.byref(d), torch.cuda.current_stream(proto.device).cuda_stream), "seg_masks")
    return masks


def _one_image(protos, masks_in, bboxes):
    """an image's (proto, mc, NMS rows, counts, keep) in the batched layout of masks_raw"""
    n = masks_in.shape[0]
    dev = protos.device
    det = torch.zeros((1, max(n, 1), 6), dtype=torch.float32, device=dev)
    det[0, :n, :4] = bboxes.float()
    mc = torch.zeros((1, max(n, 1), masks_in.shape[1]), dtype=torch.float32, device=dev)
    mc[0, :n] = masks_in.float()
    counts = torch.full((1,), n, dtype=torch.int32, device=dev)
    keep = torch.arange(max(n, 1), dtype=torch.int64, device=dev)[None]
    return protos.float()[None], mc.permute(0, 2, 1), det, counts, keep


def process_mask(protos: torch.Tensor, masks_in: torch.Tensor, bboxes: torch.Tensor, shape, upsample: bool = False):
    """Upstream's process_mask on one image: protos [nm, mh, mw], masks_in [n, nm], bboxes [n, 4] xyxy in input pixels,
    shape = the input (h, w).  Returns bool [n, h, w] (upsample) or [n, mh, mw]."""
    n = masks_in.shape[0]
    r = masks_raw(*_one_image(protos, masks_in, bboxes), "input" if upsample else "proto", shape=shape)
    return r[0, :n]


def process_mask_native(protos: torch.Tensor, masks_in: torch.Tensor, bboxes: torch.Tensor, shape):
    """Upstream's process_mask_native on one image: bboxes [n, 4] xyxy in frame pixels, shape = the frame (h0, w0).
    Returns bool [n, h0, w0]."""
    n = masks_in.shape[0]
    h0, w0 = int(shape[0]), int(shape[1])
    scale = torch.tensor([[0.0, 0.0, 1.0, w0, h0]], dtype=torch.float32, device=protos.device)
    r = masks_raw(*_one_image(protos, masks_in, bboxes), "native", shape=(h0, w0), scale=scale)
    return r[0, :n]
