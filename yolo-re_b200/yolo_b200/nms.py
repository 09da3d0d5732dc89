"""Batched class-aware NMS on the GPU -- drop-in for ``yolo.utils.nms.non_max_suppression``
(src/yolo/utils/nms.py:19-94): same signature, same return type (list of ``[n,6]`` tensors
``[x1,y1,x2,y2,conf,cls]`` per image), bit-identical results given the same predictions.

``multi_label=True`` (an extension, default off) takes upstream YOLOv9's candidate set, as its val.py does for every
published mAP: every (anchor, class) pair whose score is above ``conf_thres`` is a candidate of its own, not only the best
class of each anchor.  The rest of the algorithm is the reference's unchanged (INTEGRATION.md section 4)."""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib as L


def _workspace(lib, Bn: int, A: int, nc: int, multi_label: bool, dev: torch.device) -> torch.Tensor:
    """Scratch of one call (candidate keys, class map, counters).  It comes from torch's caching allocator, which
    is stream-ordered: the block is handed to a later call on the SAME stream only, or to another stream after this
    stream's work on it has finished -- so calls in flight on different streams / threads never share scratch and
    the entry point stays re-entrant (SURVEY.md 8b).  Steady state: no cudaMalloc, one cached block per stream."""
    n = lib.yre_nms_multi_label_workspace_bytes(Bn, A, nc) if multi_label else lib.yre_nms_workspace_bytes(Bn, A)
    if n == 0:
        raise L.YreError(f"nms: multi-label with {A} anchors x {nc} classes exceeds 2^30 candidates per image")
    return torch.empty((n,), dtype=torch.uint8, device=dev)


def nms_raw(predictions: torch.Tensor, conf_thres=0.25, iou_thres=0.45, max_det=300, classes=None, agnostic=False,
            scale=None, multi_label=False):
    """Runs K7 and returns the padded device results ``(out[B,max_det,6], counts[B] int32,
    keep_anchor[B,max_det] int64)`` without any host synchronisation.

    ``scale`` (optional, fp32 CUDA tensor [B,5] = pad_w, pad_h, gain, orig_w, orig_h per image): the kept boxes are
    written already mapped back to the original image, i.e. ``scale_boxes`` (scripts/detect.py:74-109) fused into the
    NMS output pass -- same fp32 arithmetic as the stand-alone K9 kernel.

    ``multi_label``: every class above ``conf_thres`` of an anchor is a candidate (upstream val.py's setting);
    ``keep_anchor`` is then the anchor of each kept row, so several rows may share one anchor."""
    if not predictions.is_cuda:
        raise L.YreError("the yolo-re B200 path runs on CUDA tensors only (there is no CPU fallback)")
    if predictions.dim() != 3 or predictions.shape[2] <= 4:
        raise ValueError("predictions must be [batch, num_anchors, 4 + num_classes]")
    lib = L.lib()
    pred = predictions.contiguous().float()
    Bn, A, ch = pred.shape
    dev = pred.device
    out = torch.empty((Bn, max_det, 6), dtype=torch.float32, device=dev)
    counts = torch.empty((Bn,), dtype=torch.int32, device=dev)
    keep = torch.empty((Bn, max_det), dtype=torch.int64, device=dev)
    if Bn == 0 or A == 0:
        return out, counts.zero_(), keep
    with torch.cuda.device(dev):
        ws = _workspace(lib, Bn, A, ch - 4, multi_label, dev)
        cls_t = None
        if classes is not None:
            cls_t = torch.as_tensor(list(classes), dtype=torch.int32, device=dev)
        if scale is not None:
            if not (scale.is_cuda and scale.dtype == torch.float32 and tuple(scale.shape) == (Bn, 5) and scale.is_contiguous()):
                raise ValueError("scale must be a contiguous fp32 CUDA tensor [B, 5] = (pad_w, pad_h, gain, orig_w, orig_h)")
        d = L.NmsDesc(pred.data_ptr(), Bn, A, ch - 4, float(conf_thres), float(iou_thres), int(max_det),
                      cls_t.data_ptr() if cls_t is not None and cls_t.numel() else None,
                      (cls_t.numel() if cls_t is not None else -1), int(bool(agnostic)),
                      out.data_ptr(), counts.data_ptr(), keep.data_ptr(), ws.data_ptr(), ws.numel(),
                      scale.data_ptr() if scale is not None else None)
        fn = lib.yre_nms_batched_multi_label if multi_label else lib.yre_nms_batched
        L.check(fn(C.byref(d), torch.cuda.current_stream(dev).cuda_stream), "nms_batched")
    return out, counts, keep


class PendingDetections:
    """Detections of one ``non_max_suppression_async`` call that are still on the device.  ``result()`` waits for
    the counts (one small D2H that was enqueued right behind the NMS kernels) and slices the padded output into
    the reference's ``list[Tensor[n, 6]]``."""

    def __init__(self, out, counts, keep):
        self.out, self.counts, self.keep = out, counts, keep
        self._host = torch.empty(counts.shape, dtype=torch.int32, pin_memory=True)
        self._host.copy_(counts, non_blocking=True)
        self._event = torch.cuda.Event()
        self._event.record(torch.cuda.current_stream(out.device))

    def result(self) -> list[torch.Tensor]:
        self._event.synchronize()
        n = self._host.tolist()
        rows = self.out.unbind(0)
        return [rows[i][: n[i]] for i in range(len(rows))]


def non_max_suppression_async(predictions: torch.Tensor, conf_thres: float = 0.25, iou_thres: float = 0.45,
                              max_det: int = 300, classes: list[int] | None = None, agnostic: bool = False,
                              scale=None, multi_label: bool = False) -> PendingDetections:
    """Same arguments as ``non_max_suppression``; returns immediately.  Lets a caller enqueue the next batch's
    forward before it blocks on this batch's counts (``.result()``)."""
    return PendingDetections(*nms_raw(predictions, conf_thres, iou_thres, max_det, classes, agnostic, scale, multi_label))


def non_max_suppression(predictions: torch.Tensor, conf_thres: float = 0.25, iou_thres: float = 0.45,
                        max_det: int = 300, classes: list[int] | None = None, agnostic: bool = False,
                        multi_label: bool = False) -> list[torch.Tensor]:
    """predictions: (batch, num_anchors, 4 + num_classes), boxes xywh in pixels, scores already
    sigmoided.  Returns one (n, 6) tensor per image.  The only host sync is reading the B counts.
    multi_label=True keeps every class above conf_thres of an anchor as its own candidate (upstream val.py)."""
    if predictions.is_cuda and (predictions.shape[0] == 0 or predictions.shape[1] == 0):
        out, counts, _ = nms_raw(predictions, conf_thres, iou_thres, max_det, classes, agnostic, multi_label=multi_label)
        return [out[i, :0] for i in range(out.shape[0])]
    return non_max_suppression_async(predictions, conf_thres, iou_thres, max_det, classes, agnostic,
                                     multi_label=multi_label).result()
