"""Evaluator fast path (SURVEY.md 8f row 3): mAP with the detections kept on the device.

    compute_map(pred_boxes, pred_scores, pred_classes, gt_boxes, gt_classes, num_classes, iou_thresholds=None)
        same signature and result dict as the reference (src/yolo/eval/metrics.py:63-198)
    DetectionAccumulator  -- what src/yolo/eval/evaluator.py:96-161 does with Python lists of CPU tensors, but the
        per-batch detections (straight from non_max_suppression) and ground truths stay on the GPU until compute()

The reference walks every prediction in Python (one `.item()` and one IoU row per prediction and threshold).  Here
libyre's K11 kernel (yre_match_detections) produces the true-positive flag of every detection at every threshold in one
launch; only those flags, the scores and the classes come back to the host, where the precision/recall/AP arithmetic is
done in float64 numpy with the reference's exact operation order.  Results are bit-identical to the reference's
(tests/test_gpu_metrics.py, fixtures from the reference's own compute_map).  There is no CPU path for the matching.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib as L


def _cat_offsets(ts, dtype, width, dev):
    n = [int(t.shape[0]) for t in ts]
    off = torch.tensor([0] + list(np.cumsum(n)), dtype=torch.int32)
    if sum(n):
        flat = torch.cat([t.reshape(-1, width).to(device=dev, dtype=dtype) for t in ts if t.shape[0]])
    else:
        flat = torch.zeros((0, width), dtype=dtype, device=dev)
    return flat.contiguous(), off, (max(n) if n else 0)


def match_detections(dets, gt_boxes, gt_classes, iou_thresholds) -> tuple[torch.Tensor, torch.Tensor]:
    """dets: list (one per image) of CUDA [n, 6] rows (xyxy, conf, cls) in descending-score order, as
    non_max_suppression returns them.  Returns (tp uint8 [N, T] on the device, det_off int32 [B+1] on the host)."""
    if not dets:
        return torch.zeros((0, len(iou_thresholds)), dtype=torch.uint8), torch.zeros(1, dtype=torch.int32)
    dev = next((d.device for d in dets if d.is_cuda), None)
    if dev is None:
        raise L.YreError("match_detections: detections must be CUDA tensors (no CPU path)")
    if not 1 <= len(iou_thresholds) <= 16:
        raise ValueError("1..16 IoU thresholds")
    det, det_off, _ = _cat_offsets(dets, torch.float32, 6, dev)
    gtb, gt_off, max_gt = _cat_offsets(gt_boxes, torch.float32, 4, dev)
    gtc, _, _ = _cat_offsets([g.reshape(-1, 1) for g in gt_classes], torch.int32, 1, dev)
    tp = torch.zeros((det.shape[0], len(iou_thresholds)), dtype=torch.uint8, device=dev)
    if det.shape[0] == 0:
        return tp, det_off
    d = L.MatchDesc()
    det_off_d, gt_off_d = det_off.to(dev), gt_off.to(dev)
    d.det, d.det_stride, d.det_off = det.data_ptr(), 6, det_off_d.data_ptr()
    d.gt_boxes, d.gt_cls, d.gt_off = gtb.data_ptr(), gtc.data_ptr(), gt_off_d.data_ptr()
    d.B, d.n_thr, d.max_gt_per_image, d.tp = len(dets), len(iou_thresholds), max_gt, tp.data_ptr()
    for i, t in enumerate(iou_thresholds):
        d.thr[i] = float(t)
    with torch.cuda.device(dev):
        L.check(L.lib().yre_match_detections(C.byref(d), torch.cuda.current_stream(dev).cuda_stream), "match_detections")
    return tp, det_off


def _ap(recall: np.ndarray, precision: np.ndarray) -> float:
    """compute_ap (metrics.py:34-60) vectorised: same sentinels, running max from the right, first mrec >= t."""
    mrec = np.concatenate(([0.0], recall, [1.0]))
    mpre = np.concatenate(([1.0], precision, [0.0]))
    mpre = np.maximum.accumulate(mpre[::-1])[::-1]
    ts = np.linspace(0, 1, 101)
    idx = np.searchsorted(mrec, ts, side="left")
    out = np.where(idx < len(mrec), mpre[np.minimum(idx, len(mrec) - 1)], 0.0)
    return float(out.mean())


def _aggregate(scores, classes, tp, det_off, gt_classes, num_classes, iou_thresholds) -> dict[str, float]:
    """Host side of compute_map from the kernel's flags (all arrays numpy; detections image-major, score-descending)."""
    img = np.repeat(np.arange(len(det_off) - 1), np.diff(det_off))
    gt_all = np.concatenate([np.asarray(g).reshape(-1) for g in gt_classes]) if gt_classes else np.zeros(0, np.int64)
    all_aps: dict[float, list[float]] = {t: [] for t in iou_thresholds}
    for c in range(num_classes):
        total_gt = int((gt_all == c).sum())
        if total_gt == 0:
            continue
        sel = np.nonzero(classes == c)[0]                       # image-major, score-descending inside an image
        if sel.size == 0:
            for t in iou_thresholds:
                all_aps[t].append(0.0)
            continue
        order = sel[np.argsort(-scores[sel], kind="stable")]     # the reference's stable global sort
        flags = tp[order].astype(np.float64)
        for ti, t in enumerate(iou_thresholds):
            tpc, fpc = np.cumsum(flags[:, ti]), np.cumsum(1.0 - flags[:, ti])
            all_aps[t].append(_ap(tpc / total_gt, tpc / (tpc + fpc)))
    res = {"map50": float(np.mean(all_aps[0.5])) if 0.5 in all_aps and all_aps[0.5] else 0.0,
           "map75": float(np.mean(all_aps[0.75])) if 0.75 in all_aps and all_aps[0.75] else 0.0}
    vals: list[float] = []
    for t in iou_thresholds:
        vals.extend(all_aps.get(t, []))
    res["map"] = float(np.mean(vals)) if vals else 0.0
    del img
    return res


def _ordered_dets(pred_boxes, pred_scores, pred_classes, dev):
    dets = []
    for b, s, c in zip(pred_boxes, pred_scores, pred_classes):
        b, s, c = b.to(dev).float().reshape(-1, 4), s.to(dev).float().reshape(-1), c.to(dev).reshape(-1)
        if s.numel() > 1:
            o = torch.sort(s, descending=True, stable=True).indices
            b, s, c = b[o], s[o], c[o]
        dets.append(torch.cat([b, s[:, None], c.float()[:, None]], 1))
    return dets


def compute_map(pred_boxes, pred_scores, pred_classes, gt_boxes, gt_classes, num_classes: int,
                iou_thresholds: list[float] | None = None) -> dict[str, float]:
    """Drop-in for the reference's compute_map; tensors may live on the GPU (they are moved there otherwise)."""
    if iou_thresholds is None:
        iou_thresholds = [0.5 + 0.05 * i for i in range(10)]
    dev = next((t.device for t in list(pred_boxes) + list(gt_boxes) if t.is_cuda), torch.device("cuda"))
    dets = _ordered_dets(pred_boxes, pred_scores, pred_classes, dev)
    tp, det_off = match_detections(dets, [g.to(dev) for g in gt_boxes], [g.to(dev) for g in gt_classes], iou_thresholds)
    flat = torch.cat(dets) if dets and sum(d.shape[0] for d in dets) else torch.zeros((0, 6), device=dev)
    return _aggregate(flat[:, 4].cpu().numpy(), flat[:, 5].long().cpu().numpy(), tp.cpu().numpy(), det_off.numpy(),
                      [g.cpu().numpy() for g in gt_classes], num_classes, iou_thresholds)


class DetectionAccumulator:
    """Collects per-batch detections (as returned by non_max_suppression) and ground truths ON THE DEVICE; compute()
    runs the matching kernel once over everything and returns the reference's result dict."""

    def __init__(self, num_classes: int, iou_thresholds: list[float] | None = None):
        self.num_classes = num_classes
        self.iou_thresholds = iou_thresholds or [0.5 + 0.05 * i for i in range(10)]
        self.dets: list[torch.Tensor] = []
        self.gt_boxes: list[torch.Tensor] = []
        self.gt_classes: list[torch.Tensor] = []

    def update(self, detections, gt_boxes, gt_classes) -> None:
        """detections: list of [n, 6] CUDA tensors (one per image, NMS order); gt_boxes / gt_classes: matching lists."""
        if not (len(detections) == len(gt_boxes) == len(gt_classes)):
            raise ValueError("one detection tensor, gt box tensor and gt class tensor per image")
        for d in detections:
            if not d.is_cuda:
                raise L.YreError("DetectionAccumulator: detections must be CUDA tensors (no CPU path)")
        self.dets += [d.detach() for d in detections]
        self.gt_boxes += [g.detach().to(detections[0].device) if len(detections) else g for g in gt_boxes]
        self.gt_classes += [g.detach() for g in gt_classes]

    def compute(self) -> dict[str, float]:
        if not self.dets:
            return {"map50": 0.0, "map75": 0.0, "map": 0.0}
        dev = self.dets[0].device
        tp, det_off = match_detections(self.dets, self.gt_boxes, [g.to(dev) for g in self.gt_classes], self.iou_thresholds)
        flat = torch.cat(self.dets)
        return _aggregate(flat[:, 4].cpu().numpy(), flat[:, 5].long().cpu().numpy(), tp.cpu().numpy(), det_off.numpy(),
                          [g.cpu().numpy() for g in self.gt_classes], self.num_classes, self.iou_thresholds)


class Evaluator:
    """Device-side mirror of the reference's Evaluator (src/yolo/eval/evaluator.py:23-213): same constructor arguments and
    `evaluate()` result.  Every batch runs model -> NMS on the GPU and the detections never leave it until the final
    aggregation (the reference copies every image's detections to the CPU and loops over predictions in Python).
    The dataloader yields `(images [B,3,H,W] float in [0,1], targets [n,6] = (image index, class, cx, cy, w, h normalised),
    _, orig_shapes)` like the reference's (evaluator.py:96, 133-150), whose batches are square (H = W); a batch may also be
    a rectangle, as upstream val.py's rect batches are: normalised x and w then scale by W, y and h by H.  Debug visualisation is out of scope.
    augment=True evaluates with test-time augmentation (``model(images, augment=True)``, like upstream's
    ``val.py --augment``).  multi_label=True runs multi-label NMS (every class above conf_thres of an anchor is a
    candidate), as upstream's val.py does for its published mAPs; the default is the reference's single-label NMS."""

    def __init__(self, model, dataloader, num_classes: int = 80, conf_thres: float = 0.001, iou_thres: float = 0.6,
                 device="cuda", debug_dir=None, augment: bool = False, multi_label: bool = False):
        if debug_dir is not None:
            raise NotImplementedError("debug visualisation is outside the B200 hot path (SURVEY.md section 2)")
        self.model, self.dataloader, self.num_classes = model, dataloader, num_classes
        self.conf_thres, self.iou_thres, self.augment, self.multi_label = conf_thres, iou_thres, augment, multi_label
        self.device = torch.device("cuda" if device == "auto" else device)
        if self.device.type != "cuda":
            raise L.YreError("Evaluator: the B200 path needs a CUDA device (no CPU fallback)")
        self.model.to(self.device)

    @torch.no_grad()
    def evaluate(self, epoch: int = 0) -> dict[str, float]:
        from .nms import non_max_suppression
        self.model.eval()
        acc = DetectionAccumulator(self.num_classes)
        for images, targets, _, _orig_shapes in self.dataloader:
            images = images.to(self.device, non_blocking=True)
            bsz, H, W = images.shape[0], images.shape[2], images.shape[3]
            outputs = self.model(images, augment=True) if self.augment else self.model(images)
            if not isinstance(outputs, tuple):
                raise NotImplementedError("Raw feature map decoding not implemented")     # evaluator.py:113-115
            preds = outputs[0]
            if isinstance(preds, list):
                preds = preds[1]                                                           # main branch (evaluator.py:107-109)
            dets = non_max_suppression(preds.permute(0, 2, 1).contiguous(), conf_thres=self.conf_thres, iou_thres=self.iou_thres,
                                       multi_label=self.multi_label)
            targets = targets.to(self.device)
            # fp32 (x, y, w, h) * (W, H, W, H): for a square batch the same fp32 products as the reference's * img_size
            size = torch.tensor([W, H, W, H], dtype=torch.float32, device=self.device)
            gtb, gtc = [], []
            for i in range(bsz):
                t = targets[targets[:, 0] == i]
                xywh = t[:, 2:6].float() * size                                           # evaluator.py:139-141
                xyxy = torch.zeros_like(xywh)
                xyxy[:, 0] = xywh[:, 0] - xywh[:, 2] / 2
                xyxy[:, 1] = xywh[:, 1] - xywh[:, 3] / 2
                xyxy[:, 2] = xywh[:, 0] + xywh[:, 2] / 2
                xyxy[:, 3] = xywh[:, 1] + xywh[:, 3] / 2
                gtb.append(xyxy)
                gtc.append(t[:, 1].long())
            acc.update(dets, gtb, gtc)
        return acc.compute()
