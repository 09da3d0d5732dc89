"""Multi-label NMS oracle (test infrastructure, not product code): upstream YOLOv9's multi-label candidate set on top of
yolo-re's non_max_suppression, restated three ways that must agree bit for bit.

  * ``nms_image_numpy``  numpy fp32 on top of oracle/nms_ref.py's greedy step;
  * ``nms_image_c``      tests/nms_ml_oracle.c through ctypes, for the big cases (up to 2.69 M candidates per image);
  * ``nms_image_torch``  a literal restatement with torch: ``(cls > conf).nonzero()``, the reference's class offset
                         (nms.py:79-81) and ``torchvision.ops.nms``.

Candidates are every (anchor a, class c) with ``score[a, c] > conf_thres`` (strict, fp32), also c in ``classes`` when
given, in row-major order (a, then c).  Everything after that is the reference's algorithm (oracle/nms_ref.py).
``multi_label=False`` is oracle/nms_ref.py itself.  The C port is compiled on first use into the temporary directory."""
from __future__ import annotations

import ctypes
import hashlib
import os
import subprocess
import tempfile
from pathlib import Path

import numpy as np

from oracle import nms_ref as N

_SRC = Path(__file__).resolve().parent / "nms_ml_oracle.c"
_LIB = None


def _candidates(pred, conf_thres, classes):
    sc = pred[:, 4:]
    a, c = np.nonzero(sc > np.float32(conf_thres))      # row-major: a ascending, then c
    if classes is not None:
        m = np.isin(c, np.asarray(classes))
        a, c = a[m], c[m]
    return a, c, sc[a, c]


def nms_image_numpy(pred: np.ndarray, conf_thres=0.25, iou_thres=0.45, max_det=300, classes=None, agnostic=False,
                    multi_label=False):
    """One image.  pred [A, 4+nc] fp32.  Returns (det [n,6] fp32, keep_anchor [n] int64)."""
    if not multi_label:
        return N.nms_image_numpy(pred, conf_thres, iou_thres, max_det, classes, agnostic)
    pred = np.ascontiguousarray(pred, np.float32)
    a, k, c = _candidates(pred, conf_thres, classes)
    if len(a) == 0:
        return np.zeros((0, 6), np.float32), np.zeros((0,), np.int64)
    xywh = pred[a, :4]
    half_w, half_h = xywh[:, 2] / np.float32(2), xywh[:, 3] / np.float32(2)
    boxes = np.stack((xywh[:, 0] - half_w, xywh[:, 1] - half_h,
                      xywh[:, 0] + half_w, xywh[:, 1] + half_h), 1).astype(np.float32)
    if agnostic:
        nms_boxes = boxes
    else:
        off = k.astype(np.float32) * (boxes.max() + np.float32(1))
        nms_boxes = boxes + off[:, None]
    keep = N.greedy_nms_numpy(nms_boxes, c, iou_thres)[:max_det]
    det = np.concatenate((boxes[keep], c[keep, None], k[keep, None].astype(np.float32)), 1)
    return det.astype(np.float32), a[keep].astype(np.int64)


def nms_image_torch(pred: np.ndarray, conf_thres=0.25, iou_thres=0.45, max_det=300, classes=None, agnostic=False):
    """Multi-label, written as upstream's general.py and the reference's nms.py write it, with torchvision's greedy step."""
    import torch
    import torchvision
    x = torch.from_numpy(np.ascontiguousarray(pred, np.float32))
    i, j = (x[:, 4:] > conf_thres).nonzero(as_tuple=False).T
    if classes is not None:
        m = (j[:, None] == torch.tensor(list(classes))).any(1)
        i, j = i[m], j[m]
    if len(i) == 0:
        return np.zeros((0, 6), np.float32), np.zeros((0,), np.int64)
    xywh = x[i, :4]
    boxes = torch.stack((xywh[:, 0] - xywh[:, 2] / 2, xywh[:, 1] - xywh[:, 3] / 2,
                         xywh[:, 0] + xywh[:, 2] / 2, xywh[:, 1] + xywh[:, 3] / 2), 1)
    conf, cls = x[i, 4 + j], j.float()
    nms_boxes = boxes if agnostic else boxes + cls[:, None] * (boxes.max() + 1)
    keep = torchvision.ops.nms(nms_boxes, conf, iou_thres)[:max_det]
    det = torch.cat((boxes[keep], conf[keep, None], cls[keep, None]), 1)
    return det.numpy(), i[keep].numpy().astype(np.int64)


def _lib():
    global _LIB
    if _LIB is None:
        src = _SRC.read_bytes()
        so = Path(tempfile.gettempdir()) / f"yre_nms_ml_oracle_{os.getuid()}_{hashlib.sha256(src).hexdigest()[:16]}.so"
        if not so.exists():
            tmp = so.with_suffix(f".{os.getpid()}.tmp")
            subprocess.check_call([os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-ffp-contract=off", "-fno-fast-math",
                                   "-Wall", "-shared", "-o", str(tmp), str(_SRC)])
            os.replace(tmp, so)
        _LIB = ctypes.CDLL(str(so))
        _LIB.yre_oracle_nms_image_multi_label.restype = ctypes.c_int
        _LIB.yre_oracle_nms_image_multi_label.argtypes = [
            ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_double, ctypes.c_int,
            ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
    return _LIB


def nms_image_c(pred: np.ndarray, conf_thres=0.25, iou_thres=0.45, max_det=300, classes=None, agnostic=False,
                multi_label=False):
    if not multi_label:
        return N.nms_image_c(pred, conf_thres, iou_thres, max_det, classes, agnostic)
    pred = np.ascontiguousarray(pred, np.float32)
    a, ch = pred.shape
    det = np.zeros((max_det, 6), np.float32)
    keep = np.zeros((max_det,), np.int64)
    cl = np.ascontiguousarray(classes if classes is not None else [], np.int32)
    n = _lib().yre_oracle_nms_image_multi_label(pred.ctypes.data, a, ch - 4, conf_thres, iou_thres, max_det,
                                                cl.ctypes.data if classes is not None else None,
                                                len(cl) if classes is not None else -1, int(bool(agnostic)),
                                                det.ctypes.data, keep.ctypes.data)
    if n < 0:
        raise MemoryError("multi-label oracle nms: allocation failed")
    return det[:n].copy(), keep[:n].copy()


def non_max_suppression(predictions, conf_thres=0.25, iou_thres=0.45, max_det=300, classes=None, agnostic=False,
                        impl: str = "c", return_keep: bool = False, multi_label: bool = False):
    """Batch wrapper with oracle/nms_ref.py's signature plus ``multi_label``.  predictions [B, A, 4+nc]."""
    if hasattr(predictions, "detach"):
        predictions = predictions.detach().cpu().float().numpy()
    fn = nms_image_c if impl == "c" else nms_image_numpy
    dets, keeps = [], []
    for i in range(predictions.shape[0]):
        d, k = fn(predictions[i], conf_thres, iou_thres, max_det, classes, agnostic, multi_label)
        dets.append(d)
        keeps.append(k)
    return (dets, keeps) if return_keep else dets
