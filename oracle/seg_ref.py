"""ORACLE (test infrastructure, NOT product code) -- CPU restatement of instance segmentation on gelan-c-seg.

What it restates (upstream YOLOv9; yolo-re has no segmentation head):
  * Proto                          models/common.py: Conv(c1, c_, 3) -> Upsample(2, nearest) -> Conv(c_, c_, 3) -> Conv(c_, c2)
  * Segment's mask towers          models/yolo.py: Conv(x, c4, 3) -> Conv(c4, c4, 3) -> nn.Conv2d(c4, nm, 1), c4 = max(ch0 // 4, nm)
  * process_mask, process_mask_native, crop_mask     utils/segment/general.py, literally, in torch
on top of ``gelan_ref`` (the detection head's inputs come from ``gelan_ref.forward(..., capture=...)``), and K15's
fp32 operation order in numpy (``k15_probs`` / ``k15_masks``), which the GPU kernel must reproduce outside the
derived band (``k15_band``)."""
from __future__ import annotations

import math
import tempfile
from collections import OrderedDict
from pathlib import Path

import numpy as np
import torch
import torch.nn.functional as F
import yaml

from . import gelan_ref as G


# --------------------------------------------------------------------------- graph and parameters
def load_graph(cfg_path: str | Path):
    """(nodes, nc, nm, npr) of a segmentation YAML: its layers are gelan_ref's, with the SegmentDFL head read as the
    DetectDFL it extends."""
    data = yaml.safe_load(open(cfg_path))
    head = data["layers"][-1]
    if head["type"] != "SegmentDFL":
        raise ValueError("the last layer must be a SegmentDFL head")
    nm, npr = head.get("num_masks", 32), head.get("num_protos", 256)
    det = {k: v for k, v in head.items() if k not in ("num_masks", "num_protos")}
    data["layers"] = data["layers"][:-1] + [dict(det, type="DetectDFL")]
    with tempfile.NamedTemporaryFile("w", suffix=".yaml") as f:
        yaml.safe_dump(data, f)
        f.flush()
        nodes, nc = G.load_graph(f.name)
    return nodes, nc, nm, npr


def mask_width(ch0: int, nm: int) -> int:
    return max(ch0 // 4, nm)                              # models/yolo.py Segment: c4


def seg_schema(nodes, nc: int, nm: int, npr: int) -> "OrderedDict[str, tuple]":
    """gelan_ref.param_schema plus the segmentation keys, in the order a SegmentDFL registers them."""
    out = G.param_schema(nodes, nc)
    det = nodes[-1]
    p = f"layers.{det.name}"
    ch0 = det.cin[0]
    G._conv_keys(out, f"{p}.proto.cv1", ch0, npr, 3)
    G._conv_keys(out, f"{p}.proto.cv2", npr, npr, 3)
    G._conv_keys(out, f"{p}.proto.cv3", npr, nm, 1)
    c4 = mask_width(ch0, nm)
    for i, ch in enumerate(det.cin):
        G._conv_keys(out, f"{p}.mask_convs.{i}.0", ch, c4, 3)
        G._conv_keys(out, f"{p}.mask_convs.{i}.1", c4, c4, 3)
        out[f"{p}.mask_convs.{i}.2.weight"] = ((nm, c4, 1, 1), torch.float32)
        out[f"{p}.mask_convs.{i}.2.bias"] = ((nm,), torch.float32)
    return out


# --------------------------------------------------------------------------- forward
def _proto(cx, p: str, x):
    return cx.cba(f"{p}.proto.cv3", cx.cba(f"{p}.proto.cv2", F.interpolate(cx.cba(f"{p}.proto.cv1", x), scale_factor=2.0,
                                                                            mode="nearest")))


def _mask_tower(cx, p: str, i: int, x):
    t = cx.cba(f"{p}.mask_convs.{i}.1", cx.cba(f"{p}.mask_convs.{i}.0", x))
    return F.conv2d(t, cx.sd[f"{p}.mask_convs.{i}.2.weight"], cx.sd[f"{p}.mask_convs.{i}.2.bias"])


@torch.no_grad()
def forward(nodes, nc: int, sd, x, *, calibrate: bool = False):
    """(y [B,4+nc,A], (raws, mc [B,nm,A], proto [B,nm,H/4,W/4])): the detection output of gelan_ref.forward and the
    segmentation parts on the head's captured inputs (levels concatenated along A in decode's order)."""
    cap: dict = {}
    y, raws = G.forward(nodes, nc, sd, x, capture=cap)
    det = nodes[-1]
    feats = [cap[s] for s in det.src]
    cx = G._Ctx(sd, calibrate)
    p = f"layers.{det.name}"
    proto = _proto(cx, p, feats[0])
    mc = torch.cat([_mask_tower(cx, p, i, f).flatten(2) for i, f in enumerate(feats)], 2)
    return y, (raws, mc, proto)


def calibrated_state_dict(nodes, nc: int, nm: int, npr: int, *, seed: int = 1234, cal_size: int = 640, cal_batch: int = 4):
    """gelan_ref.calibrated_state_dict for the detection keys (so a gelan-c loaded with them computes the same y), plus
    the segmentation keys: BN affine terms drawn as there, running statistics from one train-mode pass over the same
    calibration batch, and the mask towers' final convs re-drawn like the head's other final convs, N(0, 1/fan_in) with
    bias N(0, 0.5), which gives mask logits of O(1) spread."""
    sd = G.calibrated_state_dict(nodes, nc, seed=seed, cal_size=cal_size, cal_batch=cal_batch)
    g = torch.Generator().manual_seed(seed + 7)
    schema = seg_schema(nodes, nc, nm, npr)
    for k, (shape, dt) in schema.items():
        if k in sd:
            continue
        leaf = k.rsplit(".", 1)[1]
        if dt == torch.int64:
            t = torch.zeros((), dtype=torch.int64)
        elif leaf == "weight" and len(shape) == 4:
            bound = 1.0 / math.sqrt(shape[1] * shape[2] * shape[3])
            t = (torch.rand(shape, generator=g) * 2 - 1) * bound
        elif k.endswith(".bn.weight"):
            t = torch.empty(shape).uniform_(0.8, 1.2, generator=g)
        elif k.endswith(".bn.bias"):
            t = torch.empty(shape).normal_(0, 0.2, generator=g)
        elif leaf == "running_var":
            t = torch.ones(shape)
        else:
            t = torch.zeros(shape)
        sd[k] = t
    xcal = G.fractal(cal_batch, cal_size, torch.Generator().manual_seed(99))
    forward(nodes, nc, sd, xcal, calibrate=True)          # the segmentation BNs take their running statistics here
    det = nodes[-1].name
    for i in range(len(nodes[-1].cin)):
        w = sd[f"layers.{det}.mask_convs.{i}.2.weight"]
        sd[f"layers.{det}.mask_convs.{i}.2.weight"] = torch.empty_like(w).normal_(0, 1 / math.sqrt(w[0].numel()), generator=g)
        b = sd[f"layers.{det}.mask_convs.{i}.2.bias"]
        sd[f"layers.{det}.mask_convs.{i}.2.bias"] = torch.empty_like(b).normal_(0, 0.5, generator=g)
    return sd


# --------------------------------------------------------------------------- upstream utils/segment/general.py
def crop_mask(masks, boxes):
    n, h, w = masks.shape
    x1, y1, x2, y2 = torch.chunk(boxes[:, :, None], 4, 1)
    r = torch.arange(w, device=masks.device, dtype=x1.dtype)[None, None, :]
    c = torch.arange(h, device=masks.device, dtype=x1.dtype)[None, :, None]
    return masks * ((r >= x1) * (r < x2) * (c >= y1) * (c < y2))


def process_mask_probs(protos, masks_in, bboxes, shape, upsample=False):
    """process_mask before its final gt_(0.5)"""
    c, mh, mw = protos.shape
    ih, iw = shape
    masks = (masks_in @ protos.float().view(c, -1)).sigmoid().view(-1, mh, mw)
    downsampled_bboxes = bboxes.clone()
    downsampled_bboxes[:, 0] *= mw / iw
    downsampled_bboxes[:, 2] *= mw / iw
    downsampled_bboxes[:, 3] *= mh / ih
    downsampled_bboxes[:, 1] *= mh / ih
    masks = crop_mask(masks, downsampled_bboxes)
    if upsample:
        masks = F.interpolate(masks[None], shape, mode='bilinear', align_corners=False)[0]
    return masks


def process_mask(protos, masks_in, bboxes, shape, upsample=False):
    return process_mask_probs(protos, masks_in, bboxes, shape, upsample).gt_(0.5)


def native_slice(mh: int, mw: int, shape) -> tuple[int, int, int, int]:
    """(top, bottom, left, right) of process_mask_native"""
    gain = min(mh / shape[0], mw / shape[1])
    pad = (mw - shape[1] * gain) / 2, (mh - shape[0] * gain) / 2
    top, left = int(pad[1]), int(pad[0])
    bottom, right = int(mh - pad[1]), int(mw - pad[0])
    return top, bottom, left, right


def process_mask_native_probs(protos, masks_in, bboxes, shape):
    """process_mask_native before its final gt_(0.5)"""
    c, mh, mw = protos.shape
    masks = (masks_in @ protos.float().view(c, -1)).sigmoid().view(-1, mh, mw)
    top, bottom, left, right = native_slice(mh, mw, shape)
    masks = masks[:, top:bottom, left:right]
    masks = F.interpolate(masks[None], shape, mode='bilinear', align_corners=False)[0]
    return crop_mask(masks, bboxes)


def process_mask_native(protos, masks_in, bboxes, shape):
    return process_mask_native_probs(protos, masks_in, bboxes, shape).gt_(0.5)


# --------------------------------------------------------------------------- K15's operation order, in numpy
f32 = np.float32


def k15_logits(proto_hwc: np.ndarray, mc: np.ndarray) -> np.ndarray:
    """[n, mh, mw] logits: k = 0..nm-1 in order, one fp32 rounding per product and per sum"""
    acc = np.zeros((mc.shape[0],) + proto_hwc.shape[:2], dtype=f32)
    for k in range(mc.shape[1]):
        acc = (acc + (mc[:, k, None, None].astype(f32) * proto_hwc[None, :, :, k].astype(f32)).astype(f32)).astype(f32)
    return acc


def k15_sigmoid(x: np.ndarray) -> np.ndarray:
    with np.errstate(over="ignore"):
        return (f32(1) / (f32(1) + np.exp(-x.astype(f32)))).astype(f32)


def bilinear_axis(out: int, scale: float, n_in: int):
    """K12 / K15's bilinear_coeff for every destination index: (i0, i1, l0, l1)"""
    d = np.arange(out, dtype=f32)
    src = (f32(scale) * (d + f32(0.5))).astype(f32) - f32(0.5)
    src = np.maximum(src.astype(f32), f32(0))
    i0 = src.astype(np.int64)
    i1 = i0 + (i0 < n_in - 1)
    l1 = (src - i0.astype(f32)).astype(f32)
    return i0, i1, (f32(1) - l1).astype(f32), l1


def bilinear(m: np.ndarray, oh: int, ow: int) -> np.ndarray:
    """[n, h, w] -> [n, oh, ow]: v = hl0 (wl0 v00 + wl1 v01) + hl1 (wl0 v10 + wl1 v11), each op rounded to fp32"""
    _, h, w = m.shape
    y0, y1, h0, h1 = bilinear_axis(oh, f32(h) / f32(oh), h)
    x0, x1, w0, w1 = bilinear_axis(ow, f32(w) / f32(ow), w)
    r0, r1 = m[:, y0], m[:, y1]
    top = (w0 * r0[:, :, x0]).astype(f32) + (w1 * r0[:, :, x1]).astype(f32)
    bot = (w0 * r1[:, :, x0]).astype(f32) + (w1 * r1[:, :, x1]).astype(f32)
    return ((h0[:, None] * top.astype(f32)).astype(f32) + (h1[:, None] * bot.astype(f32)).astype(f32)).astype(f32)


def _keep(n: int, lo: np.ndarray, hi: np.ndarray) -> np.ndarray:
    """[k, n] bool: index r with r >= lo and r < hi (fp32 comparisons)"""
    r = np.arange(n, dtype=f32)[None]
    return (r >= lo[:, None]) & (r < hi[:, None])


def k15_probs(proto_hwc: np.ndarray, mc: np.ndarray, boxes: np.ndarray, mode: str, shape) -> np.ndarray:
    """K15's value before the > 0.5 for one image: proto_hwc [mh, mw, nm], mc [n, nm], boxes [n, 4] xyxy.
    mode "proto" / "input": shape = the input (h, w); "native": shape = the frame (h0, w0), boxes in frame pixels."""
    mh, mw, _ = proto_hwc.shape
    p = k15_sigmoid(k15_logits(proto_hwc, mc))
    boxes = boxes.astype(f32)
    if mode == "native":
        h0, w0 = shape
        top, bottom, left, right = native_slice(mh, mw, shape)
        v = bilinear(p[:, top:bottom, left:right], h0, w0)
        return v * (_keep(h0, boxes[:, 1], boxes[:, 3])[:, :, None] & _keep(w0, boxes[:, 0], boxes[:, 2])[:, None, :])
    ih, iw = shape
    rx, ry = f32(mw / iw), f32(mh / ih)
    keep = _keep(mh, boxes[:, 1] * ry, boxes[:, 3] * ry)[:, :, None] & _keep(mw, boxes[:, 0] * rx, boxes[:, 2] * rx)[:, None, :]
    p = np.where(keep, p, f32(0))
    return p if mode == "proto" else bilinear(p, ih, iw)


def k15_masks(proto_hwc, mc, boxes, mode, shape) -> np.ndarray:
    return k15_probs(proto_hwc, mc, boxes, mode, shape) > f32(0.5)


# --------------------------------------------------------------------------- the band
U = 2.0 ** -24


def k15_band(proto_hwc: np.ndarray, mc: np.ndarray, mode: str, shape) -> np.ndarray:
    """[n, oh, ow] bound on |p_K15 - p_ref| for any two fp32 evaluations of the same definition, in fp64.

      * dot product of nm terms, any summation order: |err| <= gamma_nm sum_k |mc_k proto_k|, gamma_n = n u / (1 - n u);
        two evaluations differ by at most twice that;
      * sigmoid is 1/4-Lipschitz, and each evaluation (exp within 2 ulp, 1 + e, the division) is within 4 u of it:
        |dp| <= 2 gamma_nm S / 4 + 8 u at a proto pixel;
      * a bilinear sample is a convex combination (weights within 2 u of each other's) of at most 4 such pixels, rounded
        in 3 steps: the largest pixel bound of the taps, plus 8 u.
    u = 2^-24.  Masks are compared where |p_ref - 0.5| exceeds this bound."""
    nm = mc.shape[1]
    gamma = nm * U / (1 - nm * U)
    S = np.abs(mc.astype(np.float64))[:, :, None, None] * np.abs(proto_hwc.astype(np.float64)).transpose(2, 0, 1)[None]
    e = 2 * gamma * S.sum(1) / 4 + 8 * U                  # [n, mh, mw]
    mh, mw = e.shape[1:]
    if mode == "proto":
        return e
    if mode == "native":
        h0, w0 = shape
        top, bottom, left, right = native_slice(mh, mw, shape)
        e, oh, ow = e[:, top:bottom, left:right], h0, w0
    else:
        oh, ow = shape
    y0, y1, _, _ = bilinear_axis(oh, f32(e.shape[1]) / f32(oh), e.shape[1])
    x0, x1, _, _ = bilinear_axis(ow, f32(e.shape[2]) / f32(ow), e.shape[2])
    taps = [e[:, ya][:, :, xa] for ya in (y0, y1) for xa in (x0, x1)]
    return np.maximum.reduce(taps) + 8 * U
