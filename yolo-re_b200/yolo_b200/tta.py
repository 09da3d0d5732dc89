"""Test-time augmentation: ``model(x, augment=True)`` of YOLOv5 / v8 / v9 (upstream ``_forward_augment``).

The batch runs at three branches -- scale 1; scale 0.83 mirrored left-right; scale 0.67 -- and their decoded
predictions are merged before NMS: de-scaled, de-flipped, the large-object level of the first branch and the
small-object level of the last one dropped, concatenated along the anchor axis.  Returns ``(y [B, 4+nc, A_tot], None)``
like upstream; feed y to ``non_max_suppression`` as a plain forward's y.  oracle/tta_ref.py restates the definition.

  * branch 0 is the plain forward of x, on the plan a plain ``model(x)`` uses;
  * branches 1 and 2 read fp32 images that K12 (yre_tta_scale_img) writes from x -- fp32 NCHW or uint8 BGR frames --
    into buffers allocated once per input shape and batch capacity, and run on ordinary fp32-input plans of their own;
  * K13 (yre_tta_merge) writes the merged y.
A dual-head model (yolov9-c) runs all three branches on main-only plans: every caller keeps the main head's y.  Height
and width must be multiples of 32 (ValueError otherwise).  fresh_outputs, use_cuda_graph, max_batch and the precision
apply to every branch as they do to a plain forward.  With model.max_shape, the plans of each branch take their buffers
from an arena of that branch's own (their plan tag differs), sized for the branch input of model.max_shape.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib as L
from . import engine as E
from .heads import DualDetectDFL


def geometry(h: int, w: int) -> L.TtaGeom:
    """Branch sizes and kept anchor windows of an h x w input (yre_tta_geometry)."""
    g = L.TtaGeom()
    if L.lib().yre_tta_geometry(int(h), int(w), C.byref(g)) != 0:
        raise ValueError(f"test-time augmentation needs a height and width that are multiples of 32, got {h}x{w}")
    return g


def _stream(t: torch.Tensor) -> int:
    return torch.cuda.current_stream(t.device).cuda_stream


def scale_img(x: torch.Tensor, g: L.TtaGeom, i: int, out: torch.Tensor | None = None, n: int | None = None) -> torch.Tensor:
    """K12: the input of branch i (upstream scale_img of x, flipped first for the mirrored branch) for the first n images
    of x (default: all), written to out (default: a new fp32 [B, 3, out_h, out_w] tensor).  x: fp32 [B,3,H,W] or uint8
    [B,H,W,3] BGR frames, CUDA, contiguous."""
    u8 = x.dtype == torch.uint8
    H, W = (x.shape[1], x.shape[2]) if u8 else (x.shape[2], x.shape[3])
    if (H, W) != (g.h, g.w) or not x.is_contiguous() or not x.is_cuda or x.dtype not in (torch.uint8, torch.float32):
        raise ValueError(f"tta scale_img: x must be a contiguous CUDA fp32 [B,3,{g.h},{g.w}] or uint8 [B,{g.h},{g.w},3] tensor")
    shape = (3, g.out_h[i], g.out_w[i])
    if out is None:
        out = torch.empty((x.shape[0],) + shape, dtype=torch.float32, device=x.device)
    if tuple(out.shape[1:]) != shape or out.dtype != torch.float32 or not out.is_contiguous() or out.device != x.device:
        raise ValueError(f"tta scale_img: out must be a contiguous fp32 [B, {shape[0]}, {shape[1]}, {shape[2]}] tensor on x's device")
    n = x.shape[0] if n is None else n
    d = L.TtaScaleDesc(None if u8 else x.data_ptr(), x.data_ptr() if u8 else None, min(x.shape[0], out.shape[0]), n, H, W,
                       g.flip[i], g.rh[i], g.rw[i], g.out_h[i], g.out_w[i], out.data_ptr())
    L.check(L.lib().yre_tta_scale_img(C.byref(d), _stream(x)), "tta_scale_img")
    return out


def merge(ys: list[torch.Tensor], g: L.TtaGeom, out: torch.Tensor | None = None) -> torch.Tensor:
    """K13: the merged predictions [n, A_tot, 4+nc] of the branches' decoded rows ys[i] (fp32 [n, A_i, 4+nc], contiguous,
    the layout under forward's [n, 4+nc, A_i] view); written to out (at least n images) or a new tensor."""
    n, _, no = ys[0].shape
    if out is None:
        out = torch.empty((n, g.A_tot, no), dtype=torch.float32, device=ys[0].device)
    d = L.TtaMergeDesc()
    for i, y in enumerate(ys):
        if y.dtype != torch.float32 or not y.is_contiguous() or tuple(y.shape) != (n, g.A[i], no):
            raise ValueError(f"tta merge: branch {i} must be a contiguous fp32 [{n}, {g.A[i]}, {no}] tensor")
        d.br[i] = L.TtaMergeBranch(y.data_ptr(), g.A[i], g.a_begin[i], g.a_end[i], g.scale[i], g.w if g.flip[i] else 0)
    if tuple(out.shape[1:]) != (g.A_tot, no) or out.shape[0] < n or not out.is_contiguous() or out.dtype != torch.float32:
        raise ValueError(f"tta merge: out must be a contiguous fp32 [>= {n}, {g.A_tot}, {no}] tensor")
    d.B, d.n, d.nc, d.out = out.shape[0], n, no - 4, out.data_ptr()
    L.check(L.lib().yre_tta_merge(C.byref(d), _stream(out)), "tta_merge")
    return out


def forward_augment(model, x: torch.Tensor, cap: int | None, max_hw: tuple[int, int] | None = None):
    """model(x, augment=True) for x as model_forward checked it; cap: model.max_batch; max_hw: model.max_shape."""
    u8 = x.dtype == torch.uint8
    n = x.shape[0]
    g = geometry(*((x.shape[1], x.shape[2]) if u8 else (x.shape[2], x.shape[3])))
    _, head = model._detect_layer()
    main_only = True if isinstance(head, DualDetectDFL) else None
    rows = n if cap is None else cap
    st = model._tta.get((tuple(x.shape[1:]), x.dtype, x.device.index, rows))
    if st is None:
        st = {"imgs": [torch.empty((rows, 3, g.out_h[i], g.out_w[i]), dtype=torch.float32, device=x.device) for i in (1, 2)]}
        model._tta[(tuple(x.shape[1:]), x.dtype, x.device.index, rows)] = st
    # the largest branch inputs: those of the largest height and width TTA takes (multiples of 32) up to max_hw
    gmax = None if max_hw is None else geometry(max_hw[0] // 32 * 32, max_hw[1] // 32 * 32)
    ys = [E.run_forward(model, x, cap, main_only, max_hw=max_hw)[0]]
    for i, buf in zip((1, 2), st["imgs"]):
        scale_img(x, g, i, out=buf, n=n)
        ys.append(E.run_forward(model, buf[:n], cap, main_only, tag=("tta", i),
                                max_hw=None if gmax is None else (gmax.out_h[i], gmax.out_w[i]))[0])
    ys = [y.permute(0, 2, 1) for y in ys]                      # the plans' [n, A, 4+nc] rows
    out = None
    if not model.fresh_outputs:
        out = st.get("out")
        if out is None:                                          # the static merged buffer, like a plan's own y
            out = st["out"] = torch.empty((rows, g.A_tot, ys[0].shape[2]), dtype=torch.float32, device=x.device)
    y = merge(ys, g, out)
    return y[:n].permute(0, 2, 1), None
