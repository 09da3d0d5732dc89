"""Engine-plan compiler: walks the (reference-compatible) module tree once and records a flat list
of libyre launches -- the replacement for the reference's per-forward interpreter loop
(src/yolo/model/model.py:87-107) and its ~600 ATen dispatches.

What the compiler does (SURVEY.md section 7.1):
  * folds BatchNorm into the conv weights/bias in fp64 (w' = w*g/sqrt(var+eps), b' = beta - mu*g/sqrt(var+eps),
    eps = 1e-3, src/yolo/blocks/conv.py:85), then casts the weights to bf16 (product), fp16 (opt-in) or fp32 (validation);
    the bias stays fp32;
  * folds RepConv's 1x1 branch into the 3x3 centre tap (conv.py:140-141);
  * merges sibling convs that share an input: RepNCSP conv1||conv2 (csp.py:59-60) and the detect
    towers' first 3x3s (heads/detect.py:48-64);
  * expands grouped head convs to block-diagonal dense weights;
  * turns chunk()/cat() (gelan.py:59-62, csp.py:60, common.py:33, detect.py:88) into channel windows of
    shared NHWC buffers, so producers write straight into their consumer's concat slice;
  * residual adds (bottleneck.py:51) run in the conv epilogue, in place.

PyTorch is used for device memory only (torch.empty / data_ptr / current stream).
"""
from __future__ import annotations

import ctypes as C
import math
from contextlib import contextmanager
from functools import cache
from typing import NamedTuple

import torch
import torch.nn as nn

from . import _lib as L
from . import blocks as B
from .heads import REG_MAX, DetectDFL, DualDetectDFL, SegmentDFL

_DEFAULT_PRECISION = "bf16"
# per precision: (libyre activation dtype, torch dtype)
_DTYPES = {"bf16": (L.BF16, torch.bfloat16), "fp16": (L.F16, torch.float16), "fp32": (L.F32, torch.float32)}
_TORCH_DT = {L.BF16: torch.bfloat16, L.F16: torch.float16, L.F32: torch.float32}
F16_MAX = 65504.0         # largest finite fp16


def _check_f16_range(w: torch.Tensor, name: str) -> None:
    """fp16 weights: a folded weight beyond +-65504 would become +-inf, so the compile fails instead, naming the layer."""
    m = float(w.abs().max()) if w.numel() else 0.0
    if not m <= F16_MAX:
        raise L.YreError(f"fp16 precision: layer '{name}' has a folded weight of magnitude {m:.6g} > {F16_MAX:g} "
                         "(largest finite fp16); run it in bf16 or fp32")
# Test hook: with a CPU device a plan can be *compiled* (buffers on the host, every op recorded in
# Plan.trace and in the C plan) but never run -- tests/ replays the trace with a CPU interpreter to
# check the graph wiring without a GPU.  The product path never sets this.
_ALLOW_CPU_DRY_RUN = False
# Offsets of the buffers a plan sub-allocates from a shape arena (model.max_shape) are multiples of this: the caching
# allocator's own alignment, which the TMA tensor maps (16 B base) and the 64-B channel windows of every view rely on.
ARENA_ALIGN = 512


class _LayoutOnly:
    """Stands in for libyre in a plan that only lays out its buffers (sizing a shape arena): every call succeeds and
    records nothing."""
    def __getattr__(self, name):
        return lambda *a: 0


@contextmanager
def precision(p: str):
    """Precision ("bf16", "fp16" or "fp32") used when a *block* (not a whole YOLO) is called directly."""
    if p not in _DTYPES:
        raise ValueError("precision must be 'bf16', 'fp16' or 'fp32'")
    global _DEFAULT_PRECISION
    old, _DEFAULT_PRECISION = _DEFAULT_PRECISION, p
    try:
        yield
    finally:
        _DEFAULT_PRECISION = old


def _conv_out(n: int, k: int, stride: int) -> int:
    """Output extent of a k x k conv with padding k // 2 over an extent of n."""
    return (n + 2 * (k // 2) - k) // stride + 1


class Fold(NamedTuple):
    """A conv folded to one dense kernel: w[Cout,Cin,k,k] and b[Cout] in fp64."""
    w: torch.Tensor
    b: torch.Tensor
    k: int
    stride: int
    silu: bool


class V:
    """Channel window of an NHWC / PHASE4 activation buffer."""
    __slots__ = ("t", "B", "H", "W", "C_total", "c_off", "C", "dtype", "layout")

    def __init__(self, t, B_, H, W, C_total, c_off, C_, dtype, layout=L.NHWC):
        self.t, self.B, self.H, self.W, self.C_total, self.c_off, self.C, self.dtype, self.layout = \
            t, B_, H, W, C_total, c_off, C_, dtype, layout

    def sl(self, off: int, n: int) -> "V":
        assert 0 <= off and off + n <= self.C
        return V(self.t, self.B, self.H, self.W, self.C_total, self.c_off + off, n, self.dtype, self.layout)

    def c(self) -> L.View:
        return L.View(self.t.data_ptr(), self.dtype, self.layout, self.B, self.H, self.W, self.C_total, self.c_off, self.C)

    def same_window(self, o: "V") -> bool:
        return self.t is o.t and self.c_off == o.c_off and self.C == o.C


class VCat:
    """cat([Upsample(2, nearest)(up), rest], channels) that is never materialised (parser.py:159-171, common.py:32-33): the
    1x1 conv that consumes it reads ``up`` through yre_conv_desc.xu -- on the tcgen05 engine the upsample is a TMA
    addressing mode (tensor map with two stride-0 dimensions), so the 4x larger upsampled tensor is neither written nor
    read."""
    __slots__ = ("up", "rest")

    def __init__(self, up: V, rest: V):
        assert (2 * up.H, 2 * up.W, up.B) == (rest.H, rest.W, rest.B)
        self.up, self.rest = up, rest

    B = property(lambda s: s.rest.B)
    H = property(lambda s: s.rest.H)
    W = property(lambda s: s.rest.W)
    C = property(lambda s: s.up.C + s.rest.C)


def _null_view() -> L.View:
    return L.View(None, 0, 0, 0, 0, 0, 0, 0, 0)


class Plan:
    """A compiled launch list plus the tensors it owns."""

    def __init__(self, device: torch.device, batch: int, prec: str, arena: torch.Tensor | None = None,
                 wcache: dict | None = None, layout_only: bool = False):
        """arena: a uint8 device buffer the plan sub-allocates its activations and static outputs from, instead of
        tensors of its own (model.max_shape); wcache: packed weights shared with the other plans of that arena, by the
        modules they were folded from and their packing; layout_only: a plan that lays out its buffers (arena_end, trace)
        and neither allocates device memory nor records launches."""
        self.dry = device.type != "cuda"
        if self.dry and not (_ALLOW_CPU_DRY_RUN or layout_only):
            raise L.YreError("the yolo-re B200 path runs on CUDA tensors only (there is no CPU fallback)")
        self.arena, self.wcache, self.layout_only = arena, wcache, layout_only
        self.arena_end = 0            # bytes of the arena layout used so far (every plan counts them)
        self.lib = _LayoutOnly() if layout_only else L.lib()
        if not self.dry:
            with torch.cuda.device(device):
                L.check(self.lib.yre_device_check(), "device_check")
        self.trace: list[tuple] = []
        self.device, self.batch, self.prec = device, batch, prec
        self.dt, self.tdt = _DTYPES[prec]
        # tcgen05 convs encode TMA descriptors of device buffers, so a dry (host-buffer) plan takes the FFMA engine even
        # where a CUDA driver is present
        self.engine = L.ENGINE_AUTO if prec in ("bf16", "fp16") and not self.dry else L.ENGINE_FFMA
        self.names: dict[int, str] = {}          # id(module) -> qualified name, for error messages
        h = C.c_void_p()
        L.check(self.lib.yre_plan_create(C.byref(h)), "plan_create")
        self.h = h
        self.keep: list[torch.Tensor] = []
        self.act_bytes = 0
        self.weight_version = -1
        self.in_ptr = None            # image pointer currently bound
        self.out_tensors: list[torch.Tensor] = []   # externally visible outputs (rebindable)
        self.result = None
        self.shape_name = ""          # "B x H x W", for error messages

    def __del__(self):
        try:
            if getattr(self, "h", None):
                self.lib.yre_plan_destroy(self.h)
                self.h = None
        except Exception:
            pass

    # -- memory ---------------------------------------------------------------------------------------
    def empty(self, shape: tuple, tdt: torch.dtype, zero: bool = False) -> torch.Tensor:
        """A buffer the plan owns.  With an arena: the next ARENA_ALIGN-aligned bytes of it, in call order, holding
        whatever the last plan left there (zero is ignored: the kernels write every cell they read); without: a tensor
        of its own, zeroed when asked."""
        nbytes = math.prod(shape) * tdt.itemsize
        off = self.arena_end
        self.arena_end = off + -(-nbytes // ARENA_ALIGN) * ARENA_ALIGN
        if self.layout_only:
            t = torch.empty((), dtype=tdt).expand(shape)            # no storage: only the layout is wanted
        elif self.arena is not None:
            if off + nbytes > self.arena.numel():
                raise L.YreError(f"a plan for a {self.shape_name} input does not fit the shape arena of "
                                 f"{self.arena.numel()} bytes (it needs more than {off + nbytes})")
            t = self.arena[off:off + nbytes].view(tdt).view(shape)
        else:
            t = (torch.zeros if zero else torch.empty)(shape, dtype=tdt, device=self.device)
        self.keep.append(t)
        return t

    def alloc(self, H: int, W: int, Cn: int, dtype=None, layout=L.NHWC) -> V:
        dtype = self.dt if dtype is None else dtype
        tdt = _TORCH_DT[dtype]
        if layout == L.PHASE4:
            # cells without a source pixel hold 0: the stem and ADown kernels write them, the zeroing of a buffer of
            # the plan's own only repeats that
            t = self.empty((4, self.batch, (H + 1) // 2, (W + 1) // 2, Cn), tdt, zero=True)
        else:
            t = self.empty((self.batch, H, W, Cn), tdt)
        self.act_bytes += t.numel() * t.element_size()
        return V(t, self.batch, H, W, Cn, 0, Cn, dtype, layout)

    def dev(self, t: torch.Tensor, dtype) -> torch.Tensor:
        if self.layout_only:
            return t
        t = t.to(device=self.device, dtype=dtype).contiguous()
        self.keep.append(t)
        return t

    def pack(self, key: tuple | None, w: torch.Tensor, b: torch.Tensor, wdt: torch.dtype) -> tuple[torch.Tensor, torch.Tensor]:
        """Device weights [Cout][kh][kw][Cin] in wdt and fp32 bias of a fold.  key: the modules it was folded from and
        its packing; plans that share a weight cache upload each key once."""
        key = None if key is None or self.wcache is None else key + (wdt,)
        wb = self.wcache.get(key) if key is not None else None
        if wb is None:
            wb = self.dev(w.permute(0, 2, 3, 1), wdt), self.dev(b, torch.float32)
            if key is not None:
                self.wcache[key] = wb
        else:
            self.keep.extend(wb)
        return wb

    # -- weight folding ------------------------------------------------------------------------------------
    @staticmethod
    def _dense(w: torch.Tensor, groups: int) -> torch.Tensor:
        if groups == 1:
            return w
        co, cig, kh, kw = w.shape
        cog = co // groups
        d = torch.zeros(co, cig * groups, kh, kw, dtype=w.dtype, device=w.device)
        for g in range(groups):
            d[g * cog:(g + 1) * cog, g * cig:(g + 1) * cig] = w[g * cog:(g + 1) * cog]
        return d

    def fold(self, m) -> Fold:
        """The dense fp64 fold of a blocks.Conv / RepConv / nn.Conv2d.
        The folding arithmetic runs on the HOST in fp64 (the parameters are copied down once per compile): no torch
        element-wise kernels are launched on the device, only the folded weights are uploaded."""
        if isinstance(m, B.RepConv):
            f3, f1 = self.fold(m.conv1), self.fold(m.conv2)
            w = f3.w.clone()
            w[:, :, 1:2, 1:2] += f1.w
            return Fold(w, f3.b + f1.b, 3, f3.stride, isinstance(m.act, nn.SiLU))
        if isinstance(m, B.Conv):
            cv, bn = m.conv, m.bn
            k = cv.kernel_size[0]
            if cv.kernel_size[0] != cv.kernel_size[1] or cv.padding[0] != k // 2 or cv.dilation[0] != 1:
                raise L.YreError(f"unsupported conv geometry {cv}")
            w = cv.weight.detach().cpu().double()
            scale = bn.weight.detach().cpu().double() / torch.sqrt(bn.running_var.detach().cpu().double() + bn.eps)
            w = self._dense(w * scale[:, None, None, None], cv.groups)
            b = bn.bias.detach().cpu().double() - bn.running_mean.detach().cpu().double() * scale
            if not isinstance(m.act, (nn.SiLU, nn.Identity)):
                raise L.YreError(f"unsupported activation {m.act}")
            return Fold(w, b, k, cv.stride[0], isinstance(m.act, nn.SiLU))
        if isinstance(m, nn.Conv2d):
            k = m.kernel_size[0]
            w = self._dense(m.weight.detach().cpu().double(), m.groups)
            b = m.bias.detach().cpu().double() if m.bias is not None else torch.zeros(w.shape[0], dtype=torch.float64, device=w.device)
            return Fold(w, b, k, m.stride[0], False)
        raise L.YreError(f"cannot fold {type(m).__name__}")

    # -- op emission -------------------------------------------------------------------------------------
    def name_of(self, m) -> str:
        return self.names.get(id(m), type(m).__name__)

    def conv(self, x: V | VCat, w, b, k, stride, silu, out: V | None = None, res: V | None = None, out_dtype=None,
             name: str = "conv", key: tuple | None = None) -> V:
        cout, cin = w.shape[0], w.shape[1]
        if self.prec == "fp16":
            _check_f16_range(w, name)
        assert cin == x.C, (cin, x.C)
        xu = None
        if isinstance(x, VCat):
            assert k == 1 and stride == 1, "a virtual upsample+concat input needs a 1x1 stride-1 consumer"
            xu, x = x.up, x.rest
        Ho, Wo = _conv_out(x.H, k, stride), _conv_out(x.W, k, stride)
        if out is None:
            out = self.alloc(Ho, Wo, cout, dtype=out_dtype)
        assert (out.H, out.W, out.C) == (Ho, Wo, cout), ((out.H, out.W, out.C), (Ho, Wo, cout))
        wp, bp = self.pack(key, w, b, self.tdt)                 # [Cout][kh][kw][Cin]
        d = L.ConvDesc(x.c(), out.c(), res.c() if res is not None else _null_view(), wp.data_ptr(), bp.data_ptr(),
                       k, stride, L.ACT_SILU if silu else L.ACT_NONE, self.engine, xu.c() if xu is not None else _null_view())
        L.check(self.lib.yre_plan_add_conv(self.h, C.byref(d)), "plan_add_conv")
        self.trace.append(("conv", dict(x=x, y=out, res=res, w=wp, b=bp, k=k, stride=stride, silu=silu, xu=xu)))
        return out

    def conv_m(self, m, x: V, out: V | None = None, res: V | None = None, out_dtype=None) -> V:
        w, b, k, s, silu = self.fold(m)
        return self.conv(x, w, b, k, s, silu, out, res, out_dtype, name=self.name_of(m), key=("conv", self.name_of(m)))

    def conv_merged(self, ms, x: V, out: V | None = None) -> V:
        """Sibling convs on one input -> one GEMM with concatenated output channels."""
        fs = [self.fold(m) for m in ms]
        assert len({(f.k, f.stride, f.silu) for f in fs}) == 1
        return self.conv(x, torch.cat([f.w for f in fs]), torch.cat([f.b for f in fs]), fs[0].k, fs[0].stride, fs[0].silu, out,
                         name=" + ".join(self.name_of(m) for m in ms), key=("conv",) + tuple(self.name_of(m) for m in ms))

    def stem(self, m: B.Conv, x: torch.Tensor, phase4: bool) -> V:
        """x: the fp32 NCHW image batch, or uint8 [B,H,W,3] BGR frames (BGR->RGB, HWC->CHW and /255 of
        scripts/detect.py:223-227 are then fused into the kernel's gather)."""
        w, b, k, s, silu = self.fold(m)
        if self.prec == "fp16":                 # the tensor-core stem rounds its weights to fp16
            _check_f16_range(w, self.name_of(m))
        u8 = x.dtype == torch.uint8
        if u8:
            _, H, W, Cin = x.shape
        else:
            _, Cin, H, W = x.shape
        Bn = self.batch                          # x may hold fewer images: a plan compiled for a batch capacity
        Ho, Wo = _conv_out(H, 3, s), _conv_out(W, 3, s)
        out = self.alloc(Ho, Wo, w.shape[0], layout=L.PHASE4 if phase4 else L.NHWC)
        wp, bp = self.pack(("stem", self.name_of(m)), w, b, torch.float32)
        d = L.StemDesc(None if u8 else x.data_ptr(), Bn, Cin, H, W, out.c(), wp.data_ptr(), bp.data_ptr(), s,
                       L.ACT_SILU if silu else L.ACT_NONE, x.data_ptr() if u8 else None)
        L.check(self.lib.yre_plan_add_stem(self.h, C.byref(d)), "plan_add_stem")
        self.trace.append(("stem", dict(x=x, y=out, w=wp, b=bp, stride=s, silu=silu, u8=u8)))
        return out

    def copy(self, src: V, dst: V) -> None:
        v = src.c()
        L.check(self.lib.yre_plan_add_cbfuse_sum(self.h, None, 0, C.byref(v), C.byref(dst.c())), "plan_add_copy")
        self.trace.append(("cbfuse", dict(srcs=[], target=src, y=dst)))

    # -- blocks ------------------------------------------------------------------------------------------
    def csp(self, m: B.RepNCSP, x: V) -> V:
        h = m.conv1.conv.out_channels
        T = self.conv_merged([m.conv1, m.conv2], x)                 # [t | b]
        t = T.sl(0, h)
        for bt in m.bottlenecks:
            u = self.conv_m(bt.conv1, t)                            # RepConv folded to one 3x3
            self.conv_m(bt.conv2, u, out=t, res=t if bt.add else None)   # t = t + silu(conv(u)), in place
        return self.conv_m(m.conv3, T)

    def elan(self, m: B.RepNCSPELAN4, x: V, out: V | None) -> V:
        h = m.conv_in.conv.out_channels
        c = m.block1[1].conv.out_channels
        cat = self.alloc(x.H, x.W, h + 2 * c)
        self.conv_m(m.conv_in, x, out=cat.sl(0, h))
        y = cat.sl(h // 2, h - h // 2)                              # chunk(2,1)[1]
        off = h
        for blk in (m.block1, m.block2):
            v = self.csp(blk[0], y)
            y = self.conv_m(blk[1], v, out=cat.sl(off, c))
            off += c
        return self.conv_m(m.conv_out, cat, out=out)

    def adown(self, m: B.ADown, x: V, out: V | None) -> V:
        half = x.C // 2
        co = m.conv_stride.conv.out_channels
        Ho, Wo = _conv_out(x.H - 1, 3, 2), _conv_out(x.W - 1, 3, 2)      # 2x2 average pool, stride 1, then 3x3 / 2
        lo = self.alloc(x.H - 1, x.W - 1, half, layout=L.PHASE4)
        hi = self.alloc(Ho, Wo, half)
        L.check(self.lib.yre_plan_add_adown_prepool(self.h, C.byref(x.c()), C.byref(lo.c()), C.byref(hi.c())), "plan_add_adown")
        self.trace.append(("adown", dict(x=x, lo=lo, hi=hi)))
        if out is None:
            out = self.alloc(Ho, Wo, 2 * co)
        self.conv_m(m.conv_stride, lo, out=out.sl(0, co))
        self.conv_m(m.conv_pool, hi, out=out.sl(co, co))
        return out

    def sppelan(self, m: B.SPPELAN, x: V, out: V | None) -> V:
        h = m.conv_in.conv.out_channels
        cat = self.alloc(x.H, x.W, 4 * h)
        y0 = self.conv_m(m.conv_in, x, out=cat.sl(0, h))
        L.check(self.lib.yre_plan_add_spp_maxpool(self.h, C.byref(y0.c()), C.byref(cat.sl(h, h).c()),
                                                  C.byref(cat.sl(2 * h, h).c()), C.byref(cat.sl(3 * h, h).c())), "plan_add_spp")
        self.trace.append(("spp", dict(x=y0, y5=cat.sl(h, h), y9=cat.sl(2 * h, h), y13=cat.sl(3 * h, h))))
        return self.conv_m(m.conv_out, cat, out=out)

    def upsample(self, x: V, out: V | None) -> V:
        if out is None:
            out = self.alloc(2 * x.H, 2 * x.W, x.C)
        L.check(self.lib.yre_plan_add_upsample2x(self.h, C.byref(x.c()), C.byref(out.c())), "plan_add_upsample")
        self.trace.append(("upsample", dict(x=x, y=out)))
        return out

    def cblinear(self, m: B.CBLinear, x: V) -> tuple[V, ...]:
        y = self.conv_m(m.conv, x)
        outs, off = [], 0
        for n in m.out_channels_list:
            outs.append(y.sl(off, n))
            off += n
        return tuple(outs)

    def cbfuse(self, m: B.CBFuse, ins: list, out: V | None) -> V:
        tgt = ins[-1]
        srcs = [ins[i][m.idx[i]] for i in range(len(ins) - 1)]
        if out is None:
            out = self.alloc(tgt.H, tgt.W, tgt.C)
        arr = (L.View * max(1, len(srcs)))(*[s.c() for s in srcs])
        L.check(self.lib.yre_plan_add_cbfuse_sum(self.h, arr, len(srcs), C.byref(tgt.c()), C.byref(out.c())), "plan_add_cbfuse")
        self.trace.append(("cbfuse", dict(srcs=srcs, target=tgt, y=out)))
        return out

    def concat(self, ins: list[V], out: V | None) -> V:
        if out is None:
            out = self.alloc(ins[0].H, ins[0].W, sum(v.C for v in ins))
        off = 0
        for v in ins:
            dst = out.sl(off, v.C)
            if not v.same_window(dst):
                self.copy(v, dst)
            off += v.C
        return out

    def towers(self, box, cls, dfl, feats: list[V], strides: list[float], nc: int):
        """One head: per level first 3x3 of box and cls (merged into one GEMM on the small levels), the two
        towers, fp32 raw logits; then K6."""
        raws = self.tower_convs(box, cls, feats, nc)
        y, d = self.decode_desc(raws, strides, nc, dfl)
        L.check(self.lib.yre_plan_add_decode(self.h, C.byref(d)), "plan_add_decode")
        self.trace.append(("decode", dict(raws=raws, strides=list(strides), nc=nc, dfl_w=list(d.dfl_w), y=y)))
        return y, raws

    def tower_convs(self, box, cls, feats: list[V], nc: int) -> list[V]:
        """The box and class towers of every level: the fp32 raw-logit windows [B,H,W,64+nc]."""
        raws = []
        for i, f in enumerate(feats):
            c2 = box[i][0].conv.out_channels
            c3 = cls[i][0].conv.out_channels
            # class count padded to a multiple of 16 (zero weights, zero bias): any num_classes keeps 16-byte rows for the
            # decode kernel and a tcgen05-eligible Cout; the padding channels are never read or returned
            ncp = -(-nc // 16) * 16
            raw_full = self.alloc(f.H, f.W, 4 * REG_MAX + ncp, dtype=L.F32)
            raw = raw_full.sl(0, 4 * REG_MAX + nc)
            if c3 % 128 == 0 and self.batch * f.H * f.W >= 65536:
                # large level: separate GEMMs.  The 256-wide cls conv takes CTA pairs with 256-column tiles and the box conv
                # the paired halo kernel (80x80) or 64-wide tiles; a merged 64+256 = 320-channel GEMM runs as two unpaired
                # 160-wide tiles (3x3 512->320 @40x40 B64: 337 us merged, 106 + 174 us separate).  Small levels (fewer than
                # 64 Ki output pixels) stay merged: one launch less is worth more there (20x20 B64: 95 vs 99 us)
                hb_in, hc_in = self.conv_m(box[i][0], f), self.conv_m(cls[i][0], f)
            else:
                h1 = self.conv_merged([box[i][0], cls[i][0]], f)
                hb_in, hc_in = h1.sl(0, c2), h1.sl(c2, c3)
            hb = self.conv_m(box[i][1], hb_in)
            self.conv_m(box[i][2], hb, out=raw.sl(0, 4 * REG_MAX))
            hc = self.conv_m(cls[i][1], hc_in)
            fc = self.fold(cls[i][2])
            if ncp != nc:
                fc = fc._replace(w=torch.cat([fc.w, fc.w.new_zeros((ncp - nc,) + tuple(fc.w.shape[1:]))]),
                                 b=torch.cat([fc.b, fc.b.new_zeros(ncp - nc)]))
            self.conv(hc, fc.w, fc.b, fc.k, fc.stride, fc.silu, out=raw_full.sl(4 * REG_MAX, ncp), name=self.name_of(cls[i][2]),
                      key=("conv", self.name_of(cls[i][2]), "classes padded to", ncp))
            raws.append(raw)
        return raws

    def decode_desc(self, raws: list[V], strides: list[float], nc: int, dfl) -> tuple[torch.Tensor, L.DecodeDesc]:
        """y [B,A,4+nc] (allocated here) and the K6 descriptor that fills it from the raw logits"""
        A = sum(r.H * r.W for r in raws)
        y = self.empty((self.batch, A, 4 + nc), torch.float32)
        d = L.DecodeDesc()
        for i, r in enumerate(raws):
            d.raw[i] = r.c()
            d.stride[i] = float(strides[i])
        d.levels, d.nc = len(raws), nc
        wd = dfl.conv.weight.detach().float().flatten().cpu().tolist()
        for k in range(REG_MAX):
            d.dfl_w[k] = wd[k]
        d.y = y.data_ptr()
        return y, d

    def segment(self, m: SegmentDFL, feats: list[V], strides: list[float]):
        """A segmentation head: the detection towers exactly as DetectDFL's, then the prototype branch on the first level
        (K1 convs around a K5 nearest upsample: its consumer is a 3x3 conv, which cannot read it through a tensor map;
        the last conv writes fp32 NHWC [B,H/4,W/4,nm]), then the mask-coefficient towers (fp32 [B,Hl,Wl,nm]), then K6
        writing y and mc [B,A,nm] in one launch."""
        if m.num_masks != 32:
            raise L.YreError(f"segmentation head with {m.num_masks} masks: the kernels take 32 mask coefficients only")
        nc = m.num_classes
        raws = self.tower_convs(m.box_convs, m.cls_convs, feats, nc)
        pr = m.proto
        proto = self.conv_m(pr.cv3, self.conv_m(pr.cv2, self.upsample(self.conv_m(pr.cv1, feats[0]), None)), out_dtype=L.F32)
        masks = []
        for i, f in enumerate(feats):
            t = m.mask_convs[i]
            masks.append(self.conv_m(t[2], self.conv_m(t[1], self.conv_m(t[0], f)), out_dtype=L.F32))
        y, d = self.decode_desc(raws, strides, nc, m.dfl)
        mc = self.empty((self.batch, y.shape[1], m.num_masks), torch.float32)
        dm = L.DecodeMasksDesc(d, (L.View * 8)(*[v.c() for v in masks]), m.num_masks, mc.data_ptr())
        L.check(self.lib.yre_plan_add_decode_masks(self.h, C.byref(dm)), "plan_add_decode_masks")
        # recorded as a decode (what the detection path checks) with the mask views and mc alongside
        self.trace.append(("decode", dict(raws=raws, strides=list(strides), nc=nc, dfl_w=list(d.dfl_w), y=y, masks=masks, mc=mc)))
        return ("segment", y, [raws, mc, proto])

    def detect(self, m, feats: list[V], main_only: bool = False):
        strides = m.stride.tolist()
        if isinstance(m, SegmentDFL):
            return self.segment(m, feats, strides)
        if isinstance(m, DetectDFL):
            y, raws = self.towers(m.box_convs, m.cls_convs, m.dfl, feats, strides, m.num_classes)
            return ("single", y, raws)
        if main_only:                      # feats = the main half only; result looks like a single head's
            y, raws = self.towers(m.main_box_convs, m.main_cls_convs, m.dfl2, feats, strides, m.num_classes)
            return ("single", y, raws)
        Ln = m.num_levels
        ya, ra = self.towers(m.aux_box_convs, m.aux_cls_convs, m.dfl, feats[:Ln], strides, m.num_classes)
        ym, rm = self.towers(m.main_box_convs, m.main_cls_convs, m.dfl2, feats[Ln:], strides, m.num_classes)
        return ("dual", [ya, ym], [ra, rm])

    def block(self, m, x, out: V | None = None):
        """Emits any supported module; x is a V, a tuple of V or a list of those."""
        if isinstance(m, (B.Conv, B.RepConv)):
            return self.conv_m(m, x, out=out)
        if isinstance(m, B.RepNBottleneck):
            u = self.conv_m(m.conv1, x)
            return self.conv_m(m.conv2, u, out=out, res=x if m.add else None)
        if isinstance(m, B.RepNCSP):
            return self.csp(m, x)
        if isinstance(m, B.RepNCSPELAN4):
            return self.elan(m, x, out)
        if isinstance(m, B.ADown):
            return self.adown(m, x, out)
        if isinstance(m, B.SPPELAN):
            return self.sppelan(m, x, out)
        if isinstance(m, B.Upsample):
            return self.upsample(x, out)
        if isinstance(m, B.Silence):
            return x
        if isinstance(m, B.Concat):
            return self.concat(list(x), out)
        if isinstance(m, B.CBLinear):
            return self.cblinear(m, x)
        if isinstance(m, B.CBFuse):
            return self.cbfuse(m, list(x), out)
        if isinstance(m, (DetectDFL, DualDetectDFL)):
            return self.detect(m, list(x))
        raise L.YreError(f"module {type(m).__name__} is not on the B200 hot path")

    # -- running -----------------------------------------------------------------------------------------------
    def rebind(self, old: int, new: int) -> None:
        r = self.lib.yre_plan_rebind(self.h, old, new)
        if r < 0:
            L.check(r, "plan_rebind")

    def run(self, n: int | None = None) -> None:
        """Runs the launch list for all ``batch`` images, or for the first n of them (yre_plan_run_batch: bit-identical
        results for those n, no row of a later image is written, shorter launches)."""
        s = torch.cuda.current_stream(self.device).cuda_stream
        if n is None:
            L.check(self.lib.yre_plan_run(self.h, s), "plan_run")
        else:
            L.check(self.lib.yre_plan_run_batch(self.h, n, s), "plan_run_batch")

    @property
    def capacity(self) -> int:
        """The most images one run computes (the batch every op was recorded for)."""
        r = self.lib.yre_plan_batch_capacity(self.h)
        if r < 0:
            L.check(r, "plan_batch_capacity")
        return r

    @property
    def num_launches(self) -> int:
        return self.lib.yre_plan_num_launches(self.h)

    @property
    def num_tcgen05(self) -> int:
        return self.lib.yre_plan_num_tcgen05(self.h)

    def op_table(self):
        n = self.lib.yre_plan_num_ops(self.h)
        fl = (C.c_double * n)()
        self.lib.yre_plan_op_flops(self.h, fl, n)
        return [(self.lib.yre_plan_op_name(self.h, i).decode(), fl[i]) for i in range(n)]

    def op_variants(self) -> list[str]:
        """Kernel variant + tiling of every recorded op (yre_plan_op_variant), same order as op_table()."""
        out, buf = [], C.create_string_buffer(160)
        for i in range(self.lib.yre_plan_num_ops(self.h)):
            L.check(self.lib.yre_plan_op_variant(self.h, i, buf, 160), "plan_op_variant")
            out.append(buf.value.decode())
        return out

    def op_descriptions(self) -> list[str]:
        """Human-readable shape of every recorded op (same order as op_table())."""
        out = []
        for kind, a in self.trace:
            if kind == "conv":
                x, y = a["x"], a["y"]
                cin = x.C + (a["xu"].C if a.get("xu") is not None else 0)
                out.append(f"conv{a['k']}x{a['k']}s{a['stride']} {cin}->{y.C} @{y.H}x{y.W} B{y.B}"
                           f"{' +res' if a['res'] is not None else ''}{' f32out' if y.dtype == L.F32 else ''}"
                           f"{' up2x' if a.get('xu') is not None else ''}")
            elif kind == "stem":
                y = a["y"]
                out.append(f"stem {'u8 ' if a.get('u8') else ''}3->{y.C} @{y.H}x{y.W} B{y.B}")
            elif kind in ("adown", "spp", "upsample"):
                x = a["x"]
                out.append(f"{kind} C{x.C} @{x.H}x{x.W} B{x.B}")
            else:
                out.append(kind)
        return out

    def run_op(self, i: int) -> None:
        s = torch.cuda.current_stream(self.device).cuda_stream
        L.check(self.lib.yre_plan_run_op(self.h, i, s), "plan_run_op")


# ------------------------------------------------------------------------------------------------------------
def _out_shape(m, ins: list[tuple[int, int, int]]) -> tuple[int, int, int]:
    """(H, W, C) of a layer's output from the (H, W, C) of its inputs; a CBLinear's C is that of its last chunk."""
    H, W, Cn = ins[-1] if isinstance(m, B.CBFuse) else ins[0]
    if isinstance(m, B.Conv):
        k, s = m.conv.kernel_size[0], m.conv.stride[0]
        return _conv_out(H, k, s), _conv_out(W, k, s), m.conv.out_channels
    if isinstance(m, B.ADown):
        return _conv_out(H - 1, 3, 2), _conv_out(W - 1, 3, 2), 2 * m.conv_stride.conv.out_channels
    if isinstance(m, B.Upsample):
        return 2 * H, 2 * W, Cn
    if isinstance(m, (B.RepNCSPELAN4, B.SPPELAN)):
        return H, W, m.conv_out.conv.out_channels
    if isinstance(m, B.Concat):
        return H, W, sum(c for _, _, c in ins)
    if isinstance(m, B.CBLinear):
        return H, W, m.out_channels_list[-1]
    return H, W, Cn


class Wire(NamedTuple):
    """How one layer sits in the plan, decided before anything is allocated."""
    srcs: list[str]                  # layers it reads ("input": the image), past any Silence; a main_only head: its main half
    H: int                           # output extent and channels
    W: int
    C: int
    dest: tuple[str, int] | None     # (concat, channel offset) it writes its output into
    lazy: bool                       # an Upsample its concat's consumers read in place (VCat): it emits nothing
    needed: bool                     # False: main_only prunes it
    phase4: bool                     # a stem that writes parity planes for the stride-2 3x3 conv reading it


def wire_model(model, H: int, W: int, Cin: int, main_only: bool | None = None) -> dict[str, Wire]:
    """The wiring of model.layers / model.connections for an H x W x Cin image, by layer name; it touches no tensor.
    main_only: None follows model.main_only."""
    layers, names, conn = model.layers, list(model.layers.keys()), model.connections
    srcs = {n: ([conn[n]] if isinstance(conn[n], str) else list(conn[n])) for n in names}
    consumers: dict[str, list[str]] = {n: [] for n in ["input", *names]}
    shape = {"input": (H, W, Cin)}
    for n in names:
        for s in srcs[n]:
            consumers[s].append(n)
        shape[n] = _out_shape(layers[n], [shape[s] for s in srcs[n]])
    # Upsample -> Concat([up, skip]) -> RepNCSPELAN4: the ELAN's first op is a 1x1 conv over the whole concat, which can
    # read the half-resolution tensor directly (VCat / yre_conv_desc.xu).  Such an Upsample emits no kernel and its half
    # of the concat buffer is never allocated.
    lazy: dict[str, str] = {}
    if getattr(model, "fuse_upsample", True):
        for n in names:
            if not (isinstance(layers[n], B.Concat) and len(srcs[n]) >= 2):
                continue
            u = srcs[n][0]
            if (u != "input" and isinstance(layers[u], B.Upsample) and consumers[u] == [n] and u not in srcs[n][1:]
                    and consumers[n] and all(isinstance(layers[c], B.RepNCSPELAN4) and srcs[c] == [n] for c in consumers[n])
                    and shape[u][2] % 64 == 0 and (shape[n][2] - shape[u][2]) % 64 == 0):
                lazy[u] = n
    # where should a layer write?  -> into the slice of the first Concat that consumes it, if its block takes a window
    windowed = (B.Conv, B.RepNCSPELAN4, B.ADown, B.SPPELAN, B.Upsample, B.CBFuse)
    dest: dict[str, tuple[str, int]] = {}
    for n in names:
        if isinstance(layers[n], B.Concat):
            off = 0
            for s in srcs[n]:
                if lazy.get(s) == n:
                    continue
                if s not in dest and s != "input" and isinstance(layers[s], windowed):
                    dest[s] = (n, off)
                off += shape[s][2]
    # main_only (opt-in, SURVEY.md 8f row 2): every caller of a dual-head model drops the auxiliary half
    # (scripts/detect.py:239-241, eval/evaluator.py:107-109); compile only what the main towers need.
    needed, head = set(names), names[-1]
    if not isinstance(layers[head], (DetectDFL, DualDetectDFL)):
        raise L.YreError("the last layer of the model must be a detection head")
    if _main_only(model, main_only) and isinstance(layers[head], DualDetectDFL):
        srcs[head] = srcs[head][layers[head].num_levels:]
        needed = {head}
        for n in reversed(names):                 # a layer comes after every layer it reads
            if n in needed:
                needed.update(srcs[n])
    wire: dict[str, Wire] = {}
    for n in names:
        # a Silence passes its input on: it is nobody's source and emits nothing
        srcs[n] = [srcs[s][0] if s != "input" and isinstance(layers[s], B.Silence) else s for s in srcs[n]]
        c = consumers[n]
        phase4 = ("input" in srcs[n] and len(c) == 1 and isinstance(layers[c[0]], B.Conv)
                  and layers[c[0]].conv.stride[0] == 2 and layers[c[0]].conv.kernel_size[0] == 3 and n not in dest
                  and model.precision in ("bf16", "fp16"))
        wire[n] = Wire(srcs[n], *shape[n], dest.get(n), n in lazy, n in needed, phase4)
    return wire


def _weights_version(model: nn.Module) -> int:
    """Fingerprint of the weights a plan was folded from: storage address and in-place version counter of every
    parameter and buffer.  Catches optimizer steps, ``load_state_dict``, ``p.copy_()``, ``p.data = new`` ...;
    writes THROUGH ``.data`` (``p.data.copy_()``, ``bias.data[:] = ...``) bump no counter and move no storage --
    after such an edit call ``model.invalidate()``."""
    ts = model.__dict__.get("_wt_tensors")
    if ts is None or len(ts[1]) != ts[0]:
        # the module-tree walk is the expensive part (~1 ms for 937 tensors): do it once per structure
        lst = list(model.parameters()) + list(model.buffers())
        ts = (len(lst), lst)
        model.__dict__["_wt_tensors"] = ts
    return hash(tuple([(t.data_ptr(), t._version) for t in ts[1]]))


def _main_only(model, main_only: bool | None = None) -> bool:
    """main_only, or model.main_only when it is None"""
    return bool(getattr(model, "main_only", False)) if main_only is None else bool(main_only)


def compile_model(model, x: torch.Tensor, capacity: int | None = None, main_only: bool | None = None,
                  arena: torch.Tensor | None = None, wcache: dict | None = None, layout_only: bool = False) -> Plan:
    """Compiles the whole YOLO graph for x's shape/device (x: fp32 [B,C,H,W] or uint8 [B,H,W,3] BGR frames).
    capacity: compile for that many images instead of x's B (x may hold fewer; the plan runs any 1..capacity of them).
    main_only: None follows model.main_only.  arena, wcache, layout_only: see Plan."""
    if x.dtype == torch.uint8:
        Bn, H, W, Cin = x.shape
    else:
        Bn, Cin, H, W = x.shape
    Bn = Bn if capacity is None else capacity
    wire = wire_model(model, H, W, Cin, main_only)
    p = Plan(x.device, Bn, model.precision, arena, wcache, layout_only)
    p.names = {id(m): n for n, m in model.named_modules()}
    p.shape_name = f"{Bn} x {H} x {W}"

    @cache
    def cat_buf(n: str) -> V:
        """the buffer of concat n, allocated at first use; it holds no channels of a lazy upsample"""
        w = wire[n]
        return p.alloc(w.H, w.W, w.C - sum(wire[s].C for s in w.srcs if wire[s].lazy))

    vals: dict[str, object] = {}
    for n, m in model.layers.items():
        w = wire[n]
        if not w.needed or w.lazy or isinstance(m, B.Silence):
            continue
        if "input" in w.srcs:
            if not (isinstance(m, B.Conv) and m.conv.kernel_size[0] == 3 and Cin <= 4 and m.conv.groups == 1):
                raise L.YreError(f"layer '{n}' reads the image but is not a 3x3 Conv (unsupported stem)")
            vals[n] = p.stem(m, x, w.phase4)
            continue
        ins = [vals[s] for s in w.srcs if not wire[s].lazy]
        if isinstance(m, (DetectDFL, DualDetectDFL)):
            p.result = p.detect(m, ins, main_only=_main_only(model, main_only))
        elif isinstance(m, B.Concat):
            vals[n] = p.concat(ins, cat_buf(n))
            up = wire[w.srcs[0]]
            if up.lazy:                              # the Upsample is folded into the consumers' first conv
                vals[n] = VCat(vals[up.srcs[0]], vals[n])
        else:
            out = cat_buf(w.dest[0]).sl(w.dest[1], w.C) if w.dest else None
            vals[n] = p.block(m, ins[0] if isinstance(model.connections[n], str) else ins, out)
    p.vals = vals                 # per-layer output windows (debugging / stage-wise tests)
    p.in_ptr = x.data_ptr()
    p.weight_version = _weights_version(model)
    return p


def _fresh(p: Plan, o, rows: int | None = None):
    """o (an output tensor, a raw-logit window or a list of them) re-pointed to new tensors that the plan writes, of
    `rows` images (default: the plan's batch; a run of n images writes rows [:n] only)"""
    if isinstance(o, list):
        return [_fresh(p, e, rows) for e in o]
    if isinstance(o, V):
        o.t = _fresh(p, o.t, rows)
        return o
    n = torch.empty((p.batch if rows is None else rows,) + tuple(o.shape[1:]), dtype=o.dtype, device=o.device)
    p.rebind(o.data_ptr(), n.data_ptr())
    return n


def _rows(o) -> int:
    """images held by the output tensors of a head result (y, or the first of a dual head's)"""
    return _rows(o[0]) if isinstance(o, list) else o.shape[0]


def _replay_graph(p: Plan, x: torch.Tensor, n: int | None = None) -> None:
    """Static-buffer mode: the whole launch list (incl. its programmatic-dependent-launch edges) is captured once per
    input BUFFER (and image count n of a plan with a batch capacity, None: the whole batch) into a CUDA graph and
    replayed -- no per-launch CPU work, ~1 us between kernels.  Meant for callers that reuse a few input buffers (a
    double-buffered upload ring): every new buffer address costs a warm-up run and a capture.  At most 8 (graph, buffer)
    pairs are held; the oldest pair is dropped together, so a caller that passes a fresh tensor every time pays the
    capture each call but does not accumulate memory."""
    graphs = p.__dict__.setdefault("graphs", {})
    key = (x.data_ptr(), n)
    ent = graphs.get(key)
    g = ent[0] if ent is not None else None
    if g is None:
        cur = torch.cuda.current_stream(p.device)
        side = torch.cuda.Stream(p.device)
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            p.run(n)                                 # warm-up outside capture: one-time function attributes, lazy module load
        cur.wait_stream(side)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            p.run(n)
        if len(graphs) >= 8:
            graphs.pop(next(iter(graphs)))           # drops the graph AND the input buffer it pinned
        graphs[key] = (g, x)                         # the captured graph reads this buffer: keep it alive with the graph
    g.replay()


def model_forward(model, x: torch.Tensor, augment: bool = False):
    if not x.is_cuda:
        raise L.YreError("the yolo-re B200 path runs on CUDA tensors only (there is no CPU fallback)")
    if x.dim() != 4:
        raise ValueError("expected input [B,C,H,W] (or uint8 frames [B,H,W,3])")
    if x.dtype == torch.uint8:
        # extension of the reference API: cv2-layout frames (uint8 HWC, BGR) already letterboxed to the model size;
        # scripts/detect.py:223-227 (BGR->RGB, HWC->CHW, /255) is fused into the first conv's gather
        if x.shape[3] != 3:
            raise ValueError("uint8 input must be [B,H,W,3] BGR frames")
        x = x.contiguous()
    else:
        x = x.contiguous().float()
    cap = _capacity(model, x)
    max_hw = _max_shape(model, x)
    if augment:
        _, head = model._detect_layer()
        if isinstance(head, SegmentDFL):
            raise ValueError("augment=True: test-time augmentation is defined for detection heads only (upstream has no "
                             "segmentation TTA)")
        from .tta import forward_augment
        with torch.cuda.device(x.device):
            return forward_augment(model, x, cap, max_hw)
    return run_forward(model, x, cap, max_hw=max_hw)


def run_forward(model, x: torch.Tensor, cap: int | None, main_only: bool | None = None, tag=None,
                max_hw: tuple[int, int] | None = None):
    """forward's value for x (checked and made contiguous by model_forward) on its plan, compiled at first use.
    cap: model.max_batch (checked against x); main_only: None follows model.main_only; tag: extends the plan key, so
    that a caller's plan is never shared with another input of the same shape (the branches of forward_augment);
    max_hw: the largest input of x's shape arena (model.max_shape, checked against x; None: the plan owns its buffers)."""
    key = plan_key(model, x, main_only) + ((tag,) if tag is not None else ())
    p = model._plans.get(key)
    if p is not None and model.check_weights and p.weight_version != _weights_version(model):
        p = None
    n = None if cap is None else x.shape[0]          # None: the plan's whole batch, x's own
    with torch.cuda.device(x.device):
        if p is None:
            arena, wcache = _arena(model, x, cap, main_only, tag, max_hw) if max_hw is not None else (None, None)
            p = compile_model(model, x, capacity=cap, main_only=main_only, arena=arena, wcache=wcache)
            model._plans[key] = p
        elif p.in_ptr != x.data_ptr():
            p.rebind(p.in_ptr, x.data_ptr())
            p.in_ptr = x.data_ptr()
        kind, y, raws = p.result
        if model.fresh_outputs:
            # the reference returns new tensors every call: re-point the plan's outputs (to n-image tensors for a run of
            # n images -- nothing past row n is written)
            p.result = (kind, _fresh(p, y, n), _fresh(p, raws, n))
        elif _rows(y) != p.batch:
            # static buffers after fresh outputs of fewer images: back to buffers that hold the whole batch
            p.result = (kind, _fresh(p, y), _fresh(p, raws))
        if getattr(model, "use_cuda_graph", False) and not model.fresh_outputs:
            _replay_graph(p, x, n)
        else:
            p.run(n)
    p.x_keepalive = x
    out = _head_outputs(p.result)
    return out if n is None or model.fresh_outputs else _first_rows(out, n)


def _capacity(model, x: torch.Tensor) -> int | None:
    """model.max_batch after checking x's batch against it (None: no capacity, plans are compiled per batch size)"""
    cap = getattr(model, "max_batch", None)
    if cap is None:
        return None
    if int(cap) < 1:
        raise ValueError(f"model.max_batch must be a positive image count or None (got {cap})")
    if not 1 <= x.shape[0] <= cap:
        raise ValueError(f"a forward of {x.shape[0]} images: this model runs 1..{cap} images per forward "
                         f"(model.max_batch = {cap})")
    return int(cap)


def _max_shape(model, x: torch.Tensor) -> tuple[int, int] | None:
    """model.max_shape as (H, W) after checking it and x's height and width against it (None: every plan owns its
    buffers)"""
    ms = getattr(model, "max_shape", None)
    if ms is None:
        return None
    if getattr(model, "max_batch", None) is None:
        raise ValueError("model.max_shape needs model.max_batch: the shape arena is sized for model.max_batch images of "
                         "model.max_shape, so set both (or model.max_shape = None)")
    if len(ms) != 2 or min(int(v) for v in ms) < 1:
        raise ValueError(f"model.max_shape must be a (height, width) pair of positive extents or None (got {ms})")
    mh, mw = int(ms[0]), int(ms[1])
    H, W = (x.shape[1], x.shape[2]) if x.dtype == torch.uint8 else (x.shape[2], x.shape[3])
    if H > mh or W > mw:
        raise ValueError(f"a {H} x {W} input: this model runs inputs of up to {mh} x {mw} (model.max_shape = {ms})")
    return mh, mw


def arena_bytes(model, Cin: int, H: int, W: int, capacity: int, main_only: bool | None = None) -> int:
    """Bytes of a shape arena for plans of up to capacity images of at most H x W: the buffer layout of that largest
    plan.  Every buffer of a plan grows with the input extents, and a smaller input never lays out more buffers."""
    x = torch.empty((), dtype=torch.float32).expand(capacity, Cin, H, W)       # no storage: only its shape is read
    return compile_model(model, x, capacity, main_only, layout_only=True).arena_end


def _arena(model, x: torch.Tensor, cap: int, main_only: bool | None, tag, max_hw: tuple[int, int]):
    """(arena, weight cache) of x's plan.  One arena per precision, main_only, fuse_upsample, plan tag and device (and
    capacity and maximum shape), allocated at first use for cap images of max_hw and never reallocated, so CUDA graphs
    captured on its plans stay valid; the input dtype is not part of the key (it changes no buffer).  The weight cache
    of the device holds the packed weights of every plan with an arena, for the weights' current version."""
    key = (model.precision, _main_only(model, main_only), bool(getattr(model, "fuse_upsample", True)), tag,
           x.device.index, cap, max_hw)
    arena = model._arenas.get(key)
    if arena is None:
        Cin = x.shape[3] if x.dtype == torch.uint8 else x.shape[1]
        arena = torch.empty(arena_bytes(model, Cin, *max_hw, cap, main_only), dtype=torch.uint8, device=x.device)
        model._arenas[key] = arena
    ver = _weights_version(model)
    wc = model._arena_weights.get(x.device.index)
    if wc is None or wc[0] != ver:
        wc = model._arena_weights[x.device.index] = (ver, {})
    return arena, wc[1]


def plan_key(model, x: torch.Tensor, main_only: bool | None = None) -> tuple:
    """The key of the plan model_forward runs x on: x's shape (its batch replaced by model.max_batch when that is set),
    dtype and device, and the engine settings that change what is compiled (main_only: None follows model.main_only),
    and model.max_shape when that is set (its plans take their buffers from a shape arena)."""
    cap = getattr(model, "max_batch", None)
    shape = tuple(x.shape) if cap is None else (int(cap),) + tuple(x.shape[1:])
    key = (shape, x.dtype, x.device.index, model.precision, bool(getattr(model, "fuse_upsample", True)),
           _main_only(model, main_only))
    ms = getattr(model, "max_shape", None)
    return key if ms is None else key + (("max_shape", tuple(int(v) for v in ms)),)


def _first_rows(obj, n: int):
    """rows [:n] of every tensor of a forward's value"""
    if isinstance(obj, torch.Tensor):
        return obj[:n]
    return type(obj)(_first_rows(o, n) for o in obj)


def _head_outputs(result):
    """forward's value for a head result: (y[B,4+nc,A], [raw_i NCHW]), or ([y_aux, y_main], [raws_aux, raws_main]), or
    for a segmentation head (y[B,4+nc,A], ([raw_i NCHW], mc[B,nm,A], proto[B,nm,H/4,W/4])), mc and proto views of
    their A x nm and NHWC buffers"""
    kind, y, raws = result
    if kind == "single":
        return y.permute(0, 2, 1), [_raw_nchw(r) for r in raws]
    if kind == "segment":
        rs, mc, proto = raws
        return y.permute(0, 2, 1), ([_raw_nchw(r) for r in rs], mc.permute(0, 2, 1), _raw_nchw(proto))
    return [t.permute(0, 2, 1) for t in y], [[_raw_nchw(r) for r in rs] for rs in raws]


def _raw_nchw(r: "V") -> torch.Tensor:
    """[B,C,H,W] view of a raw-logit or prototype buffer (a raw buffer's channel count may be padded, towers())."""
    t = r.t if r.C == r.C_total else r.t[..., r.c_off:r.c_off + r.C]
    return t.permute(0, 3, 1, 2)


# ---- standalone block call (tests, teacher-forced stage checks) ----------------------------------------------
def _to_views(p: Plan, obj):
    if isinstance(obj, torch.Tensor):
        if not obj.is_cuda and not p.dry:
            raise L.YreError("the yolo-re B200 path runs on CUDA tensors only (there is no CPU fallback)")
        t = obj.contiguous().float()
        p.keep.append(t)
        Bn, Cn, H, W = t.shape
        v = p.alloc(H, W, Cn)
        L.check(p.lib.yre_plan_add_nchw_to_view(p.h, t.data_ptr(), C.byref(v.c())), "plan_add_nchw_to_view")
        p.trace.append(("nchw_to_view", dict(x=t, y=v)))
        return v
    if isinstance(obj, tuple):
        return tuple(_to_views(p, o) for o in obj)
    return [_to_views(p, o) for o in obj]


def _first_tensor(obj):
    return obj if isinstance(obj, torch.Tensor) else _first_tensor(obj[0])


def compile_module(m: nn.Module, x, prec: str | None = None):
    """Compiles one block / head for NCHW fp32 input(s).  Returns (plan, outputs); the outputs
    (NCHW fp32 tensors, same nesting as the reference module returns) are filled by plan.run()."""
    t0 = _first_tensor(x)
    p = Plan(t0.device, t0.shape[0], prec or _DEFAULT_PRECISION)
    p.names = {id(mm): n or type(m).__name__ for n, mm in m.named_modules()}
    if isinstance(m, B.Conv) and isinstance(x, torch.Tensor) and x.shape[1] <= 4 and m.conv.kernel_size[0] == 3:
        xin = x.contiguous().float()
        p.keep.append(xin)
        out = p.stem(m, xin, False)
    else:
        out = p.block(m, _to_views(p, x))

    def back(v):
        if isinstance(v, V):
            y = torch.empty((v.B, v.C, v.H, v.W), dtype=torch.float32, device=p.device)
            L.check(p.lib.yre_plan_add_view_to_nchw(p.h, C.byref(v.c()), y.data_ptr()), "plan_add_view_to_nchw")
            p.trace.append(("view_to_nchw", dict(x=v, y=y)))
            return y
        return tuple(back(o) for o in v)

    if isinstance(m, (DetectDFL, DualDetectDFL)):
        return p, _head_outputs(out)
    return p, back(out)


def run_module(m: nn.Module, x):
    """Eval-mode forward of one block / head on NCHW fp32 CUDA input(s); returns NCHW fp32."""
    if m.training:
        raise NotImplementedError("train-mode forward is outside the B200 inference path; call .eval()")
    t0 = _first_tensor(x)
    if not t0.is_cuda:
        raise L.YreError("the yolo-re B200 path runs on CUDA tensors only (there is no CPU fallback)")
    with torch.cuda.device(t0.device):
        p, res = compile_module(m, x)
        p.run()
        torch.cuda.current_stream(p.device).synchronize()   # the plan (and its buffers) die with this call
    return res
