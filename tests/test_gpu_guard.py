"""Out-of-bounds WRITE checks of every libyre kernel (the pool's GPUs do not allow compute-sanitizer -- its runs left devices
needing a reset -- so the memcheck pass SURVEY.md section 5 asks for is restated as guard bands): every output of every
kernel lives inside one arena between two 256 KiB guard zones and, for channel windows, between neighbouring channels
that the kernel must not touch.  The whole arena is filled with a byte pattern first; after the launch every byte outside
the window the op is specified to write (include/yre.h) must still hold it.  Ragged extents, odd maps, images beyond the
batch in the last tile, tile edges clipped by TMA, direct-store tails.  Everything goes through the C ABI.

Out-of-bounds READS cannot be seen this way; the TMA paths read through tensor maps whose extents are the tensor's
(out-of-range boxes are zero-filled by hardware), and the results of the same launches are compared with torch."""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from yolo_b200 import _lib as L

DEV = "cuda"
GUARD = 256 * 1024
PAT = 0xA5


class Arena:
    """Output tensors carved out of one uint8 buffer with guard zones between them."""

    def __init__(self):
        self.items = []          # (offset, nbytes, tensor)
        self.size = GUARD

    def reserve(self, shape, dtype):
        n = 1
        for s in shape:
            n *= s
        nbytes = n * torch.empty((), dtype=dtype).element_size()
        off = (self.size + 1023) // 1024 * 1024
        self.items.append((off, nbytes, shape, dtype))
        self.size = off + nbytes + GUARD
        return len(self.items) - 1

    def build(self):
        self.buf = torch.full((self.size + 1024,), PAT, dtype=torch.uint8, device=DEV)
        base = (-self.buf.data_ptr()) % 1024          # 1024-byte aligned carve (TMA wants 128)
        self.base = base
        self.t = [self.buf[base + off: base + off + nb].view(dt).view(shape) for off, nb, shape, dt in self.items]
        return self.t

    def check_guards(self, what):
        torch.cuda.synchronize()
        mask = torch.ones_like(self.buf, dtype=torch.bool)
        for off, nb, _, _ in self.items:
            mask[self.base + off: self.base + off + nb] = False
        bad = ((self.buf != PAT) & mask).nonzero()
        assert bad.numel() == 0, f"{what}: {bad.numel()} guard bytes overwritten, first at arena offset {int(bad[0]) - self.base}"


def pattern_like(t):
    return torch.full_like(t.view(torch.uint8), PAT).view(t.dtype).view(t.shape)


def view(t, dt, layout, Bn, H, W, ct, coff, c):
    return L.View(t.data_ptr(), dt, layout, Bn, H, W, ct, coff, c)


def null():
    return L.View(None, 0, 0, 0, 0, 0, 0, 0, 0)


def untouched_outside_window(y, coff, c, what):
    """channels outside [coff, coff + c) of the NHWC buffer y still hold the pattern"""
    raw = y.view(torch.uint8).view(*y.shape[:-1], y.shape[-1] * y.element_size())
    es = y.element_size()
    assert bool((raw[..., :coff * es] == PAT).all()) and bool((raw[..., (coff + c) * es:] == PAT).all()), f"{what}: wrote outside its channel window"


# (B, H, W, Cin, Cout, k, res, f32out, engine, y extra channels, y window offset, xu channels)
CONV_CASES = [
    (3, 13, 13, 64, 256, 1, 0, 0, "tc", 64, 32, 0),      # generic, ragged map, TMA-store clipping, window inside a wider buffer
    (5, 9, 11, 64, 128, 1, 0, 0, "tc", 0, 0, 0),         # tiles spanning images, 5 images: boxes beyond the batch
    (2, 37, 29, 64, 64, 3, 1, 0, "tc", 32, 0, 0),        # weight-stationary halo kernel, ragged patches, in-place style residual
    (2, 50, 19, 32, 32, 3, 0, 0, "tc", 0, 0, 0),         # halo kernel, SWIZZLE_64B
    (7, 48, 56, 128, 128, 3, 0, 0, "tc", 0, 0, 0),       # streamed halo, paired patches (147 patches: odd one out)
    (15, 48, 56, 128, 64, 3, 0, 0, "tc", 64, 64, 0),     # paired halo with a 64-wide N tile
    (42, 24, 40, 128, 64, 3, 1, 0, "tc", 64, 32, 0),     # paired halo on 8x8 patches of two images (ybx), odd pair count, residual
    (7, 20, 20, 128, 128, 3, 1, 0, "tc", 0, 0, 0),       # CTA pairs, odd number of M tiles
    (2, 16, 16, 256, 160, 1, 0, 1, "tc", 16, 0, 0),      # fp32 output, direct stores, 16-column tail
    (2, 13, 11, 256, 80, 1, 0, 1, "tc", 0, 0, 0),        # raw class logits: Cout = 80
    (3, 20, 24, 64, 128, 1, 0, 0, "tc", 0, 0, 64),       # upsampled second source (yre_conv_desc.xu)
    (2, 11, 7, 20, 36, 3, 1, 0, "ffma", 12, 4, 0),       # fp32 SIMT engine, odd everything
]


@pytest.mark.parametrize("case", CONV_CASES)
def test_conv_writes_only_its_window(case):
    Bn, H, W, Cin, Cout, k, res, f32out, eng, extra, coff, Cu = case
    lib = L.lib()
    g = torch.Generator().manual_seed(sum(case[:8]))
    tc = eng == "tc"
    xdt, xl = (torch.bfloat16, L.BF16) if tc else (torch.float32, L.F32)
    ydt, yl = (torch.float32, L.F32) if (f32out or not tc) else (torch.bfloat16, L.BF16)
    x = torch.randn((Bn, H, W, Cin), generator=g).to(xdt)
    xu = torch.randn((Bn, H // 2, W // 2, max(Cu, 1)), generator=g).to(xdt)
    w = (torch.randn((Cout, k, k, Cin + Cu), generator=g) / (k * k * (Cin + Cu)) ** 0.5).to(xdt)
    bias = torch.randn((Cout,), generator=g)
    a = Arena()
    iy = a.reserve((Bn, H, W, Cout + extra), ydt)
    (y,) = a.build()
    r = torch.randn((Bn, H, W, Cout), generator=g).to(ydt)
    inp = x.float().permute(0, 3, 1, 2)
    if Cu:
        inp = torch.cat((F.interpolate(xu.float().permute(0, 3, 1, 2), scale_factor=2.0, mode="nearest"), inp), 1)
    ref = F.silu(F.conv2d(inp, w.float().permute(0, 3, 1, 2), bias, padding=k // 2))
    if res:
        ref = ref + r.float().permute(0, 3, 1, 2)
    xd, xud, wd, bd, rd = x.to(DEV), xu.to(DEV), w.to(DEV), bias.to(DEV), r.to(DEV)
    d = L.ConvDesc(view(xd, xl, L.NHWC, Bn, H, W, Cin, 0, Cin), view(y, yl, L.NHWC, Bn, H, W, Cout + extra, coff, Cout),
                   view(rd, yl, L.NHWC, Bn, H, W, Cout, 0, Cout) if res else null(), wd.data_ptr(), bd.data_ptr(), k, 1, L.ACT_SILU,
                   L.ENGINE_TCGEN05 if tc else L.ENGINE_FFMA, view(xud, xl, L.NHWC, Bn, H // 2, W // 2, Cu, 0, Cu) if Cu else null())
    L.check(lib.yre_conv(C.byref(d), torch.cuda.current_stream().cuda_stream), "yre_conv")
    a.check_guards(f"conv {case}")
    untouched_outside_window(y, coff, Cout, f"conv {case}")
    got = y[..., coff:coff + Cout].float().cpu().permute(0, 3, 1, 2)
    tol = 1e-2 if tc else 1e-4
    assert (got - ref).abs().max().item() <= tol * max(1.0, ref.abs().max().item())


@pytest.mark.parametrize("shape", [(2, 3, 45, 37, 2), (3, 3, 64, 64, 2), (1, 3, 33, 50, 1)])
@pytest.mark.parametrize("u8", [False, True])
def test_stem_writes_only_its_output(shape, u8):
    """K2 on odd image sizes, NHWC and parity-plane outputs, fp32 image and uint8 frames."""
    Bn, Cin, H, W, stride = shape
    lib = L.lib()
    g = torch.Generator().manual_seed(H * W)
    Ho, Wo = (H + 2 - 3) // stride + 1, (W + 2 - 3) // stride + 1
    w = torch.randn((64, 3, 3, Cin), generator=g).to(DEV)
    b = torch.randn((64,), generator=g).to(DEV)
    img = torch.rand((Bn, Cin, H, W), generator=g).to(DEV)
    frames = (torch.rand((Bn, H, W, 3), generator=g) * 255).to(torch.uint8).to(DEV)
    for layout in (L.NHWC, L.PHASE4):
        a = Arena()
        shp = (Bn, Ho, Wo, 64) if layout == L.NHWC else (4, Bn, (Ho + 1) // 2, (Wo + 1) // 2, 64)
        a.reserve(shp, torch.bfloat16)
        (y,) = a.build()
        d = L.StemDesc(None if u8 else img.data_ptr(), Bn, Cin, H, W, view(y, L.BF16, layout, Bn, Ho, Wo, 64, 0, 64), w.data_ptr(), b.data_ptr(),
                       stride, L.ACT_SILU, frames.data_ptr() if u8 else None)
        L.check(lib.yre_stem_conv(C.byref(d), torch.cuda.current_stream().cuda_stream), "yre_stem_conv")
        a.check_guards(f"stem {shape} layout {layout} u8={u8}")


@pytest.mark.parametrize("shape", [(2, 128, 37, 41), (3, 64, 40, 40), (1, 256, 21, 20), (2, 80, 20, 20), (1, 32, 48, 48), (1, 32, 64, 64)])
def test_pooling_kernels_write_only_their_outputs(shape):
    """K3 (ADown pre-pool, even and odd maps, parity-plane output), K4 (SPP pyramid), K5 (upsample into a concat slice)."""
    Bn, Cn, H, W = shape
    lib = L.lib()
    s = torch.cuda.current_stream().cuda_stream
    g = torch.Generator().manual_seed(H + W)
    x = torch.randn((Bn, H, W, Cn), generator=g).bfloat16().to(DEV)
    xv = view(x, L.BF16, L.NHWC, Bn, H, W, Cn, 0, Cn)
    # ADown
    half, Ha, Wa = Cn // 2, H - 1, W - 1
    Ho, Wo = (Ha + 2 - 3) // 2 + 1, (Wa + 2 - 3) // 2 + 1
    a = Arena()
    a.reserve((4, Bn, (Ha + 1) // 2, (Wa + 1) // 2, half), torch.bfloat16)
    a.reserve((Bn, Ho, Wo, half + 32), torch.bfloat16)
    lo, hi = a.build()
    L.check(lib.yre_adown_prepool(C.byref(xv), C.byref(view(lo, L.BF16, L.PHASE4, Bn, Ha, Wa, half, 0, half)),
                                  C.byref(view(hi, L.BF16, L.NHWC, Bn, Ho, Wo, half + 32, 32, half)), s), "adown")
    a.check_guards(f"adown {shape}")
    untouched_outside_window(hi, 32, half, f"adown {shape}")
    # SPP
    a = Arena()
    a.reserve((Bn, H, W, 4 * Cn), torch.bfloat16)
    (cat,) = a.build()
    cat[..., :Cn] = x
    vs = [view(cat, L.BF16, L.NHWC, Bn, H, W, 4 * Cn, i * Cn, Cn) for i in range(4)]
    L.check(lib.yre_spp_maxpool(C.byref(vs[0]), C.byref(vs[1]), C.byref(vs[2]), C.byref(vs[3]), s), "spp")
    a.check_guards(f"spp {shape}")
    assert torch.equal(cat[..., :Cn], x)
    for i, win in enumerate((5, 9, 13)):          # bf16 plane kernel (64 / 32 / 16 / 8 channels per CTA) and the direct fallback
        ref = F.max_pool2d(x.float().permute(0, 3, 1, 2), win, 1, win // 2).permute(0, 2, 3, 1)
        assert torch.equal(cat[..., (i + 1) * Cn:(i + 2) * Cn].float(), ref), f"spp window {win} {shape}"
    # upsample into the middle of a wider buffer
    a = Arena()
    a.reserve((Bn, 2 * H, 2 * W, Cn + 64), torch.bfloat16)
    (up,) = a.build()
    L.check(lib.yre_upsample2x(C.byref(xv), C.byref(view(up, L.BF16, L.NHWC, Bn, 2 * H, 2 * W, Cn + 64, 32, Cn)), s), "upsample")
    a.check_guards(f"upsample {shape}")
    untouched_outside_window(up, 32, Cn, f"upsample {shape}")


@pytest.mark.parametrize("nc,levels", [(80, [(20, 20), (10, 10), (5, 5)]), (3, [(13, 9), (7, 5)]), (80, [(160, 160)])])
def test_decode_writes_only_y(nc, levels):
    lib = L.lib()
    Bn = 3
    g = torch.Generator().manual_seed(nc)
    ncp = -(-nc // 16) * 16
    raws = [torch.randn((Bn, h, w, 64 + ncp), generator=g).to(DEV) for h, w in levels]
    A = sum(h * w for h, w in levels)
    a = Arena()
    a.reserve((Bn, A, 4 + nc), torch.float32)
    (y,) = a.build()
    d = L.DecodeDesc()
    for i, (r, (h, w)) in enumerate(zip(raws, levels)):
        d.raw[i] = view(r, L.F32, L.NHWC, Bn, h, w, 64 + ncp, 0, 64 + nc)
        d.stride[i] = float(8 << i)
    d.levels, d.nc = len(levels), nc
    for k in range(16):
        d.dfl_w[k] = float(k)
    d.y = y.data_ptr()
    L.check(lib.yre_dfl_decode_score(C.byref(d), torch.cuda.current_stream().cuda_stream), "decode")
    a.check_guards(f"decode nc={nc} {levels}")
    assert bool(torch.isfinite(y).all())


@pytest.mark.parametrize("Bn,A,nc,conf,max_det,case", [
    pytest.param(*a, None, id="-".join(map(str, a)))
    for a in [(3, 8400, 80, 0.25, 300), (2, 33600, 80, 0.001, 300), (5, 777, 3, 0.05, 7), (1, 20000, 80, 0.0, 300)]] + [
    pytest.param(None, None, None, None, None, name, id=name) for name in ("overflow", "redo_npow2_scale", "mixed4", "mixed3_npow2")])
def test_nms_writes_only_its_outputs(Bn, A, nc, conf, max_det, case):
    """K7: out / counts / keep_anchor / workspace, incl. every anchor a candidate, more candidates than the shared-memory
    sort holds (sampled top-m selection), and the cases of tests/nms_path_cases.py that sort every candidate in global
    memory (sort_global after an overflow of the sampled threshold or after a redo), alone and next to images that take
    the other paths."""
    lib = L.lib()
    if case is None:
        g = torch.Generator().manual_seed(A)
        pred = torch.rand((Bn, A, 4 + nc), generator=g)
        pred[..., :2] *= 640
        pred[..., 2:4] = pred[..., 2:4] * 80 + 4
        pred[..., 4:] = pred[..., 4:] ** 6
        iou = 0.45
    else:
        from tests import nms_path_cases as P
        pred, kw = P.pred_of(case), P.CASES[case].kw
        Bn, A, nc = pred.shape[0], pred.shape[1], pred.shape[2] - 4
        conf, iou, max_det = kw["conf_thres"], kw["iou_thres"], kw.get("max_det", 300)
    pd = pred.to(DEV)
    wsb = lib.yre_nms_workspace_bytes(Bn, A)
    a = Arena()
    a.reserve((Bn, max_det, 6), torch.float32)
    a.reserve((Bn,), torch.int32)
    a.reserve((Bn, max_det), torch.int64)
    a.reserve((wsb,), torch.uint8)
    out, counts, keep, ws = a.build()
    d = L.NmsDesc(pd.data_ptr(), Bn, A, nc, conf, iou, max_det, None, -1, 0, out.data_ptr(), counts.data_ptr(), keep.data_ptr(),
                  ws.data_ptr(), wsb, None)
    L.check(lib.yre_nms_batched(C.byref(d), torch.cuda.current_stream().cuda_stream), "nms")
    a.check_guards(f"nms B{Bn} A{A}")
    n = counts.cpu()
    assert bool(((n >= 0) & (n <= max_det)).all())
    for b in range(Bn):
        k = keep[b, :int(n[b])].cpu()
        assert bool(((k >= 0) & (k < A)).all())
