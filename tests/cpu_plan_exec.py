"""TEST-ONLY CPU interpreter of an engine launch plan (Plan.trace).

It re-states, with torch CPU ops, what each libyre kernel is specified to compute (include/yre.h),
so that the plan compiler's wiring -- BN/RepConv folding, sibling merges, concat-slice windows,
in-place residuals, parity-plane buffers -- can be checked against the oracle without a GPU.
It is not a fallback: nothing in the product imports it."""
import torch
import torch.nn.functional as F

NHWC, PHASE4 = 0, 1


def read(v) -> torch.Tensor:
    """logical [B,H,W,C] fp32 tensor of a view"""
    t = v.t.float()
    if v.layout == NHWC:
        return t[..., v.c_off:v.c_off + v.C].clone()
    out = torch.zeros(v.B, v.H, v.W, v.C, device=t.device)
    for py in range(2):
        for px in range(2):
            plane = t[py * 2 + px][..., v.c_off:v.c_off + v.C]
            sub = out[:, py::2, px::2]
            sub.copy_(plane[:, :sub.shape[1], :sub.shape[2]])
    return out


def write(v, val: torch.Tensor) -> None:
    val = val.to(v.t.dtype)
    if v.layout == NHWC:
        v.t[..., v.c_off:v.c_off + v.C] = val
        return
    for py in range(2):
        for px in range(2):
            sub = val[:, py::2, px::2]
            plane = v.t[py * 2 + px]
            plane[:, :, :, v.c_off:v.c_off + v.C] = 0
            plane[:, :sub.shape[1], :sub.shape[2], v.c_off:v.c_off + v.C] = sub


def nchw(t):
    return t.permute(0, 3, 1, 2)


def nhwc(t):
    return t.permute(0, 2, 3, 1)


def run(plan) -> None:
    for kind, a in plan.trace:
        run_op(kind, a)


def run_op(kind: str, a: dict) -> None:
    """one op of Plan.trace"""
    if kind == "conv":
        x = nchw(read(a["x"]))
        if a.get("xu") is not None:                     # yre_conv_desc.xu: cat([upsample2x(xu), x]) read in place
            x = torch.cat((F.interpolate(nchw(read(a["xu"])), scale_factor=2.0, mode="nearest"), x), 1)
        w = a["w"].float().permute(0, 3, 1, 2)          # [Cout][kh][kw][Cin] -> OIHW
        y = F.conv2d(x, w, a["b"].float(), a["stride"], a["k"] // 2)
        if a["silu"]:
            y = F.silu(y)
        if a["res"] is not None:
            y = y + nchw(read(a["res"]))
        write(a["y"], nhwc(y))
    elif kind == "stem":
        w = a["w"].float().permute(0, 3, 1, 2)
        y = F.conv2d(a["x"].float(), w, a["b"].float(), a["stride"], 1)
        if a["silu"]:
            y = F.silu(y)
        write(a["y"], nhwc(y))
    elif kind == "adown":
        x = nchw(read(a["x"]))
        avg = F.avg_pool2d(x, 2, 1, 0)
        half = x.shape[1] // 2
        write(a["lo"], nhwc(avg[:, :half]))
        write(a["hi"], nhwc(F.max_pool2d(avg[:, half:], 3, 2, 1)))
    elif kind == "spp":
        x = nchw(read(a["x"]))
        for key, k in (("y5", 5), ("y9", 9), ("y13", 13)):
            write(a[key], nhwc(F.max_pool2d(x, k, 1, k // 2)))
    elif kind == "upsample":
        write(a["y"], nhwc(F.interpolate(nchw(read(a["x"])), scale_factor=2.0, mode="nearest")))
    elif kind == "cbfuse":
        tgt = nchw(read(a["target"]))
        acc = torch.zeros_like(tgt)
        for s in a["srcs"]:
            acc = acc + F.interpolate(nchw(read(s)), size=tgt.shape[2:], mode="nearest")
        write(a["y"], nhwc(acc + tgt))
    elif kind == "nchw_to_view":
        write(a["y"], nhwc(a["x"].float()))
    elif kind == "view_to_nchw":
        a["y"].copy_(nchw(read(a["x"])))
    elif kind == "decode":
        outs = []
        for r, st in zip(a["raws"], a["strides"]):
            z = read(r)                                   # [B,H,W,64+nc]
            Bn, H, W, _ = z.shape
            e = (z[..., :64].reshape(Bn, H, W, 4, 16).softmax(-1) * torch.tensor(a["dfl_w"])).sum(-1)
            gy, gx = torch.meshgrid(torch.arange(H) + 0.5, torch.arange(W) + 0.5, indexing="ij")
            x1, y1, x2, y2 = gx - e[..., 0], gy - e[..., 1], gx + e[..., 2], gy + e[..., 3]
            box = torch.stack(((x1 + x2) / 2, (y1 + y2) / 2, x2 - x1, y2 - y1), -1) * st
            outs.append(torch.cat((box, z[..., 64:].sigmoid()), -1).reshape(Bn, H * W, -1))
        a["y"].copy_(torch.cat(outs, 1))
    else:
        raise ValueError(kind)
