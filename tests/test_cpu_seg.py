"""CPU tests of instance segmentation (gelan-c-seg, K6's mask coefficients, K15), without a GPU:
  * the state_dict schema of gelan-c-seg against the oracle's, and the head widths;
  * the dry launch list of a seg plan is gelan-c's, op for op with the same arguments, plus the prototype branch and
    the mask towers before the decode, which also writes mc;
  * every stride-32 rectangle up to 640² fits the shape arena at capacities 16 and 64;
  * the numpy restatement of K15 (oracle/seg_ref.py) against upstream's torch functions in all three modes: the binary
    masks agree wherever upstream's probability is outside the band derived in seg_ref.k15_band;
  * process_mask_native's slicing on square, rectangular and odd-padding geometries;
  * the ctypes structs against include/yre.h compiled with gcc; the refusals of yre_seg_masks and of the compile."""
import ctypes
import subprocess
import tempfile
import zlib
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import seg_ref as S
from tests.conftest import ROOT
from tests.test_cpu_plan_launch_list import _randomize_bn, canonical_lines

from yolo_b200 import YOLO, _lib as L, engine
from yolo_b200.heads import SegmentDFL

SEG = ROOT / "configs/models/gelan-c-seg.yaml"
DET = ROOT / "configs/models/gelan-c.yaml"


@pytest.fixture()
def dry():
    engine._ALLOW_CPU_DRY_RUN = True
    yield
    engine._ALLOW_CPU_DRY_RUN = False


def _pair(shape, prec="bf16"):
    """dry plans of gelan-c and gelan-c-seg with the same weights on the shared keys"""
    torch.manual_seed(0)
    seg = YOLO.from_yaml(SEG)
    _randomize_bn(seg, 1)
    det = YOLO.from_yaml(DET)
    det.load_state_dict({k: v for k, v in seg.state_dict().items() if k in det.state_dict()})
    x = torch.empty(shape)
    return (engine.compile_model(m.eval().set_precision(prec), x) for m in (det, seg))


def test_state_dict_schema_and_widths():
    m = YOLO.from_yaml(SEG)
    sd = m.state_dict()
    nodes, nc, nm, npr = S.load_graph(SEG)
    schema = S.seg_schema(nodes, nc, nm, npr)
    assert list(sd) == list(schema) and len(sd) == 997
    assert all(tuple(sd[k].shape) == schema[k][0] and sd[k].dtype == schema[k][1] for k in sd)
    det_keys = set(YOLO.from_yaml(DET).state_dict())
    assert det_keys < set(sd) and len(set(sd) - det_keys) == 6 * 3 + 6 * 6 + 3 * 2
    head = m.layers["detect"]
    assert isinstance(head, SegmentDFL) and (head.num_masks, head.num_protos) == (32, 256)
    assert [t[0].conv.out_channels for t in head.mask_convs] == [64, 64, 64]        # c4 = max(256 // 4, 32)
    assert [t[0].conv.in_channels for t in head.mask_convs] == [256, 512, 512]
    assert (head.proto.cv1.conv.out_channels, head.proto.cv2.conv.kernel_size, head.proto.cv3.conv.out_channels) == (256, (3, 3), 32)
    assert m._detect_layer()[1] is head and head.stride.tolist() == [8.0, 16.0, 32.0]


@pytest.mark.parametrize("shape", [(2, 3, 640, 640), (3, 3, 384, 640)])
@pytest.mark.parametrize("prec", ["bf16", "fp32"])
def test_seg_launch_list_is_gelan_c_plus_the_new_ops(dry, shape, prec):
    pd, ps = _pair(shape, prec)
    ld, ls = canonical_lines(pd)[:len(pd.trace)], canonical_lines(ps)[:len(ps.trace)]
    n = len(ld)
    assert ls[:n - 1] == ld[:n - 1], "the detection ops differ"
    # the new ops, in this order: prototype branch, three mask towers, the decode that also writes mc
    new = ps.op_descriptions()[n - 1:]
    B, H, W = shape[0], shape[2], shape[3]
    h, w = H // 8, W // 8
    a = " f32out" if prec == "fp32" else ""          # activations are fp32 in the validation engine
    assert new == [f"conv3x3s1 256->256 @{h}x{w} B{B}{a}", f"upsample C256 @{h}x{w} B{B}",
                   f"conv3x3s1 256->256 @{2 * h}x{2 * w} B{B}{a}", f"conv1x1s1 256->32 @{2 * h}x{2 * w} B{B} f32out"] + \
        [d for i, c in enumerate((256, 512, 512)) for d in
         (f"conv3x3s1 {c}->64 @{h >> i}x{w >> i} B{B}{a}", f"conv3x3s1 64->64 @{h >> i}x{w >> i} B{B}{a}",
          f"conv1x1s1 64->32 @{h >> i}x{w >> i} B{B} f32out")] + ["decode"]
    kd, ad = pd.trace[-1]
    ks, as_ = ps.trace[-1]
    geo = lambda a: [(r.B, r.H, r.W, r.C_total, r.c_off, r.C, r.dtype) for r in a["raws"]]
    assert kd == ks == "decode" and geo(ad) == geo(as_) and ad["strides"] == as_["strides"] and ad["dfl_w"] == as_["dfl_w"]
    assert [v.C for v in as_["masks"]] == [32, 32, 32] and all(v.dtype == L.F32 for v in as_["masks"])
    A = sum((h >> i) * (w >> i) for i in range(3))
    assert tuple(as_["mc"].shape) == (B, A, 32) and tuple(as_["y"].shape) == (B, A, 84)
    assert [n for n, _ in ps.op_table()][-1] == "dfl_decode_masks" and [n for n, _ in pd.op_table()][-1] == "dfl_decode_score"
    kind, y, (raws, mc, proto) = ps.result
    assert kind == "segment" and mc is as_["mc"] and (proto.H, proto.W, proto.C, proto.dtype) == (2 * h, 2 * w, 32, L.F32)


def test_other_mask_counts_are_refused(dry):
    m = YOLO.from_yaml(SEG).eval()
    m.layers["detect"].num_masks = 16
    with pytest.raises(L.YreError, match="32 mask coefficients"):
        engine.compile_model(m, torch.empty(1, 3, 64, 64))


@pytest.mark.parametrize("cap", [64, 16])
def test_every_rectangle_fits_the_arena(cap):
    m = YOLO.from_yaml(SEG).eval()
    fold, memo = engine.Plan.fold, {}
    engine.Plan.fold = lambda self, mod: memo[id(mod)] if id(mod) in memo else memo.setdefault(id(mod), fold(self, mod))
    try:
        need = engine.arena_bytes(m, 3, 640, 640, cap)
        for H in range(32, 641, 32):
            for W in range(32, 641, 32):
                x = torch.empty((), dtype=torch.float32).expand(cap, 3, H, W)
                assert engine.compile_model(m, x, cap, layout_only=True).arena_end <= need, (H, W)
    finally:
        engine.Plan.fold = fold


# ---- K15's restatement against upstream ----------------------------------------------------------------------------------
def _seed(*ids) -> int:
    """a fixed seed per case (Python's hash of a str changes from process to process)"""
    return zlib.crc32(repr(ids).encode())


def _case(g, n, mh, mw, shape, frame=None):
    proto = torch.rand((32, mh, mw), generator=g) * 1.3 - 0.28                  # post-SiLU range
    # coefficients of zero sum: every row's logits are centred on 0 over the i.i.d. prototypes, so about half of the
    # pixels inside a box are on and the masks are live by construction
    mc = torch.randn((n, 32), generator=g) * 0.6
    mc -= mc.mean(1, keepdim=True)
    H, W = frame or shape
    xy = torch.rand((n, 2), generator=g) * torch.tensor([W, H]) * 1.1 - 0.05 * torch.tensor([W, H])
    wh = torch.rand((n, 2), generator=g) * torch.tensor([W, H]) * 0.7
    boxes = torch.cat([xy, xy + wh], 1)
    boxes[0] = torch.tensor([-20.0, -10.0, W + 30.0, H + 5.0])                   # beyond the image
    boxes[1] = torch.tensor([10.0, 12.0, 10.0, 40.0])                             # degenerate: no column
    boxes[2] = torch.tensor([13.25, 7.5, 61.75, 33.0])                            # fractional edges
    return proto, mc, boxes


def _agree(ref_p: torch.Tensor, ours: np.ndarray, band: np.ndarray):
    rp = ref_p.double().numpy()
    outside = np.abs(rp - 0.5) > band
    assert outside.mean() > 0.99, outside.mean()
    ref = rp > 0.5
    bad = outside & (ref != ours)
    assert not bad.any(), f"{bad.sum()} pixels differ outside the band"
    live = rp > 0                                  # the pixels the crop keeps (and, upsampled, their bilinear border)
    assert live.sum() > 100 and 0.2 < ref[live].mean() < 0.8, (live.sum(), ref[live].mean())


@pytest.mark.parametrize("mode", ["proto", "input"])
@pytest.mark.parametrize("shape", [(640, 640), (384, 640), (96, 160)])
def test_k15_restatement_matches_process_mask(mode, shape):
    g = torch.Generator().manual_seed(_seed(mode, shape))
    mh, mw = shape[0] // 4, shape[1] // 4
    proto, mc, boxes = _case(g, 12, mh, mw, shape)
    ref = S.process_mask_probs(proto, mc, boxes, shape, upsample=mode == "input")
    ph = proto.permute(1, 2, 0).numpy()
    ours = S.k15_masks(ph, mc.numpy(), boxes.numpy(), mode, shape)
    _agree(ref, ours, S.k15_band(ph, mc.numpy(), mode, shape))
    assert torch.equal(S.process_mask(proto, mc, boxes, shape, mode == "input"), ref.gt(0.5).float())
    assert not ours[1].any()                                                     # the degenerate box keeps nothing


@pytest.mark.parametrize("frame", [(480, 640), (1080, 1920), (500, 375), (427, 640), (37, 53)])
def test_k15_restatement_matches_process_mask_native(frame):
    g = torch.Generator().manual_seed(_seed("native", frame))
    proto, mc, boxes = _case(g, 10, 160, 160, (640, 640), frame)
    ref = S.process_mask_native_probs(proto, mc, boxes, frame)
    ph = proto.permute(1, 2, 0).numpy()
    ours = S.k15_masks(ph, mc.numpy(), boxes.numpy(), "native", frame)
    _agree(ref, ours, S.k15_band(ph, mc.numpy(), "native", frame))


@pytest.mark.parametrize("mh, mw, frame, want", [
    (160, 160, (640, 640), (0, 160, 0, 160)),
    (160, 160, (480, 640), (20, 140, 0, 160)),                 # pad_h = 20
    (96, 160, (480, 800), (0, 96, 0, 160)),                     # a rect input of the frame's aspect: no padding
    (160, 160, (427, 640), (26, 133, 0, 160)),                  # pad_h = 26.625: int() truncates both ends
    (160, 160, (500, 375), (0, 160, 20, 140)),
    (160, 160, (37, 53), (24, 135, 0, 160)),                    # pad_h = 24.15...
])
def test_native_slicing(mh, mw, frame, want):
    assert S.native_slice(mh, mw, frame) == want
    gain = min(mh / frame[0], mw / frame[1])
    pw, ph = (mw - frame[1] * gain) / 2, (mh - frame[0] * gain) / 2
    assert want == (int(ph), int(mh - ph), int(pw), int(mw - pw))


def test_band_is_derived_not_tuned():
    """the band at a proto pixel is 2 gamma_32 sum|mc proto| / 4 + 8u, and an upsampled pixel takes its taps' largest"""
    ph = np.full((4, 4, 32), 0.5, np.float32)
    mc = np.full((1, 32), 2.0, np.float32)
    gamma = 32 * 2.0 ** -24 / (1 - 32 * 2.0 ** -24)
    e = 2 * gamma * 32.0 / 4 + 8 * 2.0 ** -24
    assert np.allclose(S.k15_band(ph, mc, "proto", (16, 16)), e, rtol=0, atol=0)
    assert np.allclose(S.k15_band(ph, mc, "input", (16, 16)), e + 8 * 2.0 ** -24, rtol=0, atol=0)


# ---- C ABI -------------------------------------------------------------------------------------------------------------
def _c_layout(struct: str, fields: list[str]) -> list[int]:
    src = "#include <stddef.h>\n#include <stdio.h>\n#include \"yre.h\"\nint main(void){printf(\"%zu" + " %zu" * len(fields) + \
          "\\n\", sizeof(" + struct + ")" + "".join(f", offsetof({struct}, {f})" for f in fields) + ");return 0;}\n"
    with tempfile.TemporaryDirectory() as d:
        (d_ := Path(d)).joinpath("t.c").write_text(src)
        subprocess.check_call(["gcc", "-I", str(ROOT / "include"), "-o", str(d_ / "t"), str(d_ / "t.c")])
        return [int(v) for v in subprocess.check_output([str(d_ / "t")]).split()]


@pytest.mark.parametrize("cls, struct", [(L.MaskDesc, "yre_mask_desc"), (L.DecodeMasksDesc, "yre_decode_masks_desc")])
def test_ctypes_structs_match_the_header(cls, struct):
    names = [n for n, _ in cls._fields_]
    got = _c_layout(struct, names)
    assert got == [ctypes.sizeof(cls)] + [getattr(cls, n).offset for n in names]


def test_seg_masks_refusals():
    """bad descriptors fail with YRE_EINVAL before any launch (host checks only: no device is touched)"""
    lib = L.lib()
    buf = (ctypes.c_float * 64)()
    a = ctypes.addressof(buf)
    a16 = (a + 15) // 16 * 16

    def desc(**kw):
        d = dict(proto=a16, B=1, n=1, mh=8, mw=8, nm=32, proto_pitch=32, mc=a16, A=4, det=a16, counts=a16, keep_anchor=a16,
                 max_det=4, mode=L.MASK_INPUT, in_h=32, in_w=32, scale=None, masks=a16, out_h=32, out_w=32)
        d.update(kw)
        return L.MaskDesc(**d)

    bad = [dict(mode=3), dict(nm=16), dict(proto=None), dict(mc=None), dict(counts=None), dict(masks=None),
           dict(proto_pitch=30), dict(proto_pitch=16), dict(proto=a16 + 4), dict(mc=a16 + 8), dict(n=2), dict(n=0),
           dict(B=0), dict(mh=0), dict(A=0), dict(max_det=0), dict(out_h=31), dict(in_w=0, out_w=0),
           dict(mode=L.MASK_PROTO), dict(mode=L.MASK_NATIVE, scale=None)]
    for kw in bad:
        assert lib.yre_seg_masks(ctypes.byref(desc(**kw)), None) == -1, kw
    assert lib.yre_seg_masks(None, None) == -1


def test_decode_masks_refusals():
    """a decode descriptor that is valid in every other field: nm != 32 and bad mask views fail with YRE_EINVAL before
    any launch, through the entry point and the plan"""
    lib = L.lib()
    buf = (ctypes.c_float * 256)()
    a16 = (ctypes.addressof(buf) + 15) // 16 * 16
    nc = 16

    def desc(nm=32, mask_dtype=L.F32, mask_c=32):
        d = L.DecodeMasksDesc()
        d.dec.raw[0] = L.View(a16, L.F32, L.NHWC, 1, 1, 1, 64 + nc, 0, 64 + nc)
        d.dec.stride[0], d.dec.levels, d.dec.nc, d.dec.y = 8.0, 1, nc, a16
        d.mask[0] = L.View(a16, mask_dtype, L.NHWC, 1, 1, 1, mask_c, 0, mask_c)
        d.nm, d.mc = nm, a16
        return d

    for kw, why in ((dict(nm=16), "nm=16"), (dict(mask_dtype=L.BF16), "mask level 0"), (dict(mask_c=16), "mask level 0")):
        assert lib.yre_dfl_decode_score_masks(ctypes.byref(desc(**kw)), None) == -1, kw
        assert why in lib.yre_last_error().decode(), lib.yre_last_error()
    h = ctypes.c_void_p()
    L.check(lib.yre_plan_create(ctypes.byref(h)), "plan_create")
    try:
        assert lib.yre_plan_add_decode_masks(h, ctypes.byref(desc(nm=16))) == -1
        assert "nm=16" in lib.yre_last_error().decode()
        assert lib.yre_plan_num_ops(h) == 0
    finally:
        lib.yre_plan_destroy(h)
