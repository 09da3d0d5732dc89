"""The tcgen05 conv cases of the per-element parity suite, importable without a GPU.

Each case is one `yre_conv` call on the tcgen05 engine.  `tests/test_cpu_conv_tc_coverage.py` checks on the CPU that the
list reaches every kernel of `TC_KERNELS` (yolo-re_b200/csrc/k_conv_tc.cu) that the selector can pick, and the edges each
kernel must get right; `tests/test_gpu_conv_tc_exact.py` runs every case on the device against an fp64 reference.  Each
case runs twice there, with a bf16 and with an fp32 output; the two outputs of one shape get the same tiling, so one case
covers its bf16 row and, for the one-CTA generic kernel, the fp32 TMA-store row of the same shape."""
from __future__ import annotations

import ctypes as C
import re
from dataclasses import dataclass

from yolo_b200 import _lib

NUM_SMS = 148          # B200


@dataclass(frozen=True)
class Case:
    name: str
    B: int
    H: int                 # logical input extent (a PHASE4 input is stored as parity planes of this map)
    W: int
    Cin: int               # channels read from x (the upsampled source adds `cu` more, ahead of them)
    Cout: int
    k: int = 3
    stride: int = 1
    silu: bool = True
    bias: bool = True      # False: bias = NULL
    res: str = "none"      # "none" | "bf16" | "f32"; the residual has the output window's geometry
    x_ct: int = 0          # x buffer channels (0: Cin) and window offset
    x_off: int = 0
    y_ct: int = 0          # y (and residual) buffer channels (0: Cout) and window offset
    y_off: int = 0
    cu: int = 0            # channels of the half-resolution upsampled source (1x1 only)

    @property
    def Ho(self) -> int:
        return (self.H + 2 * (self.k // 2) - self.k) // self.stride + 1

    @property
    def Wo(self) -> int:
        return (self.W + 2 * (self.k // 2) - self.k) // self.stride + 1

    @property
    def xct(self) -> int:
        return self.x_ct or self.Cin

    @property
    def yct(self) -> int:
        return self.y_ct or self.Cout

    @property
    def phase4(self) -> bool:
        return self.stride == 2


_NULL = _lib.View(None, 0, 0, 0, 0, 0, 0, 0, 0)
_FAKE = dict(x=0x7f0000000000, y=0x7f0100000000, res=0x7f0200000000, w=0x7f0300000000, bias=0x7f0400000000,
             xu=0x7f0500000000)


def desc(c: Case, ptrs: dict | None = None, y_f32: bool = False) -> _lib.ConvDesc:
    """The ConvDesc of case c; ptrs maps x / y / res / w / bias / xu to device addresses (None: fake aligned ones)."""
    p = dict(_FAKE) if ptrs is None else ptrs
    ydt = _lib.F32 if y_f32 else _lib.BF16
    x = _lib.View(p["x"], _lib.BF16, _lib.PHASE4 if c.phase4 else _lib.NHWC, c.B, c.H, c.W, c.xct, c.x_off, c.Cin)
    y = _lib.View(p["y"], ydt, _lib.NHWC, c.B, c.Ho, c.Wo, c.yct, c.y_off, c.Cout)
    res = _NULL
    if c.res != "none":
        res = _lib.View(p["res"], _lib.F32 if c.res == "f32" else _lib.BF16, _lib.NHWC, c.B, c.Ho, c.Wo, c.yct, c.y_off, c.Cout)
    xu = _lib.View(p["xu"], _lib.BF16, _lib.NHWC, c.B, c.H // 2, c.W // 2, c.cu, 0, c.cu) if c.cu else _NULL
    return _lib.ConvDesc(x, y, res, p["w"], p["bias"] if c.bias else None, c.k, c.stride,
                         _lib.ACT_SILU if c.silu else _lib.ACT_NONE, _lib.ENGINE_TCGEN05, xu)


def describe(d: _lib.ConvDesc, num_sms: int = NUM_SMS) -> str:
    """yre_conv_tc_describe of d; raises with the library's reason when the engine does not take it."""
    buf = C.create_string_buffer(160)
    code = _lib.lib().yre_conv_tc_describe(C.byref(d), num_sms, buf, len(buf))
    if code != 0:
        raise _lib.YreError(f"yre_conv_tc_describe failed ({code}): {_lib.lib().yre_last_error().decode()}")
    return buf.value.decode()


def row_key(s: str) -> tuple:
    """TC_KERNELS key (halo, block_k, cout, cta2, f32_tma, nthreads, stage64) of a describe string."""
    kind = s.split()[0]
    halo = 1 if kind == "halo-ws" else 2 if kind.startswith("halo-stream") else 0
    block_k = int(re.search(r" K=\d+x(\d+)", s).group(1))
    cout = int(re.search(r" N=(\d+)", s).group(1)) if halo == 1 else 0
    return (halo, block_k, cout, int(kind == "generic-cta2"), int(" tma-f32" in s), int(re.search(r" thr=(\d+)", s).group(1)),
            int(" s64" in s))


def tiling(s: str) -> dict:
    """The fields of a describe string the coverage checks need."""
    tb, th, tw = (int(v) for v in re.search(r" M=(\d+)x(\d+)x(\d+)", s).groups())
    return dict(kind=s.split()[0], tb=tb, th=th, tw=tw, N=int(re.search(r" N=(\d+)", s).group(1)),
                grid=int(re.search(r" grid=(\d+)", s).group(1)), pair=" pair" in s)


# ---- the cases ------------------------------------------------------------------------------------------------------
# Rows are the TC_KERNELS entries at 148 SMs with the product defaults (tests/test_cpu_conv_tc_coverage.py prints the map).
CASES = [
    # one edge case per kernel: ragged M tiles, a residual, x and y windows inside wider buffers, a non-zero bias
    Case("generic_k64_tail16", 3, 27, 29, 128, 160, res="bf16", x_ct=192, x_off=32, y_ct=176, y_off=8),      # rows 0 / 10, N=80
    Case("generic_k32_tail16", 3, 23, 21, 96, 80, res="f32", x_ct=128, x_off=24, y_ct=96, y_off=16),         # rows 1 / 11
    Case("generic_k64_s64_1x1", 2, 79, 77, 64, 256, k=1, res="bf16", x_ct=96, x_off=16, y_ct=264, y_off=8),  # rows 2 / 10
    Case("generic_k32_s64_1x1", 2, 79, 77, 32, 256, k=1, res="bf16", x_ct=64, x_off=8, y_ct=272, y_off=8),   # rows 3 / 11, rounds
    Case("generic_k64_512thr", 2, 21, 19, 64, 128, k=1, res="bf16", x_ct=96, x_off=32, y_ct=160, y_off=16),  # rows 4 / 12
    Case("generic_k32_512thr", 3, 11, 13, 32, 48, k=1, res="f32", x_ct=48, x_off=16, y_ct=64, y_off=8),      # rows 5 / 13
    Case("cta2_k64", 2, 79, 77, 128, 256, res="bf16", x_ct=136, x_off=8, y_ct=272, y_off=16),                # row 6, rounds
    Case("cta2_k32_tail16", 2, 13, 13, 96, 144, res="bf16", x_ct=104, x_off=8, y_ct=160, y_off=16),          # row 7
    Case("cta2_k64_s64", 2, 79, 77, 512, 256, k=1, res="bf16", x_ct=576, x_off=64, y_ct=264, y_off=8),       # rows 8 / 6
    Case("cta2_k32_s64_up", 2, 80, 78, 512, 256, k=1, cu=32, res="bf16", x_ct=520, x_off=8, y_ct=264, y_off=8),   # rows 9 / 7
    Case("halo_stream_384", 3, 79, 78, 64, 128, res="bf16", x_ct=72, x_off=8, y_ct=136, y_off=8),            # row 14, rounds
    Case("halo_stream_512", 2, 47, 45, 128, 128, res="bf16", x_ct=136, x_off=8, y_ct=144, y_off=16),         # row 16
    Case("halo_ws_k64_64", 2, 37, 29, 64, 64, res="bf16", x_ct=96, x_off=32, y_ct=80, y_off=8),              # row 17
    Case("halo_ws_k64_32", 2, 37, 29, 64, 32, res="f32", x_ct=72, x_off=8, y_ct=48, y_off=16),               # row 18
    Case("halo_ws_k32_64", 2, 35, 27, 32, 64, res="bf16", x_ct=40, x_off=8, y_ct=72, y_off=8),               # row 19
    Case("halo_ws_k32_32", 3, 35, 27, 32, 32, res="bf16", x_ct=64, x_off=32, y_ct=40, y_off=8),              # row 20
    # no activation, NULL bias
    Case("generic_noact_cout16", 3, 20, 21, 64, 16, k=1, silu=False, y_ct=24, y_off=8),     # Cout 16: the fp32 logits of <= 16 classes
    Case("generic_null_bias", 3, 13, 11, 64, 96, k=1, bias=False, res="f32", y_ct=104, y_off=8),
    Case("generic_tiny_map", 5, 2, 3, 32, 32, k=1, y_ct=40, y_off=8),
    Case("generic_3x3_k32", 2, 33, 35, 32, 128, res="bf16", y_ct=136, y_off=8),
    Case("generic_tail16_208", 2, 40, 39, 256, 208, k=1, silu=False, res="f32", y_ct=216, y_off=8),
    Case("generic_rounds_512", 3, 29, 31, 256, 512, k=1, res="f32", x_ct=264, x_off=8, y_ct=520, y_off=8),
    Case("cta2_noact_null_bias", 2, 79, 77, 128, 256, silu=False, bias=False, y_ct=264, y_off=8),
    Case("cta2_tail16_208", 2, 40, 39, 512, 208, k=1, res="f32", y_ct=216, y_off=8),
    Case("cta2_noact_tail16", 3, 13, 15, 96, 144, silu=False, res="f32", y_ct=152, y_off=8),
    Case("halo_stream_null_bias", 3, 13, 11, 64, 96, bias=False, y_ct=104, y_off=8),
    Case("halo_stream_noact", 2, 45, 47, 128, 128, silu=False, res="bf16", y_ct=136, y_off=8),
    Case("halo_ws_noact", 2, 31, 17, 64, 32, silu=False, y_ct=40, y_off=8),
    Case("halo_ws_noact_null_bias", 2, 21, 19, 32, 32, bias=False, silu=False, res="f32", y_ct=40, y_off=8),
    Case("halo_ws_rounds", 3, 80, 79, 64, 64, res="bf16", x_ct=72, x_off=8, y_ct=72, y_off=8),
    # paired halo-stream schedules with an odd patch out, two-image 8x8 patches (ybx) with an odd patch-pair count
    Case("halo_pair_n64_odd", 15, 48, 56, 128, 64, silu=False, y_ct=72, y_off=8),
    Case("halo_pair_n128_odd", 15, 48, 56, 128, 128, res="f32", y_ct=136, y_off=8),
    Case("halo_ybx_odd", 42, 24, 40, 128, 64, res="bf16", x_ct=136, x_off=8, y_ct=72, y_off=8),
    Case("halo_ybx_noact", 42, 24, 40, 128, 64, silu=False, bias=False, y_ct=72, y_off=8),
    # stride 2 on parity planes of odd maps (plane cells without a source pixel are read at the last row and column)
    Case("s2_generic_xwin", 3, 27, 25, 64, 96, stride=2, res="bf16", x_ct=96, x_off=32, y_ct=104, y_off=8),
    Case("s2_generic_noact", 3, 41, 39, 64, 64, stride=2, silu=False, x_ct=96, x_off=16, y_ct=72, y_off=8),
    Case("s2_generic_k32", 4, 15, 13, 32, 48, stride=2, bias=False, res="bf16", y_ct=56, y_off=8),
    Case("s2_cta2", 8, 79, 77, 128, 256, stride=2, res="f32", y_ct=264, y_off=8),
    # upsampled first source: BLOCK_K 32 and 64
    Case("up_k32", 3, 20, 22, 64, 96, k=1, cu=32, res="bf16", x_ct=96, x_off=32, y_ct=104, y_off=8),
    Case("up_k64", 3, 20, 24, 64, 128, k=1, cu=64, silu=False, y_ct=136, y_off=8),
]
