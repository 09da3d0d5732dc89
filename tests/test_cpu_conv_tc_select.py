"""CPU tests of the tcgen05 kernel selection (conv_tc_select, queried through yre_conv_tc_describe): every conv of the
full-size plans of configs 2, 4 and 5 must get the kernel variant a B200 with 148 SMs reported for it
(tests/golden/conv_tc_variants.json, from profiles/r02_per_op*.csv), and the shape rules reject what the kernels cannot
take."""
import ctypes as C
import json

import pytest
import torch

from tests.conftest import ROOT

from yolo_b200 import YOLO, _lib, engine

GOLDEN = json.loads((ROOT / "tests/golden/conv_tc_variants.json").read_text())
CONFIGS = {"2": ("gelan-c", 640, 64), "4": ("yolov9-c", 640, 16), "5": ("gelan-c", 1280, 16)}


def conv_tc_describe(d: _lib.ConvDesc, num_sms: int) -> tuple[int, str]:
    buf = C.create_string_buffer(160)
    code = _lib.lib().yre_conv_tc_describe(C.byref(d), num_sms, buf, len(buf))
    return code, (buf.value if code == 0 else _lib.lib().yre_last_error()).decode()


def tc_variant(a: dict, num_sms: int) -> str:
    """The tcgen05 variant of a conv recorded in Plan.trace, with its descriptor built the way Plan.conv builds it."""
    null = engine._null_view()
    d = _lib.ConvDesc(a["x"].c(), a["y"].c(), a["res"].c() if a["res"] is not None else null, a["w"].data_ptr(),
                      a["b"].data_ptr(), a["k"], a["stride"], _lib.ACT_SILU if a["silu"] else _lib.ACT_NONE,
                      _lib.ENGINE_TCGEN05, a["xu"].c() if a["xu"] is not None else null)
    code, s = conv_tc_describe(d, num_sms)
    assert code == 0, s
    return s


@pytest.fixture()
def dry():
    engine._ALLOW_CPU_DRY_RUN = True
    yield
    engine._ALLOW_CPU_DRY_RUN = False


@pytest.mark.parametrize("config", sorted(CONFIGS))
def test_full_size_plans_get_the_recorded_variants(config, dry):
    # the real batch: the head's split rule, and with it the conv list, depends on it
    name, img, batch = CONFIGS[config]
    m = YOLO.from_yaml(ROOT / "configs/models" / f"{name}.yaml").eval().set_precision("bf16")
    p = engine.compile_model(m, torch.empty(batch, 3, img, img))
    desc = p.op_descriptions()
    golden = GOLDEN["configs"][config]
    assert [i for i, (k, _) in enumerate(p.trace) if k == "conv"] == [op for op, _, _ in golden]
    for op, shape, variant in golden:
        assert desc[op] == shape, (op, desc[op], shape)
        assert tc_variant(p.trace[op][1], GOLDEN["num_sms"]) == variant, (op, shape)


def _view(C_, H, W, dtype=_lib.BF16, layout=_lib.NHWC, ptr=0x7f0000000000):
    return _lib.View(ptr, dtype, layout, 2, H, W, C_, 0, C_)


def _desc(cin=64, k=3, stride=1, x_dtype=_lib.BF16, x_ptr=0x7f0000000000):
    Ho = (80 + 2 * (k // 2) - k) // stride + 1
    return _lib.ConvDesc(_view(cin, 80, 80, x_dtype, ptr=x_ptr), _view(64, Ho, Ho, ptr=0x7f0000100000), engine._null_view(),
                         0x7f0000200000, 0x7f0000300000, k, stride, _lib.ACT_SILU, _lib.ENGINE_TCGEN05, engine._null_view())


@pytest.mark.parametrize("kw,why", [(dict(cin=16), "Cin must be a multiple of 32"),
                                    (dict(x_dtype=_lib.F32), "input must be bf16"),
                                    (dict(stride=2), "stride-2 needs a 3x3 kernel on a PHASE4 input")])
def test_query_rejects_shapes_the_kernels_do_not_take(kw, why):
    code, msg = conv_tc_describe(_desc(**kw), 148)
    assert code == -3, (code, msg)                       # YRE_EUNSUPPORTED
    assert why in msg, msg


def test_query_ignores_address_alignment():
    """Pointers are never dereferenced, and alignment is checked when a plan encodes its tensor maps, not by the query."""
    code, aligned = conv_tc_describe(_desc(), 148)
    assert code == 0, aligned
    code, misaligned = conv_tc_describe(_desc(x_ptr=0x7f0000000040), 148)
    assert code == 0, misaligned
    assert misaligned == aligned and aligned.startswith("halo-ws ")
