"""CPU checks of the fp16 precision: an fp16 conv gets exactly the tcgen05 tiling of the same bf16 conv, the plans of the
benchmark configs are the same op list in both 16-bit precisions, the two 16-bit types never mix within one conv, the
fp16 range guard names the layer whose folded weights overflow, and the uint8 stem's x (1/255) identity holds in fp16.
Needs a build of the library, no GPU."""
import ctypes as C
import itertools

import numpy as np
import pytest
import torch

from tests.conftest import ROOT
from tests.conv_tc_cases import CASES, Case, desc, describe
from tests.test_cpu_conv_tc_coverage import sweep_rows
from tests.test_cpu_conv_tc_select import CONFIGS, GOLDEN, conv_tc_describe

from yolo_b200 import YOLO, _lib, engine
from yolo_b200 import blocks as B


def as_f16(d: _lib.ConvDesc) -> _lib.ConvDesc:
    """the same descriptor with every 16-bit view made fp16 (fp32 views stay fp32)"""
    for v in (d.x, d.y, d.res, d.xu):
        if v.ptr and v.dtype == _lib.BF16:
            v.dtype = _lib.F16
    return d


@pytest.fixture()
def dry():
    engine._ALLOW_CPU_DRY_RUN = True
    yield
    engine._ALLOW_CPU_DRY_RUN = False


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_fp16_cases_get_the_bf16_tiling(case):
    for f32 in (False, True):
        assert describe(as_f16(desc(case, y_f32=f32))) == describe(desc(case, y_f32=f32))


def test_fp16_shape_grid_gets_the_bf16_tiling():
    """the shape grid of the coverage sweep: same answer, or the same rejection"""
    n = 0
    for Bn, Hm, Cin, Cout, (k, s), f32, cu in itertools.product(
            (1, 2, 3, 16, 64), (8, 13, 20, 27, 40, 41, 80, 160), (32, 64, 96, 128, 256, 512),
            (16, 32, 48, 64, 80, 128, 144, 208, 256, 512), ((1, 1), (3, 1), (3, 2)), (False, True), (0, 32, 64)):
        if cu and (k != 1 or Hm % 2):
            continue
        c = Case("sweep", Bn, Hm, Hm, Cin, Cout, k=k, stride=s, cu=cu)
        code16, s16 = conv_tc_describe(desc(c, y_f32=f32), 148)
        codeh, sh = conv_tc_describe(as_f16(desc(c, y_f32=f32)), 148)
        assert (codeh, sh if codeh == 0 else None) == (code16, s16 if code16 == 0 else None), (c, f32, s16, sh)
        n += code16 == 0
    assert n > 1000 and len(sweep_rows()) == 20


@pytest.mark.parametrize("config", sorted(CONFIGS))
def test_fp16_plans_match_bf16_plans(config, dry):
    """a dry fp16 plan of configs 2, 4 and 5 records the bf16 plan's ops, and every conv, described on its fp16 operands,
    gets the variant recorded for the bf16 plan on a B200"""
    name, img, batch = CONFIGS[config]
    m = YOLO.from_yaml(ROOT / "configs/models" / f"{name}.yaml").eval()
    plans = {}
    for prec in ("bf16", "fp16"):
        m.set_precision(prec)
        plans[prec] = engine.compile_model(m, torch.empty(batch, 3, img, img))
    p16, ph = plans["bf16"], plans["fp16"]
    assert ph.op_descriptions() == p16.op_descriptions()
    assert [n for n, _ in ph.op_table()] == [n for n, _ in p16.op_table()]
    assert {v.dtype for k, a in ph.trace if k == "conv" for v in (a["x"], a["y"]) if v.dtype != _lib.F32} == {_lib.F16}
    for op, shape, variant in GOLDEN["configs"][config]:
        a = ph.trace[op][1]
        null = engine._null_view()
        d = _lib.ConvDesc(a["x"].c(), a["y"].c(), a["res"].c() if a["res"] is not None else null, a["w"].data_ptr(),
                          a["b"].data_ptr(), a["k"], a["stride"], _lib.ACT_SILU if a["silu"] else _lib.ACT_NONE,
                          _lib.ENGINE_TCGEN05, a["xu"].c() if a["xu"] is not None else null)
        assert a["w"].dtype == torch.float16 and a["b"].dtype == torch.float32
        code, s = conv_tc_describe(d, GOLDEN["num_sms"])
        assert code == 0 and s == variant, (op, shape, s)


def _mixed(which: str) -> _lib.ConvDesc:
    c = next(c for c in CASES if c.cu and c.res == "bf16")
    d = as_f16(desc(c))
    if which == "xu":
        d.xu.dtype = _lib.BF16
    elif which == "res":
        d.res.dtype = _lib.BF16
    else:
        d.y.dtype = _lib.BF16
    return d


@pytest.mark.parametrize("which", ["xu", "res", "y"])
def test_mixed_16bit_types_are_rejected(which):
    """fp16 x with a bf16 upsampled source, a bf16 residual on an fp16 output, fp16 x with a bf16 y"""
    d = _mixed(which)
    code, msg = conv_tc_describe(d, 148)
    assert code == -3, (code, msg)                        # YRE_EUNSUPPORTED
    for engine_ in (_lib.ENGINE_FFMA, _lib.ENGINE_AUTO):
        d.engine = engine_
        h = C.c_void_p()
        _lib.check(_lib.lib().yre_plan_create(C.byref(h)))
        try:
            assert _lib.lib().yre_plan_add_conv(h, C.byref(d)) == -3
        finally:
            _lib.lib().yre_plan_destroy(h)


def test_fp32_input_is_still_rejected_by_tcgen05():
    c = CASES[0]
    d = desc(c)
    d.x.dtype = _lib.F32
    code, msg = conv_tc_describe(d, 148)
    assert code == -3 and "input must be bf16 or fp16" in msg


def test_range_guard_names_the_layer(dry):
    """one BatchNorm weight scaled so that a folded weight of the second Conv layer is 2 x 65504"""
    m = YOLO.from_yaml(ROOT / "configs/models/gelan-c.yaml").eval()
    name = [n for n, l in m.layers.items() if type(l) is B.Conv][1]
    bn, w = m.layers[name].bn, m.layers[name].conv.weight
    with torch.no_grad():
        bn.weight[0] = 2 * 65504.0 / float(w[0].abs().max()) * float(torch.sqrt(bn.running_var[0] + bn.eps))
    x = torch.empty(2, 3, 64, 64)
    m.set_precision("bf16")
    engine.compile_model(m, x)                          # bf16's range takes it
    m.set_precision("fp16")
    with pytest.raises(_lib.YreError, match=rf"fp16 precision: layer 'layers\.{name}'") as e:
        engine.compile_model(m, x)
    assert "65504" in str(e.value)


def test_range_guard_covers_the_stem(dry):
    m = YOLO.from_yaml(ROOT / "configs/models/gelan-c.yaml").eval().set_precision("fp16")
    stem = next(iter(m.layers))
    with torch.no_grad():
        m.layers[stem].conv.weight[0, 0, 0, 0] = 1e6
    with pytest.raises(_lib.YreError, match=rf"layer 'layers\.{stem}'"):
        engine.compile_model(m, torch.empty(1, 3, 64, 64))


def test_u8_scale_identity_holds_in_fp16():
    """the uint8 stem builds x / 255 as float(v) * (1/255) in fp32 and rounds it to the 16-bit type: for every byte this
    rounds to the same fp16 as the fp32 division, so the uint8 path equals the fp32-tensor path"""
    v = np.arange(256, dtype=np.float32)
    mul = (v * np.float32(1.0 / 255.0)).astype(np.float32)
    div = (v / np.float32(255.0)).astype(np.float32)
    assert (mul != div).any()                             # not an identity in fp32 ...
    assert (mul.astype(np.float16).view(np.uint16) == div.astype(np.float16).view(np.uint16)).all()   # ... but in fp16


def test_precision_strings():
    m = YOLO.from_yaml(ROOT / "configs/models/gelan-c.yaml")
    assert m.set_precision("fp16").precision == "fp16"
    with pytest.raises(ValueError):
        m.set_precision("half")
    with engine.precision("fp16"):
        assert engine._DEFAULT_PRECISION == "fp16"
    assert engine._DEFAULT_PRECISION == "bf16"
