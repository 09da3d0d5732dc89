"""CPU check that the tcgen05 conv cases (tests/conv_tc_cases.py) reach every kernel the selector can pick, with the edges
each kernel must get right.  The kernel table is parsed from k_conv_tc.cu and the selection is queried through
yre_conv_tc_describe at 148 SMs, so the check needs a build of the library but no GPU.  It fails when the only case of a
row is deleted, or when a kernel that a product build can select is added without a case for it."""
import itertools
import re
from collections import defaultdict

import pytest

from tests.conftest import ROOT
from tests.conv_tc_cases import CASES, NUM_SMS, Case, desc, describe, row_key, tiling

from yolo_b200 import _lib

# rows the selector never picks with the product defaults, and why
TUNING_ONLY = {
    15: "streamed halo with 64-column staging: stage64 defaults to 1x1 convs only (YRE_TC_STAGE64=1 in tuning builds)",
}

_ROW = re.compile(r"^\s*\{(conv\w+)<([^>]*)>,\s*\"[^\"]*\",\s*(\d+),\s*(\d+),\s*(\d+),\s*(\d+),\s*(\d+),\s*(NT_2WG|NT_3WG),\s*(\d+)\},",
                  re.M)


def kernel_table() -> list[tuple[tuple, str]]:
    """(key, instantiation) of every TC_KERNELS row, in table order; key as conv_tc_cases.row_key returns it."""
    src = (ROOT / "yolo-re_b200/csrc/k_conv_tc.cu").read_text()
    body = src[src.index("const TcKernel TC_KERNELS[] = {"):]
    body = body[:body.index("};")]
    rows = []
    for m in _ROW.finditer(body):
        fn, targs, halo, bk, cout, cta2, f32, nt, s64 = m.groups()
        rows.append(((int(halo), int(bk), int(cout), int(cta2), int(f32), 384 if nt == "NT_2WG" else 512, int(s64)), f"{fn}<{targs}>"))
    return rows


TABLE = kernel_table()
KEYS = [k for k, _ in TABLE]


def row_of(s: str) -> int:
    return KEYS.index(row_key(s))


def case_runs() -> list[tuple[Case, bool, str, int]]:
    """(case, fp32 output, describe string, row) of every run of the GPU test"""
    out = []
    for c in CASES:
        for f32 in (False, True):
            s = describe(desc(c, y_f32=f32))
            out.append((c, f32, s, row_of(s)))
    return out


def sweep_rows() -> dict[int, str]:
    """row -> an example shape, over a grid of legal yre_conv shapes"""
    found = {}
    for B, Hm, Cin, Cout, (k, s), f32, cu in itertools.product(
            (1, 2, 3, 16, 64), (8, 13, 20, 27, 40, 41, 80, 160), (32, 64, 96, 128, 256, 512),
            (16, 32, 48, 64, 80, 128, 144, 208, 256, 512), ((1, 1), (3, 1), (3, 2)), (False, True), (0, 32, 64)):
        if cu and (k != 1 or Hm % 2):
            continue
        c = Case("sweep", B, Hm, Hm, Cin, Cout, k=k, stride=s, cu=cu)
        try:
            r = row_of(describe(desc(c, y_f32=f32)))
        except _lib.YreError:          # shapes the engine does not take (e.g. an upsampled source split across a K chunk)
            continue
        found.setdefault(r, f"B{B} {Hm}x{Hm} {Cin}(+{cu} up)->{Cout} {k}x{k} s{s} {'fp32' if f32 else 'bf16'}")
    return found


def mtiles(c: Case, t: dict) -> int:
    cd = lambda a, b: -(-a // b)
    return cd(c.Wo, t["tw"]) * cd(c.Ho, t["th"]) * cd(c.B, t["tb"])


def work_units(c: Case, t: dict) -> tuple[int, int]:
    """(work units, CTAs that take them): tiles for one-CTA kernels, CTA pairs for generic-cta2, patch pairs when paired"""
    tiles_n = c.Cout // t["N"]
    if t["kind"] == "generic-cta2":
        return -(-mtiles(c, t) // 2) * tiles_n, t["grid"] // 2
    if t["kind"].startswith("halo-stream"):
        return -(-mtiles(c, t) // (2 if t["pair"] else 1)) * tiles_n, t["grid"]
    return mtiles(c, t) * tiles_n, t["grid"]


def ragged(c: Case, t: dict) -> bool:
    return bool(c.Wo % t["tw"] or c.Ho % t["th"] or c.B % t["tb"])


def test_kernel_table_parses():
    assert len(TABLE) == 21, f"parsed {len(TABLE)} TC_KERNELS rows: the table's format changed, update the pattern"
    assert len(set(KEYS)) == len(KEYS)


def test_every_case_is_taken_and_writes_a_window():
    for c in CASES:
        assert c.yct > c.Cout, f"{c.name}: the y buffer must be wider than its window (the GPU test checks the channels around it)"
        for f32 in (False, True):
            describe(desc(c, y_f32=f32))
    assert len({c.name for c in CASES}) == len(CASES)


def test_cases_cover_every_selectable_kernel():
    runs = case_runs()
    by_row = defaultdict(list)
    for c, f32, s, r in runs:
        by_row[r].append(f"{c.name}[{'fp32' if f32 else 'bf16'}]")
    print("\nrow  kernel                                         cases")
    for r, (key, fn) in enumerate(TABLE):
        print(f"{r:3d}  {fn:45s}  " + (", ".join(sorted(set(by_row.get(r, [])))) or "TUNING_ONLY: " + TUNING_ONLY.get(r, "-")))
    reached = sweep_rows()
    missing = {r: ex for r, ex in reached.items() if r not in by_row}
    assert not missing, "kernels the selector picks that no case runs: " + "; ".join(
        f"row {r} {TABLE[r][1]} {KEYS[r]} (e.g. {ex})" for r, ex in sorted(missing.items()))
    unreached = set(range(len(TABLE))) - set(reached)
    assert unreached == set(TUNING_ONLY), f"rows the sweep does not reach: {sorted(unreached)}; TUNING_ONLY lists {sorted(TUNING_ONLY)}"
    assert not set(TUNING_ONLY) & set(by_row), "a TUNING_ONLY row is reached by a case"


def test_every_kernel_has_an_edge_case():
    """per row: ragged M tiles, a residual, x and y channel windows inside wider buffers and a non-zero bias in ONE case"""
    edge = defaultdict(bool)
    for c, f32, s, r in case_runs():
        edge[r] |= (ragged(c, tiling(s)) and c.res != "none" and c.xct > c.Cin and c.yct > c.Cout and c.bias)
    bad = [f"row {r} {TABLE[r][1]}" for r in sorted(edge) if not edge[r]]
    assert not bad, "no case combines ragged tiles, a residual, x / y windows and a bias for: " + "; ".join(bad)


def test_case_list_features():
    runs = case_runs()
    missing = []

    def need(what, ok):
        if not ok:
            missing.append(what)

    families = ("generic", "generic-cta2", "halo-ws", "halo-stream", "halo-stream-ybx")
    for fam in families:
        for silu in (True, False):
            need(f"{fam} with {'SiLU' if silu else 'no activation'}",
                 any(tiling(s)["kind"] == fam and c.silu == silu for c, f32, s, r in runs))
    need("NULL bias on a generic kernel", any(tiling(s)["kind"].startswith("generic") and not c.bias for c, f32, s, r in runs))
    need("NULL bias on a halo kernel", any(tiling(s)["kind"].startswith("halo") and not c.bias for c, f32, s, r in runs))
    need("fp32 residual", any(c.res == "f32" for c in CASES))
    s2 = [(c, tiling(s)) for c, f32, s, r in runs if c.phase4 and c.H % 2 and c.W % 2]
    need("stride 2 on a PHASE4 input with odd H and W, one-CTA kernel", any(t["kind"] == "generic" for c, t in s2))
    need("stride 2 on a PHASE4 input with odd H and W, CTA pair", any(t["kind"] == "generic-cta2" for c, t in s2))
    need("stride 2 on a PHASE4 input with odd H and W and an x channel window", any(c.xct > c.Cin for c, t in s2))
    for kind in ("generic", "generic-cta2"):
        need(f"16-column N tail on {kind}", any(tiling(s)["kind"] == kind and tiling(s)["N"] % 32 == 16 for c, f32, s, r in runs))
    need("Cout 16 with an fp32 output", any(c.Cout == 16 and f32 for c, f32, s, r in runs))
    for bk in (32, 64):
        need(f"upsampled source with BLOCK_K {bk}", any(c.cu and row_key(s)[1] == bk for c, f32, s, r in runs))
    for kind in ("halo-stream", "halo-stream-ybx"):
        need(f"paired {kind} with an odd patch count",
             any(tiling(s)["kind"] == kind and tiling(s)["pair"] and mtiles(c, tiling(s)) % 2 for c, f32, s, r in runs))
    for kind in ("generic", "generic-cta2", "halo-ws", "halo-stream"):
        need(f"{kind} with more work units than CTAs",
             any(tiling(s)["kind"] == kind and work_units(c, tiling(s))[0] > work_units(c, tiling(s))[1] for c, f32, s, r in runs))
    assert not missing, "the case list lacks: " + "; ".join(missing)


@pytest.mark.parametrize("s,key", [
    ("generic-cta2 M=1x8x16 N=256 K=16x64 stages=4 s64 tma thr=384 grid=148", (0, 64, 0, 1, 0, 384, 1)),
    ("generic M=1x8x16 N=80 K=1x32 stages=8 tma-f32 thr=384 grid=25", (0, 32, 0, 0, 1, 384, 0)),
    ("halo-ws M=1x16x8 N=32 K=9x32 stages=8 direct thr=512 grid=12", (1, 32, 32, 0, 0, 512, 0)),
    ("halo-stream-ybx M=2x8x8 N=64 K=18x64 stages=2 pair tma thr=384 grid=148", (2, 64, 0, 0, 0, 384, 0)),
])
def test_row_key(s, key):
    assert row_key(s) == key
