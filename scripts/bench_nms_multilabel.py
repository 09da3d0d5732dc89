"""Multi-label against single-label NMS (K7) on the engine's own predictions, on cuda:0.

    python scripts/bench_nms_multilabel.py [--iters 20] [--warmup 5] [--out DIR]

Inputs: y of gelan-c (bf16, calibrated weights, bench.py's recipe) on seeded multi-octave noise images:
  config 2   64 x 640²   (8 400 anchors)  at conf 0.25 / IoU 0.45 and conf 0.001 / IoU 0.7 (upstream val.py's setting)
  config 5   16 x 1280²  (33 600 anchors) at conf 0.001 / IoU 0.7
For every setting the two modes alternate (the order flips every iteration) after a warm-up of both.  Per batch, CUDA events
time the candidate pass alone (yre_nms_filter_only / yre_nms_multi_label_filter_only: counter reset + filter, 2 launches)
and the whole call (3 launches); select = whole - candidate pass.  Medians over the iterations are reported.

Also reported per setting and mode: candidates and kept boxes per image (min / median / max), the way the select kernel got
its sorted list per image (smem: n <= 8192; sampled: above that, the workspace keys are still in filter order after the
call; sort_global: they were sorted in place, after an overflow or a redo -- the two are not told apart), and the candidate
pass's bytes (pred read once, the keys written: 8 B per candidate, plus the 4 B class map entry in single-label) over its
time against the measured 6 549.8 GB/s.  The device name, power limit and maximum SM clock are read in the same run.
Prints one JSON line and, with --out DIR, writes it to DIR/bench_nms_multilabel.json."""
from __future__ import annotations

import argparse
import ctypes as C
import json
import statistics
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
for p in (ROOT, ROOT / "yolo-re_b200", ROOT / "scripts"):
    if str(p) not in sys.path:
        sys.path.insert(0, str(p))

import numpy as np
import torch

from bench_fp16 import power_limit

HBM_GBS = 6549.8
SMEM_KEYS = 8192
SETTINGS = [("config2", 64, 640, 0.25, 0.45), ("config2", 64, 640, 0.001, 0.7), ("config5", 16, 1280, 0.001, 0.7)]


class Call:
    """one NMS configuration with its own buffers, so the workspace can be read after the call"""

    def __init__(self, L, pred, conf, iou, ml):
        lib = L.lib()
        B, A, ch = pred.shape
        self.lib, self.ml, self.B, self.A, self.nc = lib, ml, B, A, ch - 4
        nbytes = lib.yre_nms_multi_label_workspace_bytes(B, A, ch - 4) if ml else lib.yre_nms_workspace_bytes(B, A)
        dev = pred.device
        self.ws = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
        self.out = torch.empty((B, 300, 6), dtype=torch.float32, device=dev)
        self.counts = torch.empty((B,), dtype=torch.int32, device=dev)
        self.keep = torch.empty((B, 300), dtype=torch.int64, device=dev)
        self.d = L.NmsDesc(pred.data_ptr(), B, A, ch - 4, conf, iou, 300, None, -1, 0, self.out.data_ptr(),
                           self.counts.data_ptr(), self.keep.data_ptr(), self.ws.data_ptr(), nbytes, None)
        self.stream = torch.cuda.current_stream(dev).cuda_stream
        self.fn = lib.yre_nms_batched_multi_label if ml else lib.yre_nms_batched
        self.filter_fn = lib.yre_nms_multi_label_filter_only if ml else lib.yre_nms_filter_only
        self.check = L.check

    def filter(self):
        self.check(self.filter_fn(C.byref(self.d), self.stream), "nms filter")

    def full(self):
        self.check(self.fn(C.byref(self.d), self.stream), "nms")

    def census(self):
        """(candidates, kept, path) per image, read from the workspace and outputs of the last full call"""
        cap = 1
        while cap < (self.A * self.nc if self.ml else self.A):
            cap <<= 1
        keys = self.ws[: 8 * self.B * cap].view(torch.int64).view(self.B, cap)
        off = 8 * self.B * cap + (0 if self.ml else 4 * self.B * self.A)
        n = self.ws[off: off + 4 * self.B].view(torch.int32).tolist()
        kept = self.counts.tolist()
        paths = []
        for b in range(self.B):
            if n[b] <= SMEM_KEYS:
                paths.append("smem")
                continue
            k = keys[b, : n[b]].cpu().numpy().view(np.uint64)
            paths.append("sort_global" if bool(np.all(k[1:] >= k[:-1])) else "sampled")
        return n, kept, paths


def _stats(v):
    return {"min": min(v), "median": statistics.median(v), "max": max(v)}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default="", metavar="DIR")
    args = ap.parse_args()
    if args.iters < 1:
        ap.error("--iters must be at least 1")
    if not torch.cuda.is_available():
        raise SystemExit("bench_nms_multilabel.py needs a CUDA device (B200)")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)

    from oracle import gelan_ref as G
    from yolo_b200 import YOLO
    from yolo_b200 import _lib as L

    yaml_path = ROOT / "configs" / "models" / "gelan-c.yaml"
    nodes, nc = G.load_graph(yaml_path)
    m = YOLO.from_yaml(yaml_path)
    m.load_state_dict(G.calibrated_state_dict(nodes, nc), strict=True)
    m = m.to(dev).eval().set_precision("bf16")

    preds = {}
    with torch.no_grad():
        for cfg, B, S, _, _ in SETTINGS:
            if cfg not in preds:
                x = G.fractal(B, S, torch.Generator().manual_seed(3)).to(dev)
                y, _ = m(x)
                preds[cfg] = y.permute(0, 2, 1).contiguous().float()
                del x
    del m
    torch.cuda.empty_cache()

    ev = lambda: torch.cuda.Event(enable_timing=True)   # noqa: E731
    results = []
    for cfg, B, S, conf, iou in SETTINGS:
        pred = preds[cfg]
        A = pred.shape[1]
        calls = {"single": Call(L, pred, conf, iou, False), "multi": Call(L, pred, conf, iou, True)}
        for _ in range(args.warmup):
            for c in calls.values():
                c.filter()
                c.full()
        torch.cuda.synchronize()
        times = {k: {"filter": [], "full": []} for k in calls}
        for it in range(args.iters):
            order = list(calls) if it % 2 == 0 else list(calls)[::-1]
            for k in order:
                c = calls[k]
                e0, e1, e2 = ev(), ev(), ev()
                e0.record()
                c.filter()
                e1.record()
                c.full()
                e2.record()
                e2.synchronize()
                times[k]["filter"].append(e0.elapsed_time(e1) * 1e3)
                times[k]["full"].append(e1.elapsed_time(e2) * 1e3)
        row = {"config": cfg, "B": B, "img": S, "anchors": A, "conf": conf, "iou": iou}
        for k, c in calls.items():
            n, kept, paths = c.census()
            t_f = statistics.median(times[k]["filter"])
            t_all = statistics.median(times[k]["full"])
            nbytes = pred.numel() * 4 + sum(n) * (8 if k == "multi" else 12)
            row[k] = {
                "filter_us": round(t_f, 1), "select_us": round(t_all - t_f, 1), "total_us": round(t_all, 1),
                "filter_us_spread": [round(min(times[k]["filter"]), 1), round(max(times[k]["filter"]), 1)],
                "total_us_spread": [round(min(times[k]["full"]), 1), round(max(times[k]["full"]), 1)],
                "candidates_per_image": _stats(n), "kept_per_image": _stats(kept),
                "paths": {p: paths.count(p) for p in sorted(set(paths))},
                "filter_bytes": nbytes, "filter_gbs": round(nbytes / (t_f * 1e-6) / 1e9, 1),
                "filter_frac_hbm": round(nbytes / (t_f * 1e-6) / 1e9 / HBM_GBS, 3),
            }
        results.append(row)
        del calls
        torch.cuda.empty_cache()

    out = {"bench": "nms_multilabel", "device": torch.cuda.get_device_name(dev), "power_limit_max_sm_clock": power_limit(),
           "hbm_gbs_reference": HBM_GBS, "iters": args.iters, "warmup": args.warmup, "model": "gelan-c bf16 calibrated",
           "note": "filter = counter reset + candidate pass (2 launches); select = whole call - filter; medians",
           "results": results}
    line = json.dumps(out)
    print(line)
    if args.out:
        Path(args.out).mkdir(parents=True, exist_ok=True)
        (Path(args.out) / "bench_nms_multilabel.json").write_text(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
