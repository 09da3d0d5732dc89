"""bf16 against fp16 on config 2 (gelan-c, 64 x 640 x 640, conf 0.25, iou 0.45), in one process, on cuda:0.

    python scripts/bench_fp16.py [--rounds 3] [--steps 20] [--warmup 5] [--out DIR]

Timing is bench.py's `value`: YOLO.forward (static buffers, CUDA graph) + non_max_suppression_async().result() through the
public API, one batch in flight, device-timed with CUDA events.  The two precisions run as two models with the same
calibrated weights, alternating round by round (the order flips every round) so that clock and neighbour drift hit both.
Each timed region also records the median SM clock and the active clock-event reasons (bench.py's nvidia-smi sampler).
For each precision it also reports the detection agreement with the fp32 engine on the first 8 images (same class,
IoU >= 0.9, bench.py's metric), and the per-op device times of both plans (Plan.run_op, CUDA events, the two precisions'
launches of an op interleaved, best of 3), summed per kernel family.  The device name and power limit are read in the
same run.  Prints the result as one JSON line and, with --out DIR, also writes it to DIR/bench_fp16.json."""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from collections import defaultdict
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
for p in (ROOT, ROOT / "yolo-re_b200"):
    if str(p) not in sys.path:
        sys.path.insert(0, str(p))

import numpy as np
import torch

from bench import ClockSampler
from bench_data import make_inputs

MODEL, IMG, BATCH, CONF, IOU, MAX_DET = "gelan-c", 640, 64, 0.25, 0.45, 300


def power_limit() -> str | None:
    try:
        r = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip() or None
    except (OSError, subprocess.TimeoutExpired):
        return None


def match(ref: np.ndarray, got: np.ndarray) -> float:
    """fraction of `ref` detections with a `got` detection of the same class at IoU >= 0.9 (bench.py's metric)"""
    if len(ref) == 0:
        return 1.0
    if len(got) == 0:
        return 0.0
    x1 = np.maximum(ref[:, None, 0], got[None, :, 0]); y1 = np.maximum(ref[:, None, 1], got[None, :, 1])
    x2 = np.minimum(ref[:, None, 2], got[None, :, 2]); y2 = np.minimum(ref[:, None, 3], got[None, :, 3])
    inter = np.clip(x2 - x1, 0, None) * np.clip(y2 - y1, 0, None)
    ar = (ref[:, 2] - ref[:, 0]) * (ref[:, 3] - ref[:, 1]); ag = (got[:, 2] - got[:, 0]) * (got[:, 3] - got[:, 1])
    iou = inter / (ar[:, None] + ag[None, :] - inter + 1e-12)
    return float(((iou >= 0.9) & (ref[:, None, 5] == got[None, :, 5])).any(1).mean())


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default="", metavar="DIR", help="also write the result to DIR/bench_fp16.json")
    args = ap.parse_args()
    if args.rounds < 3 or args.steps < 1:
        ap.error("--rounds must be at least 3 and --steps at least 1")
    if not torch.cuda.is_available():
        raise SystemExit("bench_fp16.py needs a CUDA device (B200)")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)

    from oracle import gelan_ref as G
    from yolo_b200 import YOLO, non_max_suppression, non_max_suppression_async

    yaml_path = ROOT / "configs" / "models" / f"{MODEL}.yaml"
    nodes, nc = G.load_graph(yaml_path)
    sd = G.calibrated_state_dict(nodes, nc)
    x = make_inputs(BATCH, IMG, seed=7).to(dev)

    def build(prec):
        m = YOLO.from_yaml(yaml_path)
        m.load_state_dict(sd, strict=True)
        m = m.to(dev).eval().set_precision(prec)
        m.check_weights, m.fresh_outputs, m.use_cuda_graph = False, False, True
        return m

    models = {p: build(p) for p in ("bf16", "fp16")}

    def run_public(m, steps):
        pend, dets = None, None
        for _ in range(steps):
            y, _ = m(x)
            cur = non_max_suppression_async(y.permute(0, 2, 1), CONF, IOU, MAX_DET)
            if pend is not None:
                dets = pend.result()
            pend = cur
        return pend.result()

    rates, clocks, dets = defaultdict(list), defaultdict(list), {}
    for p, m in models.items():
        run_public(m, args.warmup)
    torch.cuda.synchronize()
    for r in range(args.rounds):
        for p in (("bf16", "fp16") if r % 2 == 0 else ("fp16", "bf16")):
            m = models[p]
            sampler = ClockSampler(0)
            sampler.start()
            run_public(m, args.warmup)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            sampler.begin()
            e0.record()
            dets[p] = run_public(m, args.steps)
            e1.record()
            torch.cuda.synchronize()
            sampler.end()
            rates[p].append(BATCH * args.steps / (e0.elapsed_time(e1) / 1e3))
            c = sampler.stop()
            clocks[p].append({"sm_mhz": c.get("sm_mhz"), "reasons": c.get("reasons")})

    # detection agreement with the fp32 engine on the first 8 images
    nb = 8
    m32 = YOLO.from_yaml(yaml_path)
    m32.load_state_dict(sd, strict=True)
    m32 = m32.to(dev).eval().set_precision("fp32")
    y32, _ = m32(x[:nb].contiguous())
    d32 = [d.cpu().numpy() for d in non_max_suppression(y32.permute(0, 2, 1), CONF, IOU, MAX_DET)]
    del m32
    agree = {}
    for p in models:
        dp = [d.cpu().numpy() for d in dets[p][:nb]]
        agree[p] = {f"fp32_detections_matched_by_{p}": float(np.mean([match(a, b) for a, b in zip(d32, dp)])),
                    f"{p}_detections_matched_by_fp32": float(np.mean([match(b, a) for a, b in zip(d32, dp)]))}

    # per-op device times, summed per kernel family: op i of the bf16 plan and op i of the fp16 plan are timed back to back
    # (5 launches each, mean), three times in alternating order, best of the three -- so drifting clocks hit both alike
    plans = {p: next(iter(m._plans.values())) for p, m in models.items()}
    names = [n for n, _ in plans["bf16"].op_table()]
    assert names == [n for n, _ in plans["fp16"].op_table()]
    fam = {p: defaultdict(float) for p in plans}
    ops = []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for i, name in enumerate(names):
        best = {p: float("inf") for p in plans}
        for r in range(3):
            for p in (("bf16", "fp16") if r % 2 == 0 else ("fp16", "bf16")):
                plans[p].run_op(i)
                e0.record()
                for _ in range(5):
                    plans[p].run_op(i)
                e1.record()
                torch.cuda.synchronize()
                best[p] = min(best[p], e0.elapsed_time(e1) / 5)
        for p in plans:
            fam[p][name] += best[p]
        ops.append((best["fp16"] - best["bf16"], i, best["bf16"], best["fp16"]))
    per_op = {p: {k: round(v, 4) for k, v in sorted(f.items())} for p, f in fam.items()}

    med = {p: float(np.median(v)) for p, v in rates.items()}
    out = {"config": 2, "model": MODEL, "batch": BATCH, "img": IMG, "device": torch.cuda.get_device_name(dev),
           "power_limit_and_max_sm_clock": power_limit(), "rounds": args.rounds, "steps": args.steps,
           "images_per_s": {p: [round(v, 1) for v in vs] for p, vs in rates.items()},
           "median_images_per_s": {p: round(v, 1) for p, v in med.items()},
           "sm_clock_during_timed_rounds": dict(clocks),
           "fp16_over_bf16": round(med["fp16"] / med["bf16"], 4),
           "detection_agreement_with_fp32_first_8_images": agree,
           "per_op_ms_by_family": per_op,
           "largest_per_op_differences": [{"op": i, "desc": plans["bf16"].op_descriptions()[i], "variant": plans["bf16"].op_variants()[i],
                                           "bf16_ms": round(b, 4), "fp16_ms": round(h, 4)}
                                          for _, i, b, h in sorted(ops, reverse=True)[:10]]}
    if args.out:
        od = Path(args.out)
        od.mkdir(parents=True, exist_ok=True)
        (od / "bench_fp16.json").write_text(json.dumps(out, indent=1))
    print(json.dumps(out))


if __name__ == "__main__":
    main()
