"""Square against rectangular letterboxing of 16:9 video frames, gelan-c bf16, batch 64, in one process, on cuda:0.

    python scripts/bench_rect.py [--rounds 3] [--steps 20] [--warmup 5] [--out DIR]

The workload is 64 seeded synthetic 1920 x 1080 uint8 BGR frames held on the device (398 MB, more than the L2).  Each pass
runs the whole detection path through the public API: preprocess(..., dtype=torch.uint8) letterboxes on the device, then
model(x_u8) (static buffers, CUDA graph, BGR->RGB and /255 fused into the stem), then non_max_suppression_async with the
scale_rows of the batch, so the detections come out in original-frame pixels.  The two arms differ only in the letterbox:
square pads every frame to 640 x 640; rect (auto=True, stride 32) pads to the smallest stride-32 rectangle, 640 x 384.

Timing is bench.py's `value`: images x steps over the device-event time of the steps, one batch in flight.  The two arms
alternate round by round (the order flips every round), both warmed up first, and each timed region records the median
SM clock and the active clock-event reasons (bench.py's nvidia-smi sampler).  Also reported: the per-op device times of
both plans (Plan.run_op, CUDA events, the two arms' launches of an op interleaved, best of 3) summed per kernel family,
the conv ops of each plan with the lowest achieved TFLOP/s (with their kernel variants), and the detection agreement between the arms in
original-frame pixels (same class, IoU >= 0.9, bench.py's metric).  The device name and power limit are read in the
same run.  Prints one JSON line and, with --out DIR, also writes it to DIR/bench_rect.json."""
from __future__ import annotations

import argparse
import json
import sys
from collections import defaultdict
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
for p in (ROOT, ROOT / "yolo-re_b200", ROOT / "scripts"):
    if str(p) not in sys.path:
        sys.path.insert(0, str(p))

import numpy as np
import torch
import torch.nn.functional as F

from bench import ClockSampler
from bench_fp16 import match, power_limit

MODEL, IMG, BATCH, FRAME_H, FRAME_W, CONF, IOU, MAX_DET = "gelan-c", 640, 64, 1080, 1920, 0.25, 0.45, 300


def make_frames(n: int, seed: int, dev) -> list[torch.Tensor]:
    """n uint8 HWC BGR frames of FRAME_H x FRAME_W on the device: eight distinct multi-octave noise frames repeated with a
    per-frame brightness ramp, as bench_data.make_inputs builds its images"""
    g = torch.Generator().manual_seed(seed)
    base = []
    for _ in range(min(n, 8)):
        x = torch.zeros(1, 3, FRAME_H, FRAME_W)
        amp, tot, r = 1.0, 0.0, 270
        while r >= 5:
            x += amp * F.interpolate(torch.rand(1, 3, r, r * 16 // 9, generator=g), size=(FRAME_H, FRAME_W), mode="bilinear",
                                     align_corners=False)
            tot += amp
            r //= 2
            amp *= 1.6
        x /= tot
        base.append((x[0] - x.min()) / (x.max() - x.min()))
    ramp = torch.linspace(0.85, 1.0, n)
    return [(base[i % len(base)] * ramp[i] * 255.0).round().to(torch.uint8).permute(1, 2, 0).contiguous().to(dev) for i in range(n)]


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default="", metavar="DIR", help="also write the result to DIR/bench_rect.json")
    args = ap.parse_args()
    if args.rounds < 3 or args.steps < 1:
        ap.error("--rounds must be at least 3 and --steps at least 1")
    if not torch.cuda.is_available():
        raise SystemExit("bench_rect.py needs a CUDA device (B200)")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)

    from oracle import gelan_ref as G
    from yolo_b200 import YOLO, non_max_suppression_async, preprocess, scale_rows

    yaml_path = ROOT / "configs" / "models" / f"{MODEL}.yaml"
    nodes, nc = G.load_graph(yaml_path)
    sd = G.calibrated_state_dict(nodes, nc)
    frames = make_frames(BATCH, seed=7, dev=dev)
    origs = [tuple(f.shape[:2]) for f in frames]
    arms = {"square": False, "rect": True}

    def build():
        m = YOLO.from_yaml(yaml_path)
        m.load_state_dict(sd, strict=True)
        m = m.to(dev).eval().set_precision("bf16")
        m.check_weights, m.fresh_outputs, m.use_cuda_graph = False, False, True
        return m

    models = {a: build() for a in arms}
    bufs = {a: preprocess(frames, IMG, dtype=torch.uint8, auto=auto)[0] for a, auto in arms.items()}   # static input buffers

    def run_public(a, steps):
        pend = None
        for _ in range(steps):
            xu, ratios, pads = preprocess(frames, IMG, out=bufs[a], dtype=torch.uint8, auto=arms[a])
            y, _ = models[a](xu)
            cur = non_max_suppression_async(y.permute(0, 2, 1), CONF, IOU, MAX_DET,
                                            scale=scale_rows(ratios, pads, origs, device=dev))
            if pend is not None:
                pend.result()
            pend = cur
        return pend.result()

    rates, clocks, dets = defaultdict(list), defaultdict(list), {}
    for a in arms:
        run_public(a, args.warmup)
    torch.cuda.synchronize()
    for r in range(args.rounds):
        for a in (("square", "rect") if r % 2 == 0 else ("rect", "square")):
            sampler = ClockSampler(0)
            sampler.start()
            run_public(a, args.warmup)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            sampler.begin()
            e0.record()
            dets[a] = run_public(a, args.steps)
            e1.record()
            torch.cuda.synchronize()
            sampler.end()
            rates[a].append(BATCH * args.steps / (e0.elapsed_time(e1) / 1e3))
            c = sampler.stop()
            clocks[a].append({"sm_mhz": c.get("sm_mhz"), "reasons": c.get("reasons")})

    d = {a: [t.cpu().numpy() for t in dets[a]] for a in arms}
    agree = {"square_detections_matched_by_rect": float(np.mean([match(s, q) for s, q in zip(d["square"], d["rect"])])),
             "rect_detections_matched_by_square": float(np.mean([match(q, s) for s, q in zip(d["square"], d["rect"])])),
             "detections_per_image": {a: round(float(np.mean([len(t) for t in d[a]])), 2) for a in arms}}

    # per-op device times (5 launches each, mean, best of 3 rounds).  The two plans need not have the same op list (the head
    # splits its towers by B*H*W), so each round times all ops of one plan, then all of the other, in alternating order.
    plans = {a: next(iter(m._plans.values())) for a, m in models.items()}
    best = {a: [float("inf")] * len(p.op_table()) for a, p in plans.items()}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for r in range(3):
        for a in (("square", "rect") if r % 2 == 0 else ("rect", "square")):
            for i in range(len(best[a])):
                plans[a].run_op(i)
                e0.record()
                for _ in range(5):
                    plans[a].run_op(i)
                e1.record()
                torch.cuda.synchronize()
                best[a][i] = min(best[a][i], e0.elapsed_time(e1) / 5)
    per_op, conv_ms, slowest = {}, {}, {}
    for a, p in plans.items():
        table, desc, var = p.op_table(), p.op_descriptions(), p.op_variants()
        fam = defaultdict(float)
        for (name, _), t in zip(table, best[a]):
            fam[name] += t
        per_op[a] = {k: round(v, 4) for k, v in sorted(fam.items())}
        conv_ms[a] = round(sum(v for k, v in fam.items() if k.startswith("conv")), 4)
        rate = sorted((f / (t * 1e9), i) for i, ((name, f), t) in enumerate(zip(table, best[a])) if name.startswith("conv") and f > 0)
        slowest[a] = [{"op": i, "desc": desc[i], "variant": var[i], "ms": round(best[a][i], 4), "tflops": round(tf, 1)}
                      for tf, i in rate[:8]]
    flops = {a: sum(f for n, f in p.op_table() if n.startswith("conv")) for a, p in plans.items()}

    med = {a: float(np.median(v)) for a, v in rates.items()}
    out = {"model": MODEL, "precision": "bf16", "batch": BATCH, "frames": f"{FRAME_W}x{FRAME_H} uint8 BGR on the device",
           "input_hw": {a: list(bufs[a].shape[1:3]) for a in arms},
           "device": torch.cuda.get_device_name(dev), "power_limit_and_max_sm_clock": power_limit(),
           "rounds": args.rounds, "steps": args.steps,
           "images_per_s": {a: [round(v, 1) for v in vs] for a, vs in rates.items()},
           "median_images_per_s": {a: round(v, 1) for a, v in med.items()},
           "rect_over_square": round(med["rect"] / med["square"], 4),
           "conv_flops_ratio_rect_over_square": round(flops["rect"] / flops["square"], 4),
           "sm_clock_during_timed_rounds": dict(clocks),
           "detection_agreement_in_frame_pixels": agree,
           "sum_conv_ms": conv_ms,
           "per_op_ms_by_family": per_op,
           "conv_ops_with_the_lowest_tflops": slowest}
    if args.out:
        od = Path(args.out)
        od.mkdir(parents=True, exist_ok=True)
        (od / "bench_rect.json").write_text(json.dumps(out, indent=1))
    print(json.dumps(out))


if __name__ == "__main__":
    main()
