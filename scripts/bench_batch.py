"""One plan with a batch capacity of 64 against one plan per batch size, gelan-c bf16 at 640 x 640, on cuda:0.

    python scripts/bench_batch.py [--rounds 3] [--steps 20] [--warmup 5] [--out DIR]

Arms, for n in 1, 2, 4, 8, 16, 32, 64 images per forward:
  capacity   model.max_batch = 64: one plan, compiled for 64 images, runs every n (yre_plan_run_batch);
  dedicated  model.max_batch = None: a plan compiled for exactly n images, one per batch size.
Both use static output buffers and CUDA graphs (one graph per input buffer and n), on the config-2 shape of bench.py:
64 seeded multi-octave noise images (fp32, 315 MB on the device, more than the 126 MB L2), the n-image input being the
first n of them.  A step is one model(x[:n]); images/s = n x steps over the device-event time of the steps.  The arms
alternate n by n inside every round (the order flips every round), each warmed up before its timed window, which records
the median SM clock and the active clock-event reasons (bench.py's sampler).

Also reported:
  * device memory the plans hold: torch.cuda.memory_allocated / memory_reserved growth over compiling and running the one
    capacity plan for every n, and over compiling and running the seven dedicated plans (eager runs, before any graph);
  * host time of one eager forward of the capacity plan (Plan.run, synchronised before each call, so the enqueue is not
    held up by a full launch queue) when n differs from the previous run's -- every tcgen05 conv re-encodes its output
    tensor map -- against the same n again;
  * whether y of the two arms is bit-identical at every n (the dedicated plans choose tilings and kernel variants for
    their own batch, so below n = 64 it need not be).
The device name, power limit and maximum SM clock are read in the same run.  Prints one JSON line and, with --out DIR,
also writes it to DIR/bench_batch.json."""
from __future__ import annotations

import argparse
import json
import statistics
import sys
import time
from collections import defaultdict
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
for p in (ROOT, ROOT / "yolo-re_b200", ROOT / "scripts"):
    if str(p) not in sys.path:
        sys.path.insert(0, str(p))

import torch

from bench import ClockSampler
from bench_fp16 import power_limit

MODEL, IMG, CAP = "gelan-c", 640, 64
NS = (1, 2, 4, 8, 16, 32, 64)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default="", metavar="DIR", help="also write the result to DIR/bench_batch.json")
    args = ap.parse_args()
    if args.rounds < 1 or args.steps < 1:
        ap.error("--rounds and --steps must be at least 1")
    if not torch.cuda.is_available():
        raise SystemExit("bench_batch.py needs a CUDA device (B200)")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)

    from oracle import gelan_ref as G
    from yolo_b200 import YOLO

    yaml_path = ROOT / "configs" / "models" / f"{MODEL}.yaml"
    nodes, nc = G.load_graph(yaml_path)
    sd = G.calibrated_state_dict(nodes, nc)
    x = G.fractal(CAP, IMG, torch.Generator().manual_seed(3)).to(dev)

    def build(max_batch):
        m = YOLO.from_yaml(yaml_path)
        m.load_state_dict(sd, strict=True)
        m = m.to(dev).eval().set_precision("bf16")
        m.check_weights, m.fresh_outputs, m.use_cuda_graph = False, False, False
        m.max_batch = max_batch
        return m

    # ---- memory: eager runs of every n, before any graph ----
    torch.cuda.synchronize()
    memory, models, y_eager = {}, {}, {}
    for arm, mb in (("capacity", CAP), ("dedicated", None)):
        a0, r0 = torch.cuda.memory_allocated(), torch.cuda.memory_reserved()
        models[arm] = build(mb)
        for n in NS:
            y, _ = models[arm](x[:n])
            y_eager[arm, n] = y.clone()
        torch.cuda.synchronize()
        memory[arm] = {"plans": len(models[arm]._plans),
                       "allocated_gib": round((torch.cuda.memory_allocated() - a0 - sum(y_eager[arm, n].nbytes for n in NS)) / 2**30, 3),
                       "reserved_gib": round((torch.cuda.memory_reserved() - r0) / 2**30, 3)}
    identical = {n: torch.equal(y_eager["capacity", n].view(torch.int32), y_eager["dedicated", n].view(torch.int32)) for n in NS}

    # ---- host time of a run whose n differs from the previous one ----
    p = next(iter(models["capacity"]._plans.values()))
    host = defaultdict(list)
    for i in range(40):
        for label, n in (("same_n", 8), ("same_n", 8), ("changed_n", 9), ("changed_n", 8)):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            p.run(n)
            t1 = time.perf_counter()
            if i >= 5:
                host[label].append((t1 - t0) * 1e6)
    torch.cuda.synchronize()
    host_us = {k: round(statistics.median(v), 1) for k, v in host.items()}

    # ---- throughput, CUDA graphs ----
    for m in models.values():
        m.use_cuda_graph = True

    def run(arm, n, steps):
        for _ in range(steps):
            models[arm](x[:n])

    for arm in models:
        for n in NS:
            run(arm, n, args.warmup)
    torch.cuda.synchronize()
    rates, clocks = defaultdict(list), defaultdict(list)
    for r in range(args.rounds):
        for n in NS:
            for arm in (("capacity", "dedicated") if r % 2 == 0 else ("dedicated", "capacity")):
                sampler = ClockSampler(0)
                sampler.start()
                run(arm, n, args.warmup)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                sampler.begin()
                e0.record()
                run(arm, n, args.steps)
                e1.record()
                torch.cuda.synchronize()
                sampler.end()
                rates[arm, n].append(n * args.steps / (e0.elapsed_time(e1) / 1e3))
                c = sampler.stop()
                clocks[arm].append(c.get("sm_mhz"))
                clocks[arm + "_reasons"] += [s for s in c.get("reasons", []) if s not in clocks[arm + "_reasons"]]

    med = {k: statistics.median(v) for k, v in rates.items()}
    table = [{"n": n, "capacity_images_per_s": round(med["capacity", n], 1), "dedicated_images_per_s": round(med["dedicated", n], 1),
              "capacity_over_dedicated": round(med["capacity", n] / med["dedicated", n], 4), "y_bit_identical_to_dedicated": identical[n],
              "capacity_runs": [round(v, 1) for v in rates["capacity", n]], "dedicated_runs": [round(v, 1) for v in rates["dedicated", n]]}
             for n in NS]
    out = {"model": MODEL, "precision": "bf16", "input": f"{IMG}x{IMG} fp32 images on the device", "capacity": CAP,
           "cuda_graph": True, "device": torch.cuda.get_device_name(dev), "power_limit_and_max_sm_clock": power_limit(),
           "rounds": args.rounds, "steps": args.steps, "warmup": args.warmup,
           "median_sm_mhz_in_timed_windows": {a: statistics.median([c for c in clocks[a] if c is not None] or [0]) for a in models},
           "clock_event_reasons_seen": {a: clocks[a + "_reasons"] for a in models},
           "per_n": table, "memory": memory, "host_us_per_eager_run_n8_n9": host_us,
           "tcgen05_convs_per_run": p.num_tcgen05}
    if args.out:
        od = Path(args.out)
        od.mkdir(parents=True, exist_ok=True)
        (od / "bench_batch.json").write_text(json.dumps(out, indent=1))
    print(json.dumps(out))


if __name__ == "__main__":
    main()
