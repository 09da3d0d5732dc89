"""Test-time augmentation against the plain forward: gelan-c bf16 at 640 x 640, batch 64, CUDA graphs, with NMS, on cuda:0.

    python scripts/bench_tta.py [--rounds 3] [--steps 20] [--warmup 5] [--out DIR]

A step is one forward of the 64 images followed by NMS (conf 0.25, IoU 0.45) on its y:
  plain  y = model(x)                  8400 anchors
  tta    y = model(x, augment=True)    15 049 anchors (branches 640², 544² mirrored, 448²; K12 + 3 plan replays + K13)
Both arms use static output buffers and CUDA graphs (one per plan and input buffer); K12 and K13 are launched eagerly
around the graph replays.  The input is 64 seeded multi-octave noise images (fp32, 315 MB on the device, more than the
126 MB L2).  The arms alternate inside every round (the order flips every round), each warmed up before its timed window;
images/s = 64 x steps over the device-event time of the window, whose median SM clock and clock-event reasons are recorded
(bench.py's sampler).

Also reported:
  * K12 and K13 on their own: CUDA events around 50 back-to-back launches at the workload's shapes, with the bytes each
    must move (K12: the fp32 source read once, its branch image written; K13: the kept rows read and written) over that
    time;
  * agreement of the bf16 TTA detections with the fp32 engine's TTA detections on the first 8 images: the fraction of the
    fp32 detections matched by a bf16 detection of the same class at IoU >= 0.9 (bench.py's metric), and the counts; the
    same for the plain forward beside it, as the scale of what bf16 rounding alone does to the detections.
The device name, power limit and maximum SM clock are read in the same run.  Prints one JSON line and, with --out DIR,
also writes it to DIR/bench_tta.json."""
from __future__ import annotations

import argparse
import json
import statistics
import sys
from collections import defaultdict
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
for p in (ROOT, ROOT / "yolo-re_b200", ROOT / "scripts"):
    if str(p) not in sys.path:
        sys.path.insert(0, str(p))

import torch

from bench import ClockSampler
from bench_fp16 import match, power_limit

MODEL, IMG, BATCH, N_AGREE = "gelan-c", 640, 64, 8


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default="", metavar="DIR", help="also write the result to DIR/bench_tta.json")
    args = ap.parse_args()
    if args.rounds < 1 or args.steps < 1:
        ap.error("--rounds and --steps must be at least 1")
    if not torch.cuda.is_available():
        raise SystemExit("bench_tta.py needs a CUDA device (B200)")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)

    from oracle import gelan_ref as G
    from yolo_b200 import YOLO, nms_raw, non_max_suppression, tta

    yaml_path = ROOT / "configs" / "models" / f"{MODEL}.yaml"
    nodes, nc = G.load_graph(yaml_path)
    sd = G.calibrated_state_dict(nodes, nc)
    x = G.fractal(BATCH, IMG, torch.Generator().manual_seed(3)).to(dev)
    g = tta.geometry(IMG, IMG)

    def build(prec):
        m = YOLO.from_yaml(yaml_path)
        m.load_state_dict(sd, strict=True)
        return m.to(dev).eval().set_precision(prec)

    m = build("bf16")
    m.check_weights, m.fresh_outputs, m.use_cuda_graph = False, False, True

    def step(augment: bool):
        y, _ = m(x, augment=True) if augment else m(x)
        nms_raw(y.permute(0, 2, 1), 0.25, 0.45)

    # ---- throughput ----
    arms = {"plain": False, "tta": True}
    for a in arms.values():
        for _ in range(args.warmup):
            step(a)
    torch.cuda.synchronize()
    rates, clocks = defaultdict(list), defaultdict(list)
    for r in range(args.rounds):
        for arm in (("plain", "tta") if r % 2 == 0 else ("tta", "plain")):
            sampler = ClockSampler(0)
            sampler.start()
            for _ in range(args.warmup):
                step(arms[arm])
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            sampler.begin()
            e0.record()
            for _ in range(args.steps):
                step(arms[arm])
            e1.record()
            torch.cuda.synchronize()
            sampler.end()
            rates[arm].append(BATCH * args.steps / (e0.elapsed_time(e1) / 1e3))
            c = sampler.stop()
            clocks[arm].append(c.get("sm_mhz"))
            clocks[arm + "_reasons"] += [s for s in c.get("reasons", []) if s not in clocks[arm + "_reasons"]]
    med = {a: statistics.median(v) for a, v in rates.items()}

    # ---- K12 / K13 on their own ----
    def timed(fn, reps=50):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e3 / reps

    kernels = {}
    for i in (1, 2):
        buf = torch.empty((BATCH, 3, g.out_h[i], g.out_w[i]), device=dev)
        us = timed(lambda: tta.scale_img(x, g, i, out=buf))
        nbytes = x.nbytes + buf.nbytes
        kernels[f"k12_branch{i}_{g.out_h[i]}x{g.out_w[i]}"] = {"us": round(us, 1), "bytes": nbytes,
                                                               "gb_per_s": round(nbytes / us / 1e3, 1)}
    ys = [torch.rand((BATCH, g.A[i], 4 + nc), device=dev) for i in range(3)]
    out = torch.empty((BATCH, g.A_tot, 4 + nc), device=dev)
    us = timed(lambda: tta.merge(ys, g, out=out))
    nbytes = 2 * out.nbytes
    kernels["k13_merge"] = {"us": round(us, 1), "bytes": nbytes, "gb_per_s": round(nbytes / us / 1e3, 1)}
    del ys, out

    # ---- agreement with the fp32 engine, TTA and plain ----
    m32 = build("fp32")
    xa = x[:N_AGREE].contiguous()
    agreement = {}
    for arm, augment in arms.items():
        dets = {}
        for prec, mm in (("bf16", m), ("fp32", m32)):
            y, _ = mm(xa, augment=True) if augment else mm(xa)
            dets[prec] = non_max_suppression(y.permute(0, 2, 1).contiguous(), 0.25, 0.45)
        agreement[arm] = {"matched_fraction_per_image": [round(match(a.cpu().numpy(), b.cpu().numpy()), 4)
                                                         for a, b in zip(dets["fp32"], dets["bf16"])],
                          "fp32_detections": [len(d) for d in dets["fp32"]], "bf16_detections": [len(d) for d in dets["bf16"]]}

    res = {"model": MODEL, "precision": "bf16", "input": f"{BATCH} x {IMG}x{IMG} fp32 images on the device", "batch": BATCH,
           "cuda_graph": True, "nms": "conf 0.25, IoU 0.45, after every forward",
           "device": torch.cuda.get_device_name(dev), "power_limit_and_max_sm_clock": power_limit(),
           "rounds": args.rounds, "steps": args.steps, "warmup": args.warmup,
           "plain_images_per_s": round(med["plain"], 1), "tta_images_per_s": round(med["tta"], 1),
           "tta_over_plain": round(med["tta"] / med["plain"], 4),
           "plain_runs": [round(v, 1) for v in rates["plain"]], "tta_runs": [round(v, 1) for v in rates["tta"]],
           "median_sm_mhz_in_timed_windows": {a: statistics.median([c for c in clocks[a] if c is not None] or [0]) for a in arms},
           "clock_event_reasons_seen": {a: clocks[a + "_reasons"] for a in arms},
           "anchors": {"plain": g.A[0], "tta": g.A_tot},
           "kernels_batch64": kernels,
           "bf16_vs_fp32_engine": {"images": N_AGREE, **agreement}}
    if args.out:
        od = Path(args.out)
        od.mkdir(parents=True, exist_ok=True)
        (od / "bench_tta.json").write_text(json.dumps(res, indent=1))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
