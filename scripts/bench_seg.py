"""Instance segmentation (gelan-c-seg) against detection (gelan-c): bf16, 640², batch 64, CUDA graphs, cuda:0.

    python scripts/bench_seg.py [--rounds 3] [--steps 10] [--warmup 3] [--out DIR]

Arms, alternated inside every round (the order flips every round), each warmed up before its timed window:
  det  gelan-c forward (graph replay) + NMS at conf 0.25
  seg  gelan-c-seg forward (graph replay) + NMS at conf 0.25 + K15 input-resolution masks ("input" mode)
images/s = 64 x steps over the device-event time of the window; the median SM clock and clock-event reasons inside the
windows are recorded (bench.py's sampler).  The two models share the detection weights (the oracle's calibrated
state_dict), so the detections of both arms are the same and are compared.

Also reported, with CUDA events around back-to-back launches:
  * K15 in "proto" mode on upstream val's NMS setting (multi-label, conf 0.001, IoU 0.7, max_det 300): the masks of up to
    300 detections per image at 160²;
  * K15 in "input" mode on the conf 0.25 detections, with the bytes of mask rows it writes;
  * the prototype branch's and the mask towers' share of the seg plan: each op launched on its own (plan.run_op) against
    one eager run of the whole plan.
The device name, power limit and maximum SM clock are read in the same run.  Prints one JSON line and, with --out DIR,
also writes it to DIR/bench_seg.json (profiles/r03_bench_seg.json is that file from a B200)."""
from __future__ import annotations

import argparse
import json
import statistics
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
for p in (ROOT, ROOT / "yolo-re_b200", ROOT / "scripts"):
    if str(p) not in sys.path:
        sys.path.insert(0, str(p))

import torch

from bench import ClockSampler
from bench_data import make_inputs
from bench_fp16 import power_limit

BATCH, IMG = 64, 640


def events_ms(fn, n: int) -> float:
    """ms per call of fn over n back-to-back calls, CUDA events"""
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / n


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default="", metavar="DIR", help="also write the result to DIR/bench_seg.json")
    args = ap.parse_args()
    if args.rounds < 1 or args.steps < 1:
        ap.error("--rounds and --steps must be at least 1")
    if not torch.cuda.is_available():
        sys.exit("bench_seg needs a CUDA device (a B200)")
    from oracle import seg_ref as S
    from yolo_b200 import YOLO, masks_raw, nms_raw

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    nodes, nc, nm, npr = S.load_graph(ROOT / "configs/models/gelan-c-seg.yaml")
    sd = S.calibrated_state_dict(nodes, nc, nm, npr)
    models = {}
    for arm, cfg in (("det", "gelan-c"), ("seg", "gelan-c-seg")):
        m = YOLO.from_yaml(ROOT / "configs/models" / f"{cfg}.yaml")
        keys = set(m.state_dict())
        m.load_state_dict({k: v for k, v in sd.items() if k in keys}, strict=True)
        m = m.to(dev).eval().set_precision("bf16")
        m.fresh_outputs, m.use_cuda_graph = False, True
        models[arm] = m
    x = make_inputs(BATCH, IMG, seed=7).to(dev)
    res = {}

    def step(arm: str):
        if arm == "det":
            y, _ = models["det"](x)
            res[arm] = nms_raw(y.permute(0, 2, 1), 0.25, 0.45)
        else:
            y, (_, mc, proto) = models["seg"](x)
            out, counts, keep = nms_raw(y.permute(0, 2, 1), 0.25, 0.45)
            res[arm] = (out, counts, keep, masks_raw(proto, mc, out, counts, keep, "input", shape=(IMG, IMG)))

    rates = {"det": [], "seg": []}
    clocks = []
    for r in range(args.rounds):
        for arm in (("det", "seg") if r % 2 == 0 else ("seg", "det")):
            for _ in range(args.warmup):
                step(arm)
            torch.cuda.synchronize()
            sampler = ClockSampler(0)
            sampler.start()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            sampler.begin()
            a.record()
            for _ in range(args.steps):
                step(arm)
            b.record()
            b.synchronize()
            sampler.end()
            clocks.append(sampler.stop())
            rates[arm].append(BATCH * args.steps / (a.elapsed_time(b) / 1e3))
    torch.cuda.synchronize()
    od, cd, _ = res["det"]
    os_, cs, ks, masks = res["seg"]
    same = torch.equal(cd, cs) and all(torch.equal(od[i, :int(cd[i])], os_[i, :int(cd[i])]) for i in range(BATCH))
    kept = int(cs.sum())

    # K15 alone
    seg = models["seg"]
    y, (_, mc, proto) = seg(x)
    vo, vc, vk = nms_raw(y.permute(0, 2, 1), 0.001, 0.7, max_det=300, multi_label=True)
    t_proto = events_ms(lambda: masks_raw(proto, mc, vo, vc, vk, "proto", shape=(IMG, IMG)), 20)
    kept_val = int(vc.sum())
    t_input = events_ms(lambda: masks_raw(proto, mc, os_, cs, ks, "input", shape=(IMG, IMG)), 20)

    # the prototype branch's and the mask towers' share of the plan
    p = next(iter(seg._plans.values()))
    n_ops = len(p.trace)
    proto_ops, mask_ops = range(n_ops - 14, n_ops - 10), range(n_ops - 10, n_ops - 1)
    t_plan = events_ms(p.run, 10)
    t_ops = {i: events_ms(lambda i=i: p.run_op(i), 10) for i in list(proto_ops) + list(mask_ops) + [n_ops - 1]}
    descs = p.op_descriptions()

    out = {
        "metric": "images/s, gelan-c-seg forward + NMS (conf 0.25) + K15 input-resolution masks vs gelan-c forward + NMS",
        "device": torch.cuda.get_device_name(dev), "power_limit_and_max_sm_clock": power_limit(),
        "batch": BATCH, "img": IMG, "precision": "bf16", "cuda_graphs": True,
        "rounds": args.rounds, "steps": args.steps, "warmup": args.warmup,
        "images_per_s": {k: {"median": statistics.median(v), "all": v} for k, v in rates.items()},
        "seg_over_det": statistics.median(rates["seg"]) / statistics.median(rates["det"]),
        "detections_identical": bool(same), "kept_conf_0.25": kept,
        "mask_bytes_written_conf_0.25": kept * IMG * IMG,
        "k15_ms": {"proto_mode_val_setting": t_proto, "kept_val_setting": kept_val,
                   "proto_mode_bytes_written": kept_val * (IMG // 4) ** 2,
                   "input_mode_conf_0.25": t_input, "kept_conf_0.25": kept},
        "plan_ms_eager": t_plan,
        "proto_branch_ms": {descs[i]: t_ops[i] for i in proto_ops},
        "mask_towers_ms": sum(t_ops[i] for i in mask_ops),
        "decode_masks_ms": t_ops[n_ops - 1],
        "proto_branch_share": sum(t_ops[i] for i in proto_ops) / t_plan,
        "mask_towers_share": sum(t_ops[i] for i in mask_ops) / t_plan,
        "sm_clock_samples": clocks,
        "tcgen05_convs": p.num_tcgen05,
    }
    line = json.dumps(out)
    print(line)
    if args.out:
        Path(args.out).mkdir(parents=True, exist_ok=True)
        (Path(args.out) / "bench_seg.json").write_text(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
