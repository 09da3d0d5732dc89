"""4:2:0 YUV frame input (K14) against BGR frames (K8): gelan-c bf16, CUDA graphs, 64 x 1920x1080 frames -> 640x384, cuda:0.

    python scripts/bench_yuv.py [--rounds 3] [--steps 10] [--warmup 3] [--out DIR]

A step is one batch of 64 frames from pinned host memory to detections:
  bgr   host BGR  [64, 1080, 1920, 3] (398 MB) -> copy_(non_blocking) -> K8  -> model(x_u8) -> NMS with scale rows
  nv12  host NV12 [64, 1620, 1920]    (199 MB) -> copy_(non_blocking) -> K14 -> model(x_u8) -> NMS with scale rows
Both arms letterbox to the same uint8 640x384 batch (auto rect), so the model and NMS work is identical; what differs is
the upload and the letterbox kernel.  The 64 frames are seeded multi-octave noise encoded to NV12 (BT.601); the BGR arm's
frames are those NV12 frames converted as cv2.cvtColor converts them, so both arms must produce identical detections.
The arms alternate inside every round (the order flips every round), each warmed up before its timed window;
images/s = 64 x steps over the device-event time of the window, whose median SM clock and clock-event reasons are
recorded (bench.py's sampler).

Also reported:
  * the letterbox kernels on device-resident frames: CUDA events around 50 back-to-back launches of the 64-frame batch
    (two launches of 32 frames each) for K8 on BGR and K14 on NV12, in both output modes, with the bytes each must read
    and write over that time;
  * agreement: the two arms' letterboxed batches and detections compared bit for bit;
  * the host CPU time of cv2.cvtColor(COLOR_YUV2BGR_NV12) over the 64 frames (cv2's own thread pool), the cost of the
    host conversion a caller pays without K14.
The device name, power limit and maximum SM clock are read in the same run.  Prints one JSON line and, with --out DIR,
also writes it to DIR/bench_yuv.json (profiles/r03_bench_yuv.json is that file from a B200)."""
from __future__ import annotations

import argparse
import importlib
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

import ctypes as C

import numpy as np
import torch

from bench import ClockSampler
from bench_fp16 import power_limit

MODEL, H, W, S, BATCH = "gelan-c", 1080, 1920, 640, 64


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default="", metavar="DIR", help="also write the result to DIR/bench_yuv.json")
    args = ap.parse_args()
    if args.rounds < 1 or args.steps < 1:
        ap.error("--rounds and --steps must be at least 1")
    if not torch.cuda.is_available():
        raise SystemExit("bench_yuv.py needs a CUDA device (B200)")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)

    from oracle import gelan_ref as G
    from oracle import yuv_ref as Y
    from yolo_b200 import YOLO, _lib as L, nms_raw, preprocess, scale_rows
    PP = importlib.import_module("yolo_b200.preprocess")          # the module; the package exports the function by its name

    # ---- frames ----
    x = G.fractal(BATCH, H, torch.Generator().manual_seed(11), w=W)
    bgr_src = (x.permute(0, 2, 3, 1).flip(-1) * 255).round().clamp(0, 255).to(torch.uint8).numpy()
    del x
    nv12 = np.stack([Y.to_frame(*Y.encode_bt601(f), "nv12") for f in bgr_src])
    bgr = np.stack([Y.yuv420_to_bgr(f, "nv12") for f in nv12])
    del bgr_src
    host = {"bgr": torch.from_numpy(bgr).pin_memory(), "nv12": torch.from_numpy(nv12).pin_memory()}
    devbuf = {k: torch.empty(v.shape, dtype=torch.uint8, device=dev) for k, v in host.items()}

    # cv2.cvtColor on the host: what converting these frames costs a caller without K14
    try:
        import cv2
        assert all(np.array_equal(cv2.cvtColor(f, cv2.COLOR_YUV2BGR_NV12), b) for f, b in zip(nv12[:4], bgr[:4]))
        times = []
        for _ in range(3):
            t0 = time.perf_counter()
            for f in nv12:
                cv2.cvtColor(f, cv2.COLOR_YUV2BGR_NV12)
            times.append(time.perf_counter() - t0)
        cvt = {"ms_for_64_frames_median_of_3": round(1e3 * statistics.median(times), 2), "cv2": cv2.__version__,
               "cv2_threads": cv2.getNumThreads()}
    except ImportError:
        cvt = "cv2 not installed: not measured"

    # ---- model ----
    yaml_path = ROOT / "configs" / "models" / f"{MODEL}.yaml"
    nodes, nc = G.load_graph(yaml_path)
    m = YOLO.from_yaml(yaml_path)
    m.load_state_dict(G.calibrated_state_dict(nodes, nc), strict=True)
    m = m.to(dev).eval().set_precision("bf16")
    m.check_weights, m.fresh_outputs, m.use_cuda_graph = False, False, True

    xu = torch.empty((BATCH, 384, 640, 3), dtype=torch.uint8, device=dev)
    origs = [(H, W)] * BATCH
    last = {}

    def step(arm: str):
        devbuf[arm].copy_(host[arm], non_blocking=True)
        frames = list(devbuf[arm].unbind(0))
        _, ratios, pads = preprocess(frames, S, out=xu, dtype=torch.uint8, auto=True, fmt=arm)
        y, _ = m(xu)
        last[arm] = nms_raw(y.permute(0, 2, 1), 0.25, 0.45, scale=scale_rows(ratios, pads, origs, device=dev))

    # ---- agreement ----
    agree = {}
    for arm in ("bgr", "nv12"):
        step(arm)
        torch.cuda.synchronize()
        out, cnt, _ = last[arm]
        n = cnt.cpu()
        agree[arm] = (xu.clone(), [out[i, :int(n[i])].clone() for i in range(BATCH)])
    agreement = {"letterboxed_batches_identical": bool(torch.equal(agree["bgr"][0], agree["nv12"][0])),
                 "detections_identical": all(torch.equal(a, b) for a, b in zip(agree["bgr"][1], agree["nv12"][1])),
                 "detections": sum(len(d) for d in agree["nv12"][1])}
    del agree

    # ---- throughput ----
    arms = ("bgr", "nv12")
    for a in arms:
        for _ in range(args.warmup):
            step(a)
    torch.cuda.synchronize()
    rates, clocks = defaultdict(list), defaultdict(list)
    for r in range(args.rounds):
        for arm in (arms if r % 2 == 0 else arms[::-1]):
            sampler = ClockSampler(0)
            sampler.start()
            for _ in range(args.warmup):
                step(arm)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            sampler.begin()
            e0.record()
            for _ in range(args.steps):
                step(arm)
            e1.record()
            torch.cuda.synchronize()
            sampler.end()
            rates[arm].append(BATCH * args.steps / (e0.elapsed_time(e1) / 1e3))
            c = sampler.stop()
            clocks[arm].append(c.get("sm_mhz"))
            clocks[arm + "_reasons"] += [s for s in c.get("reasons", []) if s not in clocks[arm + "_reasons"]]
    med = {a: statistics.median(v) for a, v in rates.items()}

    # ---- the letterbox kernels on device-resident frames ----
    lib, stream = L.lib(), torch.cuda.current_stream().cuda_stream
    kernels = {}
    for arm in arms:
        frames = list(devbuf[arm].unbind(0))
        srcs = [PP._Source(f, arm, "bt601") for f in frames]
        for mode, dtype, shape in ((L.LB_U8_HWC, torch.uint8, (BATCH, 384, 640, 3)), (L.LB_F32_CHW, torch.float32, (BATCH, 3, 384, 640))):
            out = torch.empty(shape, dtype=dtype, device=dev)
            descs = (L.LetterboxDesc * BATCH)()
            for i, s in enumerate(srcs):
                d, _, _ = PP._desc(s, S, (114, 114, 114), 32)
                d.out_mode, d.dst = mode, out[i].data_ptr()
                descs[i] = d
            if arm == "bgr":
                launch = lambda: L.check(lib.yre_letterbox_u8_batch(descs, BATCH, C.c_void_p(stream)))
            else:
                planes = (L.Yuv420Planes * BATCH)(*(s.planes for s in srcs))
                launch = lambda: L.check(lib.yre_letterbox_yuv420_batch(descs, planes, BATCH, C.c_void_p(stream)))
            launch()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 50
            e0.record()
            for _ in range(reps):
                launch()
            e1.record()
            torch.cuda.synchronize()
            us = e0.elapsed_time(e1) * 1e3 / reps
            # every source byte the resize can touch is read at most once (rows 1080 -> 360: two of every three rows)
            nbytes = devbuf[arm].nbytes + out.nbytes
            kernels[f"{'k8_bgr' if arm == 'bgr' else 'k14_nv12'}_{'u8_hwc' if mode == L.LB_U8_HWC else 'f32_chw'}"] = {
                "us_per_64_frames": round(us, 1), "source_plus_output_bytes": nbytes, "gb_per_s_over_those_bytes": round(nbytes / us / 1e3, 1)}
    kernels["k14_over_k8_u8_hwc"] = round(kernels["k14_nv12_u8_hwc"]["us_per_64_frames"] / kernels["k8_bgr_u8_hwc"]["us_per_64_frames"], 4)
    kernels["k14_over_k8_f32_chw"] = round(kernels["k14_nv12_f32_chw"]["us_per_64_frames"] / kernels["k8_bgr_f32_chw"]["us_per_64_frames"], 4)

    res = {"model": MODEL, "precision": "bf16", "cuda_graph": True, "batch": BATCH,
           "input": f"{BATCH} x {W}x{H} frames in pinned host memory, letterboxed to 640x384 (auto rect), uint8 to the stem",
           "nms": "conf 0.25, IoU 0.45, boxes scaled to frame pixels, after every forward",
           "device": torch.cuda.get_device_name(dev), "power_limit_and_max_sm_clock": power_limit(),
           "rounds": args.rounds, "steps": args.steps, "warmup": args.warmup,
           "bytes_uploaded_per_step": {a: host[a].nbytes for a in arms},
           "bgr_images_per_s": round(med["bgr"], 1), "nv12_images_per_s": round(med["nv12"], 1),
           "nv12_over_bgr": round(med["nv12"] / med["bgr"], 4),
           "bgr_runs": [round(v, 1) for v in rates["bgr"]], "nv12_runs": [round(v, 1) for v in rates["nv12"]],
           "median_sm_mhz_in_timed_windows": {a: statistics.median([c for c in clocks[a] if c is not None] or [0]) for a in arms},
           "clock_event_reasons_seen": {a: clocks[a + "_reasons"] for a in arms},
           "letterbox_kernels_device_resident": kernels,
           "agreement_bgr_vs_nv12": agreement,
           "host_cv2_cvtColor_nv12_to_bgr": cvt,
           "multi_gpu": "not measured (one GPU)"}
    if args.out:
        od = Path(args.out)
        od.mkdir(parents=True, exist_ok=True)
        (od / "bench_yuv.json").write_text(json.dumps(res, indent=1))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
