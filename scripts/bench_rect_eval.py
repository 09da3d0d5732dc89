"""Rect-batch evaluation: one plan per input shape with buffers of its own against one shape arena (model.max_shape).

    python scripts/bench_rect_eval.py [--images 1000] [--batch 32] [--out DIR]

Data: a seeded synthetic set of uint8 BGR frames (smooth random blobs) whose sizes follow COCO's: long side 640, the
short side drawn from the common COCO aspect ratios (4:3 landscape and portrait dominate, then 3:2, 16:9, square ...).

Batches follow upstream YOLOv9's `--rect` evaluation (utils/dataloaders.py, LoadImagesAndLabels with rect=True,
pad=0.5): images sorted by h/w, cut into batches of --batch, and batch i letterboxed to
    shape_i = ceil(s_i * 640 / 32 + 0.5) * 32,   s_i = [maxi, 1] if every h/w of the batch is < 1,
                                                  [1, 1/mini] if every h/w is > 1, else [1, 1]     ([h, w])
so every batch of COCO-like images fits 672 x 672.  This arithmetic is restated from upstream; it could not be checked
against upstream's code here (no network).  Letterboxing here may scale up (the project's letterbox), where upstream's
val.py does not; both arms see the same inputs.

Per batch: letterbox (K8, `preprocess` into a per-shape input buffer) + gelan-c bf16 forward with CUDA graphs and static
outputs (model.max_batch = --batch) + multi-label NMS at conf 0.001 / IoU 0.7.  Two arms, one after the other, each on a
fresh model with the same weights:
  own    model.max_shape = None: every batch shape compiles a plan with buffers of its own;
  arena  model.max_shape = (672, 672): the plans of every shape take their buffers from one arena.
Reported per arm: distinct shapes, peak memory_allocated / memory_reserved (torch's counters; the frames and weights
included), the bytes each new shape's first forward added (its plan's buffers and weights: "per-plan bytes"), total
time spent in compile_model, the first pass (compile + graph capture + run) and the images/s of a second, steady
pass; and whether the two arms' detections are bit-identical.  The device name, power limit and maximum SM clock are
read in the same run.  Prints one JSON line and, with --out DIR, writes it to DIR/bench_rect_eval.json."""
from __future__ import annotations

import argparse
import json
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
for p in (ROOT, ROOT / "yolo-re_b200", ROOT / "scripts"):
    if str(p) not in sys.path:
        sys.path.insert(0, str(p))

import numpy as np
import torch

from bench_fp16 import power_limit

IMG = 640
STRIDE = 32
MAX_SHAPE = (672, 672)
# (w, h) aspect ratios of COCO images with their rough frequencies (640x480 and 480x640 make up most of the set)
ASPECTS = [((4, 3), 0.47), ((3, 4), 0.17), ((3, 2), 0.12), ((2, 3), 0.05), ((16, 9), 0.06), ((1, 1), 0.05),
           ((5, 4), 0.04), ((4, 5), 0.02), ((2, 1), 0.01), ((9, 16), 0.01)]


def synthetic_sizes(n: int, seed: int) -> list[tuple[int, int]]:
    """(h, w) of n images: long side 640, aspect ratio drawn from ASPECTS, short side jittered by a few pixels"""
    rng = np.random.default_rng(seed)
    ratios, p = zip(*ASPECTS)
    idx = rng.choice(len(ratios), size=n, p=np.array(p) / sum(p))
    out = []
    for i in idx:
        aw, ah = ratios[i]
        short = int(round(IMG * min(aw, ah) / max(aw, ah))) - int(rng.integers(0, 8))
        out.append((IMG, short) if ah >= aw else (short, IMG))
    return out


def frames(sizes, seed: int, dev) -> list[torch.Tensor]:
    """uint8 [h, w, 3] BGR frames on the device: bilinear upsampling of coarse random colours (blob-like content)"""
    g = torch.Generator(device=dev).manual_seed(seed)
    out = []
    for h, w in sizes:
        coarse = torch.rand((1, 3, h // 16 + 2, w // 16 + 2), generator=g, device=dev)
        img = torch.nn.functional.interpolate(coarse, size=(h, w), mode="bilinear", align_corners=False)
        out.append((img[0].permute(1, 2, 0) * 255).round().to(torch.uint8).contiguous())
    return out


def rect_batches(sizes, batch: int):
    """upstream's rect batching (module docstring): [(image indices, (H, W))], in aspect-ratio order"""
    ar = np.array([h / w for h, w in sizes])
    order = np.argsort(ar, kind="stable")
    out = []
    for b0 in range(0, len(order), batch):
        idx = order[b0:b0 + batch]
        mini, maxi = ar[idx].min(), ar[idx].max()
        s = [maxi, 1] if maxi < 1 else [1, 1 / mini] if mini > 1 else [1, 1]
        H, W = (np.ceil(np.array(s) * IMG / STRIDE + 0.5).astype(int) * STRIDE).tolist()
        out.append((idx.tolist(), (H, W)))
    return out


def run_arm(arm, sd, imgs, batches, batch, dev):
    import yolo_b200.engine as E
    from yolo_b200 import YOLO, non_max_suppression, preprocess

    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats(dev)
    m = YOLO.from_yaml(ROOT / "configs/models/gelan-c.yaml")
    m.load_state_dict(sd, strict=True)
    m = m.to(dev).eval().set_precision("bf16")
    m.max_batch = batch
    m.max_shape = MAX_SHAPE if arm == "arena" else None
    m.fresh_outputs, m.use_cuda_graph = False, True

    compile_s = [0.0]
    compile_model = E.compile_model

    def timed_compile(*a, **k):
        t0 = time.perf_counter()
        try:
            return compile_model(*a, **k)
        finally:
            compile_s[0] += time.perf_counter() - t0

    E.compile_model = timed_compile
    bufs: dict = {}
    per_plan: list[dict] = []

    def one_pass(keep):
        dets_all = []
        for idx, (H, W) in batches:
            new = (H, W) not in bufs
            if new:
                bufs[(H, W)] = torch.empty((batch, 3, H, W), dtype=torch.float32, device=dev)
                torch.cuda.synchronize(dev)
                before = torch.cuda.memory_allocated(dev)
            x = bufs[(H, W)][:len(idx)]
            preprocess([imgs[i] for i in idx], (H, W), out=x)
            y = m(x)[0]
            d = non_max_suppression(y.permute(0, 2, 1), 0.001, 0.7, multi_label=True)
            if new:
                torch.cuda.synchronize(dev)
                per_plan.append({"shape": [H, W], "bytes": torch.cuda.memory_allocated(dev) - before})
            if keep:
                dets_all.append([t.clone() for t in d])
        torch.cuda.synchronize(dev)
        return dets_all

    try:
        t0 = time.perf_counter()
        dets = one_pass(True)
        first_s = time.perf_counter() - t0
        t0 = time.perf_counter()
        one_pass(False)
        steady_s = time.perf_counter() - t0
    finally:
        E.compile_model = compile_model
    res = {"shapes": len(bufs), "plans": len(m._plans), "arenas": len(m._arenas),
           "arena_gib": [round(a.numel() / 2**30, 3) for a in m._arenas.values()],
           "peak_allocated_gib": round(torch.cuda.max_memory_allocated(dev) / 2**30, 3),
           "peak_reserved_gib": round(torch.cuda.max_memory_reserved(dev) / 2**30, 3),
           "compile_s": round(compile_s[0], 2), "first_pass_s": round(first_s, 2), "steady_pass_s": round(steady_s, 3),
           "images_per_s": round(len(imgs) / steady_s, 1),
           "per_plan_mib": [{"shape": p["shape"], "mib": round(p["bytes"] / 2**20, 1)} for p in per_plan]}
    if m._arena_weights:
        (_, wc), = m._arena_weights.values()
        res["shared_weight_mib"] = round(sum(t.numel() * t.element_size() for wb in wc.values() for t in wb) / 2**20, 1)
    del m, bufs
    torch.cuda.empty_cache()
    return res, [[t.cpu() for t in b] for b in dets]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=1000)
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", type=str, default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_rect_eval: needs a CUDA device")
    from oracle import gelan_ref as G
    dev = torch.device("cuda", 0)
    nodes, nc = G.load_graph(ROOT / "configs/models/gelan-c.yaml")
    sd = G.calibrated_state_dict(nodes, nc)
    sizes = synthetic_sizes(a.images, a.seed)
    imgs = frames(sizes, a.seed, dev)
    batches = rect_batches(sizes, a.batch)
    assert all(H <= MAX_SHAPE[0] and W <= MAX_SHAPE[1] for _, (H, W) in batches)

    res = {"gpu": torch.cuda.get_device_name(dev), "power_limit_and_max_sm_clock": power_limit(),
           "images": a.images, "batch": a.batch, "seed": a.seed, "model": "gelan-c", "precision": "bf16",
           "nms": "multi-label, conf 0.001, IoU 0.7", "max_shape": list(MAX_SHAPE),
           "batch_shapes": sorted({f"{H}x{W}" for _, (H, W) in batches})}
    dets = {}
    for arm in ("own", "arena"):
        res[arm], dets[arm] = run_arm(arm, sd, imgs, batches, a.batch, dev)
    same = all(torch.equal(u.view(torch.int32), v.view(torch.int32))
               for bu, bv in zip(dets["own"], dets["arena"]) for u, v in zip(bu, bv))
    res["detections_bit_identical"] = bool(same and len(dets["own"]) == len(dets["arena"]))
    res["detections"] = int(sum(t.shape[0] for b in dets["own"] for t in b))
    line = json.dumps(res)
    print(line)
    if a.out:
        Path(a.out).mkdir(parents=True, exist_ok=True)
        (Path(a.out) / "bench_rect_eval.json").write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
