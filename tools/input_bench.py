"""Input-pipeline measurement: the weak augmentation (ops.resize_pil) on a batch of eight Cityscapes frames, and what it replaces.

    python tools/input_bench.py --out DIR [--iters 200]

Writes DIR/input_bench.json with, next to the GPU name / power limit and the host CPU model / core count of the run:
  * resize_pil: device time of one launch on 8 random 1024x2048 HWC uint8 images -> 600x1200 (half flipped), inputs resident in
    HBM; four input batches (201 MB > the 126 MB L2) are rotated so that reads come from HBM; CUDA events around `iters`
    back-to-back launches from prebuilt plans (the host enqueues faster than the kernel runs).  Achieved bandwidth on the
    algorithmic bytes (3 H W read + 3 h w written per image) and its share of the copy bandwidth measured in the same run
    (device-to-device copy of 1 GiB, read + write bytes) and of DESIGN.md's 6549.4 GB/s;
  * the same step fed from pinned host memory: the 50 MB H2D copy and the launch inside the timed region;
  * weak_augment -> strong_augment -> normalize_pad for the batch (host draws included), CUDA events;
  * Pillow's resize + np.flip per image on one host core (Pillow's resampler is single-threaded), for comparison.
Starts no profiler.  Needs a CUDA device: without one it exits with an error.
"""
from __future__ import annotations

import argparse
import json
import os
import platform
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N, H, W, h, w = 8, 1024, 2048, 600, 1200
DESIGN_PEAK_GBS = 6549.4


def _gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True)
    line = q.stdout.strip().splitlines()[1] if q.returncode == 0 and len(q.stdout.strip().splitlines()) > 1 else ""
    name, _, power = line.partition(",")
    return {"gpu": name.strip() or torch.cuda.get_device_name(0), "power_limit": power.strip(), "nvidia_smi": q.stdout.strip()}


def _cpu_info() -> dict:
    model = platform.processor()
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    model = line.split(":", 1)[1].strip()
                    break
    except OSError:
        pass
    return {"cpu": model, "cpu_cores": os.cpu_count(), "cpu_cores_usable": len(os.sched_getaffinity(0))}


def _events_ms(fn, iters: int) -> float:
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(iters):
        fn(i)
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--iters", type=int, default=200)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("input_bench.py measures the GPU: no CUDA device")
    from sfod_b200 import config, engine, ops
    from PIL import Image

    dev = torch.device("cuda:0")
    res: dict = {"what": "weak augmentation of 8 x 1024x2048 uint8 HWC images -> 600x1200 CHW (Pillow BILINEAR + flip)"}
    res.update(_gpu_info())
    res.update(_cpu_info())
    flips = [bool(k % 2) for k in range(N)]

    # ---- copy bandwidth of this card, same run
    src = torch.empty(1 << 30, dtype=torch.uint8, device=dev)
    dst = torch.empty_like(src)
    for _ in range(3):
        dst.copy_(src)
    ms = _events_ms(lambda i: dst.copy_(src), 20)
    copy_gbs = 2 * src.numel() / (ms * 1e-3) / 1e9
    del src, dst
    res["copy_gbs_measured"] = round(copy_gbs, 1)

    # ---- resize_pil, inputs in HBM, four rotating batches
    g = torch.Generator(device=dev).manual_seed(1)
    batches = [torch.randint(0, 256, (N, H, W, 3), dtype=torch.uint8, device=dev, generator=g) for _ in range(4)]
    plans = [ops.ResizePlan(b, [(h, w)] * N, flips) for b in batches]
    out = torch.empty(plans[0].nbytes, dtype=torch.uint8, device=dev)
    for p in plans * 5:
        p.launch(out)
    torch.cuda.synchronize()
    launches = ops.launch_count()
    k_ms = _events_ms(lambda i: plans[i % 4].launch(out), args.iters)
    assert ops.launch_count() - launches == args.iters
    alg_bytes = N * 3 * (H * W + h * w)
    res["resize_pil"] = {
        "us_per_batch": round(k_ms * 1e3, 2), "iters": args.iters, "input_batches_rotated": 4,
        "input_bytes_rotated": 4 * N * 3 * H * W, "algorithmic_bytes": alg_bytes,
        "achieved_gbs": round(alg_bytes / (k_ms * 1e-3) / 1e9, 1),
        "share_of_copy_measured": round(alg_bytes / (k_ms * 1e-3) / 1e9 / copy_gbs, 3),
        "share_of_design_peak_6549": round(alg_bytes / (k_ms * 1e-3) / 1e9 / DESIGN_PEAK_GBS, 3),
    }
    # the public call (host work per call included), for reference
    res["resize_pil"]["ops_call_us"] = round(1e3 * _events_ms(lambda i: ops.resize_pil(batches[i % 4], [(h, w)] * N, flips), 50), 2)
    # bit-equality of one image of the timed batch against Pillow
    ref = np.asarray(Image.fromarray(batches[0][1].cpu().numpy()).resize((w, h), Image.BILINEAR))[:, ::-1].transpose(2, 0, 1)
    res["resize_pil"]["image1_equals_pillow"] = bool(np.array_equal(ops.resize_pil(batches[0], [(h, w)] * N, flips)[1].cpu().numpy(), ref))

    # ---- the same step fed from pinned host memory: H2D copy + launch
    pinned = batches[0].cpu().pin_memory()
    staging = torch.empty_like(batches[0])
    plan = ops.ResizePlan(staging, [(h, w)] * N, flips)

    def h2d_then_resize(i):
        staging.copy_(pinned, non_blocking=True)
        plan.launch(out)
    for i in range(3):
        h2d_then_resize(i)
    hd_ms = _events_ms(h2d_then_resize, max(args.iters // 4, 20))
    res["resize_pil_from_pinned_host"] = {"ms_per_batch": round(hd_ms, 3), "h2d_bytes": pinned.numel(),
                                          "h2d_gbs_incl_kernel": round(pinned.numel() / (hd_ms * 1e-3) / 1e9, 1)}

    # ---- weak -> strong -> normalize_pad, host draws included
    cfg = config.vgg_source_free_cfg()
    rng = np.random.RandomState(0)
    tg = torch.Generator().manual_seed(0)

    def chain(i):
        weak, _ = engine.weak_augment(batches[i % 4], cfg=cfg, rng=rng)
        strong = engine.strong_augment(weak, generator=tg)
        ops.normalize_pad(weak, cfg.MODEL.PIXEL_MEAN, cfg.MODEL.PIXEL_STD, 32)
        ops.normalize_pad(strong, cfg.MODEL.PIXEL_MEAN, cfg.MODEL.PIXEL_STD, 32)
    for i in range(3):
        chain(i)
    ch_ms = _events_ms(chain, 20)
    res["weak_strong_normalize_chain"] = {"ms_per_batch": round(ch_ms, 3), "iters": 20,
                                          "steps": "weak_augment, strong_augment (draws on the host), normalize_pad of the weak and the strong batch"}

    # ---- Pillow on one host core
    imgs = [b.cpu().numpy() for b in batches[0][:4]]
    t0 = time.perf_counter()
    reps = 0
    for _ in range(3):
        for k, im in enumerate(imgs):
            r = np.asarray(Image.fromarray(im).resize((w, h), Image.BILINEAR))
            if k % 2:
                r = np.ascontiguousarray(r[:, ::-1])
            reps += 1
    pil_ms = (time.perf_counter() - t0) / reps * 1e3
    res["pillow_resize_flip_ms_per_image_one_core"] = round(pil_ms, 2)
    res["pillow_cores_to_match_resize_pil"] = round(pil_ms * N / (k_ms), 1)

    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "input_bench.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
