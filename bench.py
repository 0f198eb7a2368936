"""bench.py -- pseudo-labelled images/s of the teacher pseudo-labelling hot path (BASELINE.json metric).

Workload (BASELINE.json configs[2], teacher half): Faster R-CNN VGG16-BN teacher of
faster_rcnn_VGG_cityscapes_foggy_adaptive_teacher_source_free, batch 8 images/GPU of synthetic 600x1200 Cityscapes-shaped
uint8 images, 8 classes, random-init weights (seed 42), teacher in train() mode under no_grad exactly as the reference runs
it.  One step = preprocess -> backbone (cuDNN convs; BatchNorm statistics + normalise+ReLU on the sm_100a kernels)
-> PseudoLabRPN (fused decode/top-k/NMS kernel chain) -> ROIAlignV2 kernel -> box head (cuBLAS) -> fused Fast R-CNN
post-process + pseudo-label filter -> List[Instances] pseudo-labels, followed by one mean-teacher EMA launch.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
    python bench.py --impl reference [...]                         # the reference's CPU path (oracle) on the host cores
    python bench.py [...] --dump-outputs DIR                       # + the last timed step's outputs as DIR/<name>.npy

Under torchrun (N > 1) every rank owns a teacher replica and its own 8 images (no data-path collective: weak scaling);
timing is barrier + synchronize on both sides, CUDA events, max over ranks; rank 0 prints ONE JSON line.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "pseudo_labelled_images_per_s"
UNIT = "images/s"
IMAGE_HW = (600, 1200)
NUM_CLASSES = 8
WORKLOADS = {
    "vgg": ("configs[2] teacher half: faster_rcnn_VGG_cityscapes_foggy_adaptive_teacher_source_free, VGG16-BN teacher "
            "pseudo-labelling (train-mode BN, RPN 9990->2000, ROIAlignV2, per-class NMS, >0.8 filter) + EMA, "
            "synthetic 600x1200 uint8, 8 classes, random init"),
    "r101": ("configs[4] teacher half: r101_c4_cs_foggy_adaptive_teacher_source_free, ResNet-101-C4 teacher pseudo-labelling "
             "(83 train-mode BN + 11 frozen BN layers with ReLU / residual fusions, RPN 34200->12000->2000, ROIAlignV2 on 1024x38x75, "
             "FC 2048, per-class NMS, >0.8 filter) + EMA, synthetic 600x1200 uint8, 8 classes, random init"),
}
WORKLOAD = WORKLOADS["vgg"]


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="vgg", choices=sorted(WORKLOADS),
                    help="vgg = BASELINE configs[2] (headline, the driver's default); r101 = configs[4] (ResNet-101-C4 teacher)")
    ap.add_argument("--batch", type=int, default=8, help="images per GPU per step (configs[2]: 8)")
    ap.add_argument("--num-classes", type=int, default=8,
                    help="foreground classes K of the ROI heads (8 = Cityscapes, every shipped YAML; 1 = the 'Sim10k-shaped 1-class "
                         "variant' BASELINE.json names with configs[4] -- a benchmark variant, SURVEY.md section 8(d))")
    ap.add_argument("--extras", type=int, default=1,
                    help="1 = after the headline measurement also report: the named kernels' rooflines (NMS / ROIAlign / EMA at the bench "
                         "and the N=1 config-[1] shapes), the PyTorch-default (TF32) library-math record, the AdaBN step with its "
                         "statistic all-reduce (configs[3]), the CUDA-graph record and a live exp-flip-rate sample")
    ap.add_argument("--tf32", type=int, default=0, help="1 = let cuDNN/cuBLAS use TF32 for the (library) convs/FCs")
    ap.add_argument("--channels-last", type=int, default=0, help="1 = run the backbone in NHWC")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--sfod-step", type=int, default=1,
                    help="1 = also time the full mean-teacher step of configs[2] (teacher pseudo-labelling, student forward/backward "
                         "on the pseudo-labels through the same plugins, DDP gradient all-reduce for N > 1, SGD step, EMA); reported as "
                         "the extra object `sfod_step`, it does not enter `value`")
    ap.add_argument("--profiler-range", action="store_true",
                    help="bracket the timed region with cudaProfilerStart/Stop (for `ncu --profile-from-start off`); "
                         "numbers printed under a profiler are not bench values")
    ap.add_argument("--cpu-budget-s", type=float, default=150.0, help="wall-clock budget of the reference arm")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed (RPN proposals, detections, pseudo-labels, "
                         "a seeded sample of the EMA-updated teacher state) as DIR/<name>.npy, float32, so that two builds can be "
                         "compared output for output (the inputs are seeded: the same arguments give the same inputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl b200)")
    return args


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def synth_images(batch: int, seed: int):
    import torch
    g = torch.Generator().manual_seed(seed)
    return torch.randint(0, 256, (batch, 3) + IMAGE_HW, dtype=torch.uint8, generator=g)


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons through NVML every 100 ms while the timed region runs."""
    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x10: "sync_boost",
               0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.mask, self.max_mhz, self.stop_flag, self.ok = index, [], 0, None, threading.Event(), False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and all(v.strip().isdigit() for v in vis.split(",")) else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        while not self.stop_flag.is_set():
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                self.mask |= int(self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
            except Exception:
                pass
            time.sleep(0.1)

    def result(self):
        self.stop_flag.set()
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml_unavailable"]}
        s = sorted(self.samples)
        reasons = [n for b, n in self.REASONS.items() if self.mask & b and n != "gpu_idle"]
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": reasons, "samples": len(s)}


# ------------------------------------------------------------------------------------------------ reference arm (CPU)
def build_cfg(workload: str):
    from sfod_b200 import config
    cfg = config.vgg_source_free_cfg() if workload == "vgg" else config.r101_c4_source_free_cfg()
    cfg.MODEL.ROI_HEADS.NUM_CLASSES = NUM_CLASSES
    return cfg


def workload_name(workload: str) -> str:
    name = WORKLOADS[workload]
    return name if NUM_CLASSES == 8 else name.replace("8 classes", f"{NUM_CLASSES} class(es) (--num-classes; benchmark variant)")


def cpu_reference_run(steps: int, warmup: int, budget_s: float, seed: int = 1234, images_per_step: int = 8, with_ema: bool = True,
                      workload: str = "vgg"):
    """Times the oracle (CPU restatement of the reference's path) on all host cores: each step pseudo-labels
    ``images_per_step`` synthetic image(s) (one batch, like the GPU arm) and performs one EMA update.  Returns (images/s, dict)."""
    import torch
    from oracle import teacher_cpu
    import sfod_b200  # noqa: F401  (only for the model definition that supplies the random-init state_dict)
    from sfod_b200 import modeling

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    torch.manual_seed(42)
    cfg = build_cfg(workload)
    cfg.MODEL.DEVICE = "cpu"
    teacher_sd = {k: v.clone() for k, v in modeling.SourceFreeAdaptiveTeacherGeneralizedRCNN(cfg).state_dict().items()}
    student_sd = {k: (v + 0.01 * torch.randn_like(v) if v.is_floating_point() else v.clone()) for k, v in teacher_sd.items()}
    imgs = synth_images(images_per_step, seed)
    kw = dict(sizes=(64, 128, 256, 512), stride=16) if workload == "r101" else {}

    def step():
        out = teacher_cpu.teacher_pseudo_label(teacher_sd, imgs, training=True, num_classes=NUM_CLASSES, bbox_threshold=0.8, **kw)
        if with_ema:
            teacher_cpu.ema_update(student_sd, teacher_sd, 0.9996)
        return out

    t0 = time.perf_counter()
    step()
    first = time.perf_counter() - t0
    w_done = 1
    per = first   # the first step pays for thread pools and primitive caches: size the sample by a warm step when one fits
    # bounded sample: shrink the number of executed steps if K+W steps would blow the wall-clock budget
    w_run = min(warmup - 1, max(1, int((budget_s * 0.25) // max(first, 1e-3)))) if (warmup > 1 and first < 0.25 * budget_s) else 0
    for _ in range(w_run):
        tw = time.perf_counter()
        step()
        per = time.perf_counter() - tw
        w_done += 1
    left = budget_s - (time.perf_counter() - t0)
    k_run = max(1, min(steps, int(left // max(per, 1e-3))))
    t1 = time.perf_counter()
    for _ in range(k_run):
        step()
    dt = time.perf_counter() - t1
    value = images_per_step * k_run / dt
    info = {"value": round(value, 4), "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{k_run} timed step(s) of {images_per_step} image(s) 600x1200 (+{w_done} warm-up), full teacher pseudo-labelling "
                      f"+ EMA on torch-CPU/torchvision-CPU, {1e3 * dt / k_run:.0f} ms/step"}
    return value, info, k_run, w_done, dt


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    value, info, k_run, w_done, dt = cpu_reference_run(args.steps, args.warmup, args.cpu_budget_s, images_per_step=args.batch,
                                                       workload=args.workload)
    line = {"impl": "reference", "metric": METRIC, "value": info["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": k_run,
            "warmup": w_done, "ms_per_step": round(1e3 * dt / k_run, 3), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(args.workload), "images_per_gpu": args.batch, "images_per_step": args.batch,
                       "global_batch": args.batch, "image_hw": list(IMAGE_HW), "num_classes": NUM_CLASSES,
                       "note": "CPU arm runs on rank 0 only, all host cores; same batch per step as the GPU arm, bounded number of steps"},
            "cpu_baseline": info,
            "e2e": {"value": info["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)
    return 0


# ------------------------------------------------------------------------------------------------ B200 arm: helpers
_FLUSH = None


def flush_l2(dev):
    """Writes a buffer larger than the 126 MB L2 (timing hygiene of the per-kernel measurements)."""
    import torch
    global _FLUSH
    if _FLUSH is None:
        _FLUSH = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    _FLUSH.zero_()


def event_time_us(fn, dev, iters=7, warmup=3):
    """Median device time of ``fn`` in microseconds: CUDA events on the launching stream, L2 flushed before every timed call.
    All iterations are enqueued behind a ~2 ms spin kernel without a synchronize in between, so the host runs ahead of the
    device and the interval between the two events of a call holds device time only -- with a synchronize per iteration a
    call of a few tens of microseconds is dominated by the host's launch latency (ROIAlign backward through autograd: 46 us
    measured that way, 34 us on the device).  A ``fn`` that synchronizes internally (``ops.nms`` returns a host-sized tensor)
    simply drains the queue and is timed as before."""
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize(dev)
    torch.cuda._sleep(4_000_000)
    evs = []
    for _ in range(iters):
        flush_l2(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record()
        evs.append((e0, e1))
    torch.cuda.synchronize(dev)
    ts = sorted(a.elapsed_time(b) * 1e3 for a, b in evs)
    return ts[len(ts) // 2]


def named_kernel_rooflines(dev, peak, ema_plan):
    """BASELINE.json's metric names three kernels: NMS, ROIAlign, EMA.  Each is timed alone (CUDA events, L2 flushed) at the
    bench shape (8 images/GPU) and at the literal config-[1] shape (1 image, 2000 proposals); achieved = SURVEY.md 8(d)
    algorithmic bytes / time.  NMS is latency-bound: us/image and IoU pairs/s are the meaningful figures."""
    import torch
    from sfod_b200 import ops, synth
    out = {}
    try:
        for tag, N in (("config1_shape_N1", 1), ("bench_shape_N8", 8)):
            rec = {}
            for cname, cfg in (("V", synth.V), ("R101", synth.R101)):
                x = synth.features(cfg, N, 1).to(dev)
                logits, deltas, cell, _ = synth.rpn_head_outputs(cfg, N, 2)
                boxes, _, _, _, _ = ops.rpn_select(logits.to(dev), deltas.to(dev), [cfg["image"]] * N, cell_anchors=cell,
                                                   feat_hw=(cfg["H"], cfg["W"]), stride=cfg["stride"], post_nms_topk=2000)
                rois = ops.convert_boxes_to_roi_format([boxes[i] for i in range(N)])
                R, C, H, W = rois.shape[0], cfg["C"], cfg["H"], cfg["W"]
                alg = 4.0 * (N * C * H * W + 5 * R + 49 * R * C)
                us = event_time_us(lambda: ops.roi_align(x, rois, (7, 7), 1.0 / cfg["stride"], 0, True), dev)
                rec[f"roi_align_fwd_{cname}"] = {"us": round(us, 1), "R": R, "alg_MB": round(alg / 1e6, 1), "GBps": round(alg / us / 1e3, 1),
                                                 "frac": round(alg / us / 1e3 / peak, 3)}
                if cname == "V" or N == 1:
                    Rb = 512 * N
                    rb = rois[torch.randperm(R, device=dev)[:Rb]].contiguous()
                    xg = x.clone().requires_grad_(True)
                    y = ops.roi_align(xg, rb, (7, 7), 1.0 / cfg["stride"], 0, True)
                    g = torch.randn_like(y)
                    algb = 4.0 * (49 * Rb * C + 5 * Rb + N * C * H * W)
                    us = event_time_us(lambda: torch.autograd.grad(y, xg, g, retain_graph=True), dev)
                    rec[f"roi_align_bwd_{cname}"] = {"us": round(us, 1), "R": Rb, "alg_MB": round(algb / 1e6, 1), "GBps": round(algb / us / 1e3, 1),
                                                     "frac": round(algb / us / 1e3 / peak, 3)}
                    del xg, y, g
                del x
            # NMS inside RPN selection: the sorted, clipped candidates of the VGG teacher (9990 boxes -> 2000 kept per image)
            logits, deltas, cell, _ = synth.rpn_head_outputs(synth.V, N, 3)
            ld, dd = logits.to(dev), deltas.to(dev)
            us = event_time_us(lambda: ops.rpn_select(ld, dd, [synth.V["image"]] * N, cell_anchors=cell, feat_hw=(18, 37), stride=32), dev)
            hwa = logits.shape[1]
            alg = N * (20.0 * hwa + 20.0 * 2000)
            rec["rpn_select_V"] = {"us": round(us, 1), "us_per_image": round(us / N, 1), "GBps": round(alg / us / 1e3, 2),
                                   "frac": round(alg / us / 1e3 / peak, 5), "bound": "latency"}
            if N == 1:
                for kind in ("low", "high"):
                    b, sc = (synth.boxes_low_suppression(synth.V, 9990, 1234) if kind == "low" else synth.boxes_high_suppression(9990, 1234))
                    bd, sd = b.to(dev), sc.to(dev)
                    keep = ops.nms(bd, sd, 0.7)
                    us = event_time_us(lambda: ops.nms(bd, sd, 0.7), dev)
                    n, k = b.shape[0], keep.numel()
                    rec[f"nms_{kind}_suppression_n{n}"] = {"us": round(us, 1), "kept": int(k), "alg_GBps": round((20.0 * n + 8.0 * k) / us / 1e3, 3),
                                                           "upper_triangle_pairs_per_s": round(n * (n - 1) / 2 / (us * 1e-6), 0), "bound": "latency"}
            out[tag] = rec
        us = event_time_us(lambda: ema_plan.step(0.9996), dev)
        out["ema_multi_tensor"] = {"us": round(us, 1), "elements": int(ema_plan.numel), "alg_MB": round(12.0 * ema_plan.numel / 1e6, 1),
                                   "GBps": round(12.0 * ema_plan.numel / us / 1e3, 1), "frac": round(12.0 * ema_plan.numel / us / 1e3 / peak, 3)}
        out["how"] = ("each call timed alone: CUDA events on the launching stream, median of 7 after 3 warm-ups, 256 MB L2 flush before each; the 7 "
                      "iterations are enqueued back to back behind a 2 ms spin kernel (no synchronize in between), i.e. device time without the host's launch latency")
    except Exception as e:   # a report, never a reason to lose the headline
        out["error"] = repr(e)[:300]
    return out


def flip_rate_sample(dev, seeds: int = 12):
    """Live sample of how often the CUDA path's defined exp / softmax changes a discrete result relative to ATen-CPU's (the
    reference's arithmetic): RPN keep sets and Fast R-CNN detection / pseudo-label sets for a few seeds (CPU oracle in a process
    pool).  The 200-seed measurement is tests/test_gpu_flip_rate.py -> profiles/r2_flip_rate.json."""
    import torch
    try:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import flip_workers as fw
        from sfod_b200 import ops, synth
        jobs = [("rpn", c, 9000 + s, False) for c in ("V_low", "V_high") for s in range(seeds)] + \
               [("frcnn", k, 9500 + s, False) for k in fw.FRCNN_CASES for s in range(seeds)]
        oracle = fw.run_jobs(jobs)
        imgs = sets = elems = total = 0
        for case in ("V_low", "V_high"):
            cfg = synth.V
            for s in range(seeds):
                logits, deltas, cell, _ = synth.rpn_head_outputs(cfg, 1, 9000 + s, fw.RPN_CASES[case][1])
                _, _, src, cnt, _ = ops.rpn_select(logits.to(dev), deltas.to(dev), [fw.IMAGE], cell_anchors=cell, feat_hw=(18, 37), stride=32)
                a = set(src[0, :int(cnt[0])].cpu().tolist()); b = set(oracle[("rpn", case, 9000 + s)]["aten_src"].tolist())
                imgs += 1; sets += bool(a ^ b); elems += len(a ^ b); total += len(b)
        for kind in fw.FRCNN_CASES:
            for s in range(seeds):
                cls, dl, props = fw.frcnn_inputs(kind, 9500 + s)
                o = ops.frcnn_postprocess(cls.to(dev), dl.to(dev), props.to(dev), [len(props)], [fw.IMAGE], pseudo_thresh=0.8)
                k = int(o["count"][0])
                a = set(zip(o["rows"][0, :k].cpu().tolist(), o["classes"][0, :k].cpu().tolist()))
                r = oracle[("frcnn", kind, 9500 + s)]["aten"]
                b = set(zip(r["kept_rows"].tolist(), r["pred_classes"].tolist()))
                imgs += 1; sets += bool(a ^ b); elems += len(a ^ b); total += len(b)
        return {"images": imgs, "sets_differing": sets, "elements_differing": elems, "elements": total,
                "vs": "ATen-CPU exp/softmax oracle (reference-faithful); CUDA path == defined-arithmetic oracle bit for bit",
                "full_measurement": "profiles/r2_flip_rate.json (200 seeds x 6 cases: 0 of 1200 images differ)"}
    except Exception as e:
        return {"error": repr(e)[:300]}


# What one step returns (step_resident): per image, the RPN proposals, the Fast R-CNN detections and the pseudo-labels
DUMP_FIELDS = (("rpn", ("proposal_boxes", "objectness_logits")),
               ("detections", ("pred_boxes", "scores", "pred_classes")),
               ("pseudo_labels", ("gt_boxes", "gt_classes", "scores")))
DUMP_STATE_SAMPLE = 4096          # elements drawn from each floating-point tensor of the teacher state
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, out, teacher, max_rows):
    """Writes the results ``out`` of the last timed step as float32 .npy files under ``out_dir``: every field of DUMP_FIELDS
    as one (images, max_rows[list], ...) array (``<list>_<field>.npy``) whose rows past an image's count are zero, the rows of
    each image (``<list>_per_image.npy``), and ``teacher_state_sample.npy``, a fixed, seeded sample of every floating-point
    tensor of the teacher's state_dict (in state_dict order) after the step's EMA and train-mode BatchNorm running-statistic
    updates.  The shapes follow from the configuration alone, so every file exists and two builds line up image by image
    even where their counts differ (the random-init teacher of the benchmark scores no detection above the pseudo-label
    threshold: its pseudo-label fields are all padding)."""
    import numpy as np
    import torch
    arrays = {}
    for (name, fields), insts in zip(DUMP_FIELDS, out):
        counts = [len(p) for p in insts]
        if max(counts) > max_rows[name]:
            raise RuntimeError(f"--dump-outputs: {name} has {max(counts)} rows in an image, more than {max_rows[name]}")
        arrays[f"{name}_per_image"] = torch.tensor(counts, dtype=torch.float32)
        for f in fields:
            vals = [getattr(v, "tensor", v).float() for v in (p.get(f) for p in insts)]
            padded = vals[0].new_zeros((len(vals), max_rows[name]) + vals[0].shape[1:])
            for i, v in enumerate(vals):
                padded[i, :len(v)] = v
            arrays[f"{name}_{f}"] = padded
    g = torch.Generator().manual_seed(0)
    sample = []
    for v in teacher.state_dict().values():
        if v.is_floating_point():
            flat = v.detach().reshape(-1)
            n = flat.numel()
            idx = torch.randint(n, (DUMP_STATE_SAMPLE,), generator=g) if n > DUMP_STATE_SAMPLE else torch.arange(n)
            sample.append(flat[idx.to(flat.device)].float())
    arrays["teacher_state_sample"] = torch.cat(sample)
    arrays = {k: v.cpu().numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_MAX_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


# ------------------------------------------------------------------------------------------------ B200 arm
def run_b200(args):
    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py measures the CUDA path: no CUDA device is visible (there is no CPU fallback)")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    import sfod_b200  # noqa: F401
    from sfod_b200 import engine, modeling, ops

    def set_math(tf32: bool):
        torch.backends.cudnn.allow_tf32 = bool(tf32)
        torch.backends.cuda.matmul.allow_tf32 = bool(tf32)
    set_math(args.tf32)
    torch.backends.cudnn.benchmark = True

    torch.manual_seed(42)  # SEED: 42 of the reference config; identical weights on every rank
    cfg = build_cfg(args.workload)
    cfg.MODEL.DEVICE = "cpu"
    teacher = modeling.SourceFreeAdaptiveTeacherGeneralizedRCNN(cfg)
    student = modeling.SourceFreeAdaptiveTeacherGeneralizedRCNN(cfg)
    student.load_state_dict(teacher.state_dict())
    with torch.no_grad():
        for p in student.parameters():
            p.add_(0.01 * torch.randn_like(p))
    teacher.to(dev).train()   # the reference never .eval()s the teacher (SURVEY.md fact 3)
    student.to(dev).train()
    if args.channels_last:
        teacher.to(memory_format=torch.channels_last)
        student.to(memory_format=torch.channels_last)
    ema = engine.TeacherEMA(student, teacher, world_size=1)
    thr = cfg.SEMISUPNET.BBOX_THRESHOLD
    B = args.batch

    n_rot = 4
    host_batches = [synth_images(B, 1234 + rank * 1000 + i).pin_memory() for i in range(n_rot)]
    dev_batches = [h.to(dev) for h in host_batches]

    # The teacher forward hands out lazy results (no host read inside the forward), so the EMA launch is enqueued BEHIND the
    # forward's kernels and the step's single device->host read (the counts) comes after every launch of the step.
    teacher.roi_heads.box_predictor.defer_host_read = True

    def teacher_forward(images_dev):
        with torch.no_grad():
            _, proposals_rpn, proposals_roih = teacher(images_dev.to(memory_format=torch.channels_last) if args.channels_last else images_dev,
                                                       branch="unsup_data_weak")
        return proposals_rpn, proposals_roih

    def pseudo_label(images_dev):
        proposals_rpn, proposals_roih = teacher_forward(images_dev)
        pl, _ = engine.process_pseudo_label(proposals_roih, thr, "roih", "thresholding")
        return proposals_rpn, proposals_roih, pl

    def step_resident(i):
        proposals_rpn, proposals_roih = teacher_forward(dev_batches[i % n_rot])
        ema.step(cfg.SEMISUPNET.EMA_KEEP_RATE)
        pl, _ = engine.process_pseudo_label(proposals_roih, thr, "roih", "thresholding")     # the one host read of the step
        return proposals_rpn, proposals_roih, pl

    # pinned result buffers of the end-to-end arm (what a trainer reads back: the pseudo-labels of every image)
    T = cfg.TEST.DETECTIONS_PER_IMAGE
    res_host = {"boxes": torch.empty((B, T, 4), dtype=torch.float32).pin_memory(), "scores": torch.empty((B, T), dtype=torch.float32).pin_memory(),
                "classes": torch.empty((B, T), dtype=torch.int64).pin_memory()}
    d2h_bytes = sum(t.numel() * t.element_size() for t in res_host.values()) + 2 * B * 4 + 2 * B * 4  # + the two count reads
    h2d_bytes = host_batches[0].numel()

    def step_e2e(i):
        imgs = host_batches[i % n_rot].to(dev, non_blocking=True)
        rpn, dets = teacher_forward(imgs)
        batch = dets[0]._sfod_batch
        res_host["boxes"].copy_(batch.boxes, non_blocking=True)
        res_host["scores"].copy_(batch.scores, non_blocking=True)
        res_host["classes"].copy_(batch.classes, non_blocking=True)
        ema.step(cfg.SEMISUPNET.EMA_KEEP_RATE)
        pl, _ = engine.process_pseudo_label(dets, thr, "roih", "thresholding")               # reads the counts: the step's host sync
        torch.cuda.current_stream().synchronize()
        return rpn, dets, pl

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, with_timers=False):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = ops.launch_count()
        if with_timers:
            ops.timers.start()
        e0.record()
        for i in range(steps):
            out = fn(i)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        ktimes = ops.timers.stop() if with_timers else {}
        launches = ops.launch_count() - l0
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, launches, ktimes, out

    for i in range(max(args.warmup, 3)):
        step_resident(i)
    sampler = ClockSampler(local_rank)
    sampler.start()
    if args.profiler_range:
        torch.cuda.profiler.start()
    ms, launches, ktimes, out = timed(step_resident, args.steps, with_timers=True)
    if args.profiler_range:
        torch.cuda.profiler.stop()
    clocks = sampler.result()
    if args.dump_outputs and rank == 0:
        # before the other records below step the teacher further; the teacher runs in train() mode: the TRAIN proposal budget
        dump_outputs(args.dump_outputs, out, teacher, {"rpn": cfg.MODEL.RPN.POST_NMS_TOPK_TRAIN, "detections": T, "pseudo_labels": T})
    for i in range(3):
        step_e2e(i)
    ms_e2e, _, _, _ = timed(step_e2e, args.steps)

    value = world * B * args.steps / (ms / 1e3)
    e2e_value = world * B * args.steps / (ms_e2e / 1e3)
    peak, peak_src = peaks()

    # ---- second, labelled record: PyTorch's DEFAULT library math (TF32 convolutions); the hot-path kernels are fp32 either way
    library_default = None
    if args.extras and not args.tf32:
        try:
            set_math(True)
            torch.backends.cuda.matmul.allow_tf32 = False          # PyTorch default: cudnn.allow_tf32 True, matmul.allow_tf32 False
            for i in range(3):
                step_resident(i)
            ms_d, launches_d, kt_d, _ = timed(step_resident, args.steps, with_timers=True)
            for i in range(2):
                step_e2e(i)
            ms_de, _, _, _ = timed(step_e2e, args.steps)
            hot_d = sum(t for _, t in kt_d.values()) / args.steps
            library_default = {"label": "PyTorch-default library math (cudnn.allow_tf32=True, matmul.allow_tf32=False); not the headline",
                               "value": round(world * B * args.steps / (ms_d / 1e3), 2), "unit": UNIT, "ms_per_step": round(ms_d / args.steps, 3),
                               "e2e_value": round(world * B * args.steps / (ms_de / 1e3), 2), "hot_path_ms_per_step": round(hot_d, 3),
                               "hot_path_share_of_step": round(hot_d / (ms_d / args.steps), 4), "gpu_launches": int(launches_d)}
        except Exception as e:
            library_default = {"error": repr(e)[:300]}
        finally:
            set_math(args.tf32)

    # ---- CUDA-graph record: the sync-free teacher step (preprocess .. post-process + EMA) captured once, replayed per step
    graphed = None
    if args.extras:
        try:
            from sfod_b200.engine.graph import GraphedTeacherStep
            for label, tf32 in (("strict_fp32", False), ("pytorch_default_tf32", True)):
                if args.tf32 and not tf32:
                    continue
                set_math(tf32)
                if tf32:
                    torch.backends.cuda.matmul.allow_tf32 = bool(args.tf32)
                gs = GraphedTeacherStep(teacher, dev_batches[0].shape, lambda: ema.step(cfg.SEMISUPNET.EMA_KEEP_RATE), threshold=thr)

                def step_graph(i):
                    return gs.run(dev_batches[i % n_rot])
                for i in range(3):
                    step_graph(i)
                ms_g, launches_g, _, _ = timed(step_graph, args.steps)
                graphed = graphed or {}
                graphed[label] = {"ms_per_step": round(ms_g / args.steps, 3), "value": round(world * B * args.steps / (ms_g / 1e3), 2),
                                  "host_launch_calls_per_step": "1 graph replay (+ input copy, + one D2H read of the counts)"}
                del gs
        except Exception as e:
            graphed = {"error": repr(e)[:300]}
        finally:
            set_math(args.tf32)

    # ---- optional: the full mean-teacher step of configs[2] (SURVEY.md 8d "also report full SFOD step/s")
    sfod_step = None
    if args.sfod_step and args.workload == "vgg":
        try:
            from sfod_b200.utils.events import EventStorage
            stu = student
            if world > 1:
                stu = torch.nn.parallel.DistributedDataParallel(student, device_ids=[local_rank], broadcast_buffers=False,
                                                                find_unused_parameters=True)   # DC_img / DC_ins are idle in this branch
            opt = torch.optim.SGD(student.parameters(), lr=0.0025, momentum=0.9, weight_decay=1e-4)
            ema_ddp = engine.TeacherEMA(stu, teacher, world_size=world)   # strips the DDP 'module.' prefix like the reference

            def full_step(i):
                imgs = dev_batches[i % n_rot]
                _, _, pl = pseudo_label(imgs)
                batch = [{"image": imgs[j].float(), "instances": Instances_for(pl[j])} for j in range(B)]
                losses, _, _, _ = stu(batch, branch="supervised_target")
                loss = sum(losses.values())
                opt.zero_grad(set_to_none=True)
                loss.backward()
                opt.step()
                ema_ddp.step(cfg.SEMISUPNET.EMA_KEEP_RATE)
                return loss

            def Instances_for(p):
                from sfod_b200.structures import Instances
                t = Instances(p.image_size)
                t.gt_boxes, t.gt_classes = p.gt_boxes, p.gt_classes
                return t

            n_full = max(3, min(args.steps, 5))
            with EventStorage():
                for i in range(2):
                    full_step(i)
                ms_full, launches_full, _, last_loss = timed(full_step, n_full)
            grad_bytes = sum(p.numel() * 4 for p in student.parameters() if p.requires_grad)
            sfod_step = {"ms_per_step": round(ms_full / n_full, 3), "steps": n_full, "images_per_s": round(world * B * n_full / (ms_full / 1e3), 2),
                         "loss_last": round(float(last_loss.detach()), 5), "gpu_launches": int(launches_full),
                         "collective": None if world == 1 else f"DDP bucketed ncclAllReduce of {grad_bytes / 1e6:.0f} MB fp32 gradients per step",
                         "what": "teacher pseudo-labelling + student supervised_target fwd/bwd on the pseudo-labels"
                                 + (" + DDP all-reduce (NCCL)" if world > 1 else "") + " + SGD + EMA"}
        except Exception as e:  # never lose the headline line to the optional measurement
            sfod_step = {"error": repr(e)[:300]}

    # ---- configs[3]: AdaBN statistic recomputation step WITH its collective (SURVEY.md 8e collective 2): train-mode no_grad
    # backbone forward, every BN layer all-reduces (sum, sum^2, count) so that all ranks normalise with the statistics of the
    # concatenated batch; no host read anywhere (count stays on the device)
    adabn = None
    if args.extras:
        try:
            adabn = adabn_record(teacher, dev_batches, B, world, rank, dev, timed, args.steps, cfg)
        except Exception as e:
            adabn = {"error": repr(e)[:300]}

    # ---- per-kernel algorithmic bytes of one step (DESIGN.md "Algorithmic bytes"), fp32
    R = sum(len(p) for p in out[0])          # proposals actually pooled / post-processed in the last step
    bn_elems, bn_elems_pool, bn_elems_res, bn_elems_frozen = bn_activation_elements(args.workload, B)
    stride = 32 if args.workload == "vgg" else 16
    Cf = 512 if args.workload == "vgg" else 1024
    Hf, Wf = (IMAGE_HW[0] // stride, IMAGE_HW[1] // stride) if args.workload == "vgg" else (38, 75)
    A = 15 if args.workload == "vgg" else 12
    hwa = Hf * Wf * A
    alg = {
        "bn_finalize_apply": 8.0 * (bn_elems - bn_elems_pool - bn_elems_res),  # read x + write y (normalise + ReLU, in place)
        "bn_finalize_apply_pool": 5.0 * bn_elems_pool,                        # read x + write the 2x2-pooled y (1/4 of the elements)
        "bn_finalize_apply_res": 12.0 * bn_elems_res,                         # read x + read shortcut + write y
        "bn_frozen_apply": 8.0 * bn_elems_frozen + (4.0 * 3 * 256 * 150 * 300 * B if args.workload == "r101" else 0.0),   # + shortcut reads of res2's conv3
        "bn_partial_stats": 4.0 * bn_elems,                                   # read x
        "bn_train_fused": None, "bn_train_fused_res": None,                   # single-launch L2-resident BN: filled in below
        "ema_multi_tensor": 12.0 * ema.numel,                                 # read student, read teacher, write teacher
        "roi_align_fwd": 4.0 * (B * Cf * Hf * Wf + 5 * R + 49 * R * Cf),      # feature map + rois in, (R, C, 7, 7) out
        "rpn_select": B * 20.0 * hwa + 20.0 * R,                              # logits + deltas in, boxes + logit out
        "frcnn_postprocess": 4.0 * R * (4 + 4 * NUM_CLASSES + NUM_CLASSES + 1) + B * T * 28.0,
    }
    # Layers small enough for the single-launch BatchNorm leave the two-phase tags: split the element counts by what actually ran
    fused_calls = ktimes.get("bn_train_fused", (0, 0))[0] / args.steps, ktimes.get("bn_train_fused_res", (0, 0))[0] / args.steps
    if fused_calls[0] or fused_calls[1]:
        from sfod_b200 import ops as _ops
        per_layer = bn_layer_elements(args.workload, B)               # [(elements, has_residual, pooled)] of the train-mode BN layers
        small = [(e, r) for e, r, p in per_layer if not p and 4 * e <= _ops.BN_FUSED_MAX_BYTES]
        e_f, e_fr = sum(e for e, r in small if not r), sum(e for e, r in small if r)
        alg["bn_train_fused"], alg["bn_train_fused_res"] = 8.0 * e_f, 12.0 * e_fr      # x once + y (+ shortcut): the re-read comes from L2
        alg["bn_partial_stats"] -= 4.0 * (e_f + e_fr)
        alg["bn_finalize_apply"] -= 8.0 * e_f
        alg["bn_finalize_apply_res"] -= 12.0 * e_fr
    alg = {k: v for k, v in alg.items() if v}
    kernels = {}
    for tag, (calls, tot_ms) in sorted(ktimes.items()):
        per_step_ms = tot_ms / args.steps
        rec = {"calls_per_step": calls / args.steps, "ms_per_step": round(per_step_ms, 4)}
        if tag in alg and per_step_ms > 0 and alg[tag] > 0:
            gbs = alg[tag] / (per_step_ms * 1e-3) / 1e9
            rec.update({"alg_MB_per_step": round(alg[tag] / 1e6, 2), "GBps": round(gbs, 1), "frac_of_peak": round(gbs / peak, 4)})
        kernels[tag] = rec
    hot_ms = sum(v["ms_per_step"] for v in kernels.values())

    # DRAM traffic per launch of each kernel from the committed `ncu --set full` capture of this same command
    traffic_map = {"bn_finalize_apply": "bn_apply_nchw_kernel", "bn_finalize_apply_pool": "bn_apply_pool_nchw_kernel",
                   "bn_partial_stats": "bn_stats_nchw_kernel",
                   # VGG 18 x 37: slab-resident kernel; R101-C4 38 x 75 does not fit a slab: transpose + per-ROI L2 kernel
                   "roi_align_fwd": "roi_align_fwd_slab_kernel" if args.workload == "vgg" else "roi_align_fwd_sep_kernel (+ nchw_to_nhwc transpose, roi_sep_tables)",
                   "ema_multi_tensor": "ema_multi_tensor_kernel"}
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            ncu_traffic = json.load(f)
    except Exception:
        ncu_traffic = {}
    dominant = max((t for t in kernels if "GBps" in kernels[t]), key=lambda t: kernels[t]["ms_per_step"], default=None)
    roofline = None
    if dominant is not None:
        k = kernels[dominant]
        per_launch_ms = k["ms_per_step"] / k["calls_per_step"]
        tr = ncu_traffic.get(traffic_map.get(dominant, ""), {}) if args.workload == "vgg" else {}
        roofline = {"kernel": traffic_map.get(dominant, dominant), "call": dominant, "bound": "hbm", "achieved": k["GBps"], "peak": peak,
                    "unit": "GB/s", "frac": k["frac_of_peak"], "traffic": tr.get("dram_bytes_per_launch"),
                    "alg_bytes_per_launch": round(alg[dominant] / k["calls_per_step"]), "avg_launch_ms": round(per_launch_ms, 4),
                    "launches_per_step": k["calls_per_step"], "peak_source": peak_src,
                    "traffic_source": "COMMITTED constant, not measured in this run: profiles/ncu_traffic.json (ncu --set full of this "
                                      "command, dram__bytes_read.sum + dram__bytes_write.sum, mean per launch; raw CSVs under profiles/)"
                                      if tr else None,
                    "note": "the DOMINANT hot-path call by device time inside the timed region; achieved = algorithmic bytes per launch / "
                            "mean launch duration, CUDA events around the C-ABI call on the launching stream (each call = one "
                            "bn_finalize (C threads) + one apply kernel).  The kernels BASELINE.json's metric names are under `named`."}
        if args.extras and rank == 0:
            roofline["named"] = named_kernel_rooflines(dev, peak, ema._plan)
            in_step = {}
            for tag in ("roi_align_fwd", "ema_multi_tensor", "rpn_select", "frcnn_postprocess"):
                if tag in kernels:
                    in_step[tag] = {kk: kernels[tag][kk] for kk in ("ms_per_step", "GBps", "frac_of_peak") if kk in kernels[tag]}
            roofline["named"]["in_step_bench_shape"] = in_step
    for tag, kern in traffic_map.items():
        if tag in kernels and kern in ncu_traffic and args.workload == "vgg":
            kernels[tag]["ncu_dram_MB_per_launch"] = round(ncu_traffic[kern]["dram_bytes_per_launch"] / 1e6, 2)

    line = {"metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": round(ms / args.steps, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": workload_name(args.workload), "images_per_gpu": B, "images_per_step": B, "global_batch": B * world,
                       "image_hw": list(IMAGE_HW),
                       "num_classes": NUM_CLASSES, "parallelism": f"dp{world} (images sharded per GPU, replicated teacher, no data-path collective "
                                                                  "in the headline step; the AdaBN step of configs[3] with its statistic all-reduce and the "
                                                                  "DDP student step are the `adabn` / `sfod_step` records)",
                       "library_math": "cuDNN/cuBLAS " + ("TF32 allowed" if args.tf32 else "strict fp32 (TF32 off)"),
                       "backbone_layout": "NHWC" if args.channels_last else "NCHW",
                       "l2": f"inputs larger than L2: {n_rot} rotating input batches, per-step activation footprint "
                             f"{4.0 * bn_elems / 1e9:.1f} GB per BN pass >> 126 MB L2"},
            "clocks": clocks,
            "e2e": {"value": round(e2e_value, 2), "unit": UNIT, "h2d_bytes_per_step": int(h2d_bytes), "d2h_bytes_per_step": int(d2h_bytes),
                    "ms_per_step": round(ms_e2e / args.steps, 3)},
            "gpu_launches": int(launches),
            "roofline": roofline,
            "kernels": kernels,
            "hot_path": {"ms_per_step": round(hot_ms, 3), "share_of_step": round(hot_ms / (ms / args.steps), 4),
                         "note": "sum of the event-timed C-ABI calls; the rest of the step is cuDNN conv / cuBLAS FC / torch glue"},
            "library_default_math": library_default,
            "cuda_graph": graphed,
            "adabn": adabn,
            "sfod_step": sfod_step,
            "proposals_last_step": [len(p) for p in out[0]],
            "detections_last_step": [len(p) for p in out[1]],
            "pseudo_labels_last_step": [len(p) for p in out[2]]}
    if rank == 0 and world == 1 and args.extras:
        line["exp_flip_rate"] = flip_rate_sample(dev)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            _, info, _, _, _ = cpu_reference_run(2, 1, 30.0, images_per_step=B, workload=args.workload)   # a bounded sample of the same batch
            line["cpu_baseline"] = info
        except Exception as e:  # the baseline is a report, never a reason to lose the GPU number
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {e!r}"}
    if rank == 0:
        emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


def bn_activation_elements(workload: str, B: int):
    """Activation elements entering the norm layers per step: (train-mode BN total, of which fused with the 2x2 max-pool, of which
    fused with the residual add, frozen-BN total)."""
    if workload == "vgg":   # SURVEY.md App. C: 194 342 400 per image
        hw = [(600, 1200)] * 2 + [(300, 600)] * 2 + [(150, 300)] * 3 + [(75, 150)] * 3 + [(37, 75)] * 3
        ch = [64, 64, 128, 128, 256, 256, 256, 512, 512, 512, 512, 512, 512]
        per_layer = [c * h * w for c, (h, w) in zip(ch, hw)]
        pooled = {1, 3, 6, 9, 12}
        return sum(per_layer) * B, sum(e for i, e in enumerate(per_layer) if i in pooled) * B, 0, 0
    # R101-C4 at 600x1200: stem 64 @ 300x600 (frozen); res2 @ 150x300 (frozen); res3 @ 75x150; res4 @ 38x75
    s2, s3, s4 = 150 * 300, 75 * 150, 38 * 75
    frozen = 64 * 300 * 600 + 3 * (64 + 64 + 256) * s2 + 256 * s2
    res3 = (128 + 128 + 512 + 512) * s3 + 3 * (128 + 128 + 512) * s3                    # STRIDE_IN_1X1: every layer of res3 runs at 75x150
    res4 = (256 + 256 + 1024 + 1024) * s4 + 22 * (256 + 256 + 1024) * s4
    resid = 4 * 512 * s3 + 23 * 1024 * s4                                               # conv3 norm layers (residual + ReLU fusion)
    return (res3 + res4) * B, 0, resid * B, frozen * B


def bn_layer_elements(workload: str, B: int):
    """[(activation elements, residual fusion, max-pool fusion)] of every train-mode BN layer of the backbone, per step."""
    if workload == "vgg":
        hw = [(600, 1200)] * 2 + [(300, 600)] * 2 + [(150, 300)] * 3 + [(75, 150)] * 3 + [(37, 75)] * 3
        ch = [64, 64, 128, 128, 256, 256, 256, 512, 512, 512, 512, 512, 512]
        return [(c * h * w * B, False, i in {1, 3, 6, 9, 12}) for i, (c, (h, w)) in enumerate(zip(ch, hw))]
    s3, s4 = 75 * 150, 38 * 75
    out = []
    for nblk, bc, oc, s in ((4, 128, 512, s3), (23, 256, 1024, s4)):
        for i in range(nblk):
            if i == 0:
                out.append((oc * s * B, False, False))                 # projection shortcut
            out += [(bc * s * B, False, False), (bc * s * B, False, False), (oc * s * B, True, False)]
    return out


def adabn_record(teacher, dev_batches, B, world, rank, dev, timed, steps, cfg):
    """One AdaBN iteration (reference daod/engine/trainers/base.py:270-337: train()-mode forward under no_grad, only the BN side
    effects matter) on the teacher's backbone, with every BN layer's statistics all-reduced over the ranks."""
    import copy
    import torch
    import torch.distributed as dist
    from sfod_b200.modeling.batch_norm import SfodBatchNorm2d
    bb = copy.deepcopy(teacher.backbone)
    from sfod_b200.engine import adabn as adabn_mod
    adabn_mod.recursive_traversal(bb); adabn_mod.recursive_traversal(bb)
    layers = [m for m in bb.modules() if isinstance(m, SfodBatchNorm2d)]
    bb.train()
    x_norm = [teacher.preprocess_batch(b).tensor for b in dev_batches]

    def step(i):
        with torch.no_grad():
            return bb(x_norm[i % len(x_norm)])

    def run(group):
        for m in layers:
            m.process_group = group
        for i in range(3):
            step(i)
        n_ = max(3, min(steps, 10))
        ms_, launches_, _, _ = timed(step, n_)
        return ms_, launches_, n_

    # Product path at N > 1: the statistic all-reduce fused into the finalize kernel over NVLink peer memory
    # (sfod_bn_exchange_finalize_apply); baseline beside it: one ncclAllReduce launch per BN layer.
    peer, peer_err, nccl_ms = None, None, None
    if world > 1:
        ms_b, _, n_b = run(True)
        nccl_ms = ms_b / n_b
        try:
            from sfod_b200.engine.p2p import PeerStatExchange
            peer = PeerStatExchange.from_process_group(device=dev)
        except Exception as e:   # no peer access / IPC on this box: the NCCL path is reported, and said so
            peer_err = f"{type(e).__name__}: {e}"[:200]
        ok = torch.tensor([0 if peer is None else 1], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) == 0 and peer is not None:
            peer.close(); peer = None; peer_err = peer_err or "a peer rank could not map the inboxes"
    group = peer if peer is not None else (True if world > 1 else None)
    variants = None
    if peer is not None:   # delivery by the statistics kernel's last CTA (default) vs by the finalize kernel
        from sfod_b200 import ops as _ops
        default_tail = _ops.BN_P2P_TAIL_PUSH
        _ops.BN_P2P_TAIL_PUSH = 1 - default_tail
        ms_o, _, n_o = run(group)
        _ops.BN_P2P_TAIL_PUSH = default_tail
        variants = {("payload_delivered_by_statistics_kernel_tail" if not default_tail else "payload_delivered_by_finalize_kernel"): round(ms_o / n_o, 3)}
    ms, launches, n = run(group)
    if variants is not None:
        variants[("payload_delivered_by_statistics_kernel_tail" if default_tail else "payload_delivered_by_finalize_kernel") + " (default, = ms_per_step)"] = round(ms / n, 3)
    payload = sum(2 * m.num_features + 1 for m in layers) * 8
    if world == 1:
        coll = None
    elif peer is not None:
        coll = (f"one-shot all-reduce over NVLink peer memory fused into the finalize kernel of each of the {len(layers)} BN layers "
                f"(P2P stores of self-validating 16-byte (value, tag) elements, fp64 (sum, sum^2, count) payloads, {2 * payload} B per rank and peer and step, no fence, no flag, no collective launch, no host read)")
    else:
        coll = (f"{len(layers)} ncclAllReduce per step (one per BN layer, fp64 (sum, sum^2, count) payloads, {payload} B per rank and step in total), "
                f"enqueued without any host read; peer-memory path unavailable: {peer_err}")
    rec = {"metric": "adabn_images_per_s", "value": round(world * B * n / (ms / 1e3), 2), "unit": UNIT, "ms_per_step": round(ms / n, 3), "steps": n,
           "bn_layers": len(layers), "gpu_launches": int(launches), "collective": coll,
           "what": "configs[3] AdaBN step: backbone forward in train() mode under no_grad, running statistics of the concatenated batch"}
    if nccl_ms is not None:
        rec["nccl_allreduce_baseline_ms_per_step"] = round(nccl_ms, 3)
    if variants is not None:
        rec["peer_memory_variants_ms_per_step"] = variants
    if world > 1:
        # The step above is dominated by the convolutions and by the skew between the ranks; the cost of the collective itself
        # is isolated here: one 512-channel BN layer on a tiny activation, 200 forwards back to back, microseconds per layer.
        from sfod_b200 import ops as _ops

        def layer_us(grp):
            bn_ = SfodBatchNorm2d(512, process_group=grp).to(dev).train()
            xs_ = torch.randn(2, 512, 8, 8, device=dev)
            saved = _ops.BN_FUSED_MAX_BYTES
            _ops.BN_FUSED_MAX_BYTES = 0      # two-phase path for the no-collective line as well
            try:
                with torch.no_grad():
                    for _ in range(20):
                        bn_(xs_)
                    dist.barrier(); torch.cuda.synchronize()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    for _ in range(200):
                        bn_(xs_)
                    e1.record(); torch.cuda.synchronize()
            finally:
                _ops.BN_FUSED_MAX_BYTES = saved
            t_ = torch.tensor([e0.elapsed_time(e1) * 1e3 / 200], dtype=torch.float64, device=dev)
            dist.all_reduce(t_, op=dist.ReduceOp.MAX)
            return round(float(t_.item()), 2)
        lat = {"no_collective": layer_us(None), "nccl_allreduce": layer_us(True)}
        if peer is not None:
            lat["peer_memory_fused"] = layer_us(peer)
        lat["what"] = "us per 512-channel BN layer forward (statistics + [collective] + finalize + apply) on a 2x512x8x8 activation, max over ranks"
        rec["collective_latency_us_per_layer"] = lat
    if world > 1:   # self-check of the multi-GPU statistics against a single-device computation on the concatenated batch
        g = torch.Generator().manual_seed(77)
        xs = [torch.randn(2, 8, 24, 40, generator=g) * (r + 1) + r for r in range(world)]
        bn = SfodBatchNorm2d(8, process_group=group).to(dev).train()
        with torch.no_grad():
            bn(xs[rank].to(dev))
        ref = torch.nn.BatchNorm2d(8).train()
        with torch.no_grad():
            ref(torch.cat(xs))
        err = max(((bn.running_mean.cpu() - ref.running_mean).abs() / ref.running_mean.abs().clamp_min(1e-6)).max().item(),
                  ((bn.running_var.cpu() - ref.running_var).abs() / ref.running_var.abs()).max().item())
        t = torch.tensor([err], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        rec["selfcheck_vs_cpu_batchnorm_on_concatenated_batch"] = {"max_rel_err": float(t.item()), "tolerance": 1e-5, "ok": bool(t.item() <= 1e-5)}
        if peer is not None:
            ex, to = peer.status()
            tt = torch.tensor([to], dtype=torch.int64, device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            rec["peer_exchanges"] = {"completed_on_rank0": ex, "timeouts_max_over_ranks": int(tt.item())}
            dist.barrier()
            peer.close()
    return rec


_REAL_STDOUT = None


def emit(line: dict) -> None:
    """The ONE JSON line goes to the process's real stdout; everything else any library prints (e.g. NCCL's version
    banner, which goes to stdout at C level) has been redirected to stderr by main()."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT, NUM_CLASSES
    args = parse_args()
    if args.num_classes < 1:
        raise SystemExit("--num-classes must be >= 1")
    NUM_CLASSES = args.num_classes
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)          # fd 1 -> stderr for the rest of the run
    if args.impl == "reference":
        return run_reference(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
