"""Times the box head's fully connected layers at the bench shapes (M = 16000 ROIs of 8 images x 2000 proposals): the library's
3xTF32 tensor-core kernel (ops.linear_3xtf32, ReLU fused) against F.linear + ReLU in strict fp32 and in TF32.

CUDA events around each call, with a 512 MB buffer overwritten before every timed call so that no operand is served from L2.
The rate is 2*M*N*K / time; the 3xTF32 kernel issues three TF32 MMAs per product, so its bound is a third of the dense TF32
rate (data sheet 1125 TFLOP/s for a B200 at 1000 W).  Prints one JSON line per (shape, path), with the GPU name, power limit and
SM clock read in the same run.

    python tools/fc_bench.py [--reps 20] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = [("vgg_fc1", 16000, 1024, 25088), ("vgg_fc2", 16000, 1024, 1024), ("r101_fc1", 16000, 2048, 50176),
          ("r101_fc2", 16000, 2048, 2048)]
TF32_DENSE_TFLOPS = 1125.0


def gpu_info() -> dict:
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()[0]
        return dict(zip(q.split(","), [v.strip() for v in out.split(",")]))
    except Exception as e:   # the timing does not depend on it
        return {"error": repr(e)[:200]}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import torch.nn.functional as F

    import sfod_b200  # noqa: F401
    from sfod_b200 import ops
    if not torch.cuda.is_available():
        raise RuntimeError("fc_bench measures the CUDA path: no CUDA device is visible")
    dev = torch.device("cuda:0")
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    records = []
    for name, M, N, K in SHAPES:
        g = torch.Generator(device=dev).manual_seed(0)
        x = torch.randn(M, K, device=dev, generator=g)
        w = torch.randn(N, K, device=dev, generator=g) * K ** -0.5
        b = torch.randn(N, device=dev, generator=g) * 0.1
        paths = {"native_3xtf32": (False, lambda: ops.linear_3xtf32(x, w, b, relu=True)),
                 "F.linear_fp32": (False, lambda: torch.relu(F.linear(x, w, b))),
                 "F.linear_tf32": (True, lambda: torch.relu(F.linear(x, w, b)))}
        for path, (tf32, fn) in paths.items():
            torch.backends.cuda.matmul.allow_tf32 = tf32
            for _ in range(2):
                fn()
            ms = []
            for _ in range(args.reps):
                flush.fill_(1)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                fn()
                e1.record()
                e1.synchronize()
                ms.append(e0.elapsed_time(e1))
            ms.sort()
            med = ms[len(ms) // 2]
            tflops = 2 * M * N * K / (med * 1e-3) / 1e12
            rec = {"shape": name, "M": M, "N": N, "K": K, "path": path, "ms_median": round(med, 4), "ms_min": round(ms[0], 4),
                   "ms_max": round(ms[-1], 4), "tflops": round(tflops, 1)}
            if path == "native_3xtf32":
                rec["share_of_tf32_dense_over_3"] = round(tflops / (TF32_DENSE_TFLOPS / 3), 3)
            records.append(rec)
            print(json.dumps(rec), flush=True)
        del x, w, b
        torch.cuda.empty_cache()
    torch.backends.cuda.matmul.allow_tf32 = False
    info = {"gpu": gpu_info(), "torch": torch.__version__, "reps": args.reps, "l2_flush_bytes": flush.numel()}
    print(json.dumps(info))
    if args.out:
        with open(args.out, "w") as f:
            json.dump({"info": info, "records": records}, f, indent=1)


if __name__ == "__main__":
    main()
