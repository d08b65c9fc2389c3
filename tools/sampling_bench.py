"""Cost of sampled decoding on one GPU, written to one JSON file together with the GPU's name and power limit.

    python tools/sampling_bench.py --out /tmp/sampling_bench.json

1. Per-launch time of dots_argmax_advance against dots_sample_advance for B in {1, 64, 256}, V = 151 936, random bf16 logits
   (N(0, 3)), every row of a launch with the same parameter mix; CUDA events around `--launches` back-to-back launches after
   warm-up.  The mixes isolate the passes of the sampling kernel: greedy = the argmax pass; T only = max + Gumbel pass; top-k =
   max + two radix passes + Gumbel; top-p = max + two radix passes + Gumbel; top-k + top-p = max + up to three radix passes +
   Gumbel.
2. Pages/s of the benchmark workload (bench.py: 64 synthetic 1024 x 1024 pages, 512 new tokens, full config, `random` weights,
   no stop ids): greedy against T = 0.1 p = 1.0 and T = 0.1 p = 0.9, alternated in one process.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

MIXES = {"greedy": (0.0, 1.0, 0), "T0.1": (0.1, 1.0, 0), "T0.1_p0.9": (0.1, 0.9, 0), "T1_k50": (1.0, 1.0, 50),
         "T0.7_k20_p0.8": (0.7, 0.8, 20)}


def gpu_info():
    import torch
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["nvidia_smi"] = q
    except Exception as e:      # noqa: BLE001
        info["nvidia_smi"] = f"unavailable: {e}"
    return info


def kernel_times(launches: int, warmup: int):
    import torch
    from dots_ocr_b200 import ops
    from dots_ocr_b200.sampling import SamplingParams, host_arrays
    V = 151936
    out = []
    for B in (1, 64, 256):
        g = torch.Generator(device="cuda").manual_seed(B)
        logits = (torch.randn(B, V, device="cuda", generator=g) * 3).to(torch.bfloat16)
        nxt = torch.zeros(B, dtype=torch.int64, device="cuda")

        def timed(fn):
            for _ in range(warmup):
                fn()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(launches):
                fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) * 1e3 / launches
        row = {"B": B, "argmax_us": timed(lambda: ops.argmax_advance(logits, nxt))}
        for name, (T, p, k) in MIXES.items():
            arrs = [a.cuda() for a in host_arrays([SamplingParams(T, p, k, 1000 + i) for i in range(B)])]
            step = torch.zeros(B, dtype=torch.int32, device="cuda")
            row[f"sample_{name}_us"] = timed(lambda: ops.sample_advance(logits, nxt, *arrs, step=step))
        out.append(row)
        print(json.dumps(row), flush=True)
    return out


def pages_per_second(reps: int):
    import torch
    import bench
    from dots_ocr_b200 import config, weights
    from dots_ocr_b200.engine import Engine
    from dots_ocr_b200.sampling import SamplingParams
    cfg = config.full()
    dev = torch.device("cuda", 0)
    eng = Engine(cfg, weights.make_synthetic_checkpoint(cfg, 0, "random", device=dev), dev)
    B, N = 64, 512
    pv, grid, ids = bench.make_workload(cfg, B, 0, dev)
    ids = ids.to(dev)
    arms = {"greedy": None, "T0.1_p1.0": SamplingParams(0.1, 1.0, 0, 1), "T0.1_p0.9": SamplingParams(0.1, 0.9, 0, 1)}
    for s in arms.values():                                          # warm-up: every arm compiles its graph once
        eng.generate(ids, pixel_values=pv, image_grid_thw=grid, max_new_tokens=N, sampling=s)
    times = {k: [] for k in arms}
    for _ in range(reps):
        for name, s in arms.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            eng.generate(ids, pixel_values=pv, image_grid_thw=grid, max_new_tokens=N, sampling=s)
            torch.cuda.synchronize()
            times[name].append(time.perf_counter() - t0)
    res = {}
    for name, ts in times.items():
        med = sorted(ts)[len(ts) // 2]
        res[name] = {"seconds": ts, "median_s": med, "pages_per_s": B / med}
    base = res["greedy"]["median_s"]
    for name in res:
        res[name]["vs_greedy"] = res[name]["median_s"] / base
    print(json.dumps(res), flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--no-e2e", dest="no_e2e", action="store_true")
    a = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "sampling_bench needs a GPU"
    res = {"gpu": gpu_info(), "kernel_us": kernel_times(a.launches, a.warmup)}
    if not a.no_e2e:
        res["pages"] = pages_per_second(a.reps)
    res["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(f"wrote {a.out}")


if __name__ == "__main__":
    main()
