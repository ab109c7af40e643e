"""Poisson-disk down-sampling timings: CUDA events around the public API with CUDA tensors in (one warm-up call per
workload, then the median of `reps` calls), the radius trials and MIS rounds of each call, and the C oracle's
single-thread time on the same input for context.

    python tools/poisson_time.py [reps] [--json PATH]     (--json: the rows as JSON as well)
"""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import pcu_b200 as pcu
from pcu_b200 import _pcu_internal
from oracle import poisson_oracle

args = sys.argv[1:]
json_path = None
if "--json" in args:
    json_path = args[args.index("--json") + 1]
    del args[args.index("--json"):args.index("--json") + 2]
reps = int(args[0]) if args else 5
n = 10 ** 6
rng = np.random.default_rng(0)
cube = rng.random((n, 3)).astype(np.float32)
sph = rng.normal(size=(n, 3))
sph = (sph / np.linalg.norm(sph, axis=1, keepdims=True)).astype(np.float32)
ball = lambda per_ball: float((per_ball / (n * 4 / 3 * np.pi)) ** (1 / 3))   # radius holding ~per_ball uniform points

workloads = [
    ("uniform 1e6, ~1e5 samples", cube, dict(radius=0.0165)),
    ("uniform 1e6, ~1e3 points per ball (~1e3 samples)", cube, dict(radius=ball(1000))),
    ("sphere 1e6, r = 0.01", sph, dict(radius=0.01)),
    ("uniform 1e6, target 1e4", cube, dict(radius=0.0, target_num_samples=10 ** 4)),
    ("sphere 1e6, target 1e4", sph, dict(radius=0.0, target_num_samples=10 ** 4)),
]

card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                      capture_output=True, text=True).stdout.strip().splitlines()
print("card:", card[0] if card else "unknown")
results = {"card": card[0] if card else None, "reps": reps, "workloads": []}
for name, pts, kw in workloads:
    t = torch.from_numpy(pts).cuda()
    stream = torch.cuda.current_stream().cuda_stream
    idx = pcu.downsample_point_cloud_poisson_disk(t, random_seed=1, **kw)      # warm-up (and the workspace)
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        idx = pcu.downsample_point_cloud_poisson_disk(t, random_seed=1, **kw)
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
    trials, rounds = _pcu_internal._poisson_stats(0, stream)
    t0 = time.perf_counter()
    ref = poisson_oracle.downsample_point_cloud_poisson_disk(pts, random_seed=1, **kw)
    oracle_s = time.perf_counter() - t0
    same = bool(np.array_equal(idx.cpu().numpy(), ref))
    row = {"workload": name, "samples": int(idx.shape[0]), "ms_median": float(np.median(times)), "ms_min": float(np.min(times)),
           "ms_max": float(np.max(times)), "trials": int(trials), "mis_rounds": int(rounds), "oracle_single_thread_s": oracle_s,
           "equal_to_oracle": same, **{k: float(v) for k, v in kw.items()}}
    results["workloads"].append(row)
    print("%-52s samples %7d  %8.3f ms (min %.3f, max %.3f)  trials %2d  rounds %4d  oracle %.2f s  equal %s"
          % (name, row["samples"], row["ms_median"], row["ms_min"], row["ms_max"], trials, rounds, oracle_s, same), flush=True)
if json_path:
    with open(json_path, "w") as f:
        json.dump(results, f, indent=1)
