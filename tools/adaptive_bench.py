"""Does adaptive sampling pay?  Uniform spp against the ptc_adaptive_* passes on the same scene, both held to a high-spp fixed reference.

For each workload: a fixed reference render (--ref-spp, another seed than the renders it judges); uniform renders of 16 .. 256 spp
and adaptive renders at tau = 0.2, 0.1, 0.05 (min 16, step 16, max --max-spp), each timed with a synchronised host clock around the
whole render as a user runs it (clear, passes, read back of the sums), best of --repeat; rel_mse of every image against the reference
(tests/parity.py: mean of (x - r)^2 / (r^2 + 1e-2)).  From these it derives the time each mode needs to reach the rel_mse of uniform
64 spp (adaptive: log-log interpolation between the two tau that bracket it, null when none do), and it keeps the per-pass wall times
of the tau = 0.1 render (every pass ends in one host synchronisation).  Prints the card's name and power limit and one JSON object per
workload; writes them to --out/adaptive_<workload>.json.

    python tools/adaptive_bench.py [--workloads cornell-glass dragon] [--out DIR]
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from parity import rel_mse  # noqa: E402

from pathed_b200 import load_scene  # noqa: E402

WORKLOADS = {
    "cornell-glass": dict(scene="scenes/cornell-glass.json", width=512, height=512, last_bounce=10),
    "dragon": dict(scene="scenes/dragon.json", width=1024, height=1024, last_bounce=10),
}
UNIFORM_SPP = [16, 32, 64, 128, 256]
THRESHOLDS = [0.2, 0.1, 0.05]
MIN_SPP, STEP_SPP = 16, 16
SEED, REF_SEED = 1, 2


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        limit = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                               text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = "unknown"
    return name, limit


def uniform(ctx, spp, last):
    t0 = time.perf_counter()
    ctx.framebuffer_clear()
    ctx.framebuffer_render(SEED, 0, spp, 0, last)
    sums = ctx.framebuffer_gather([], divisor=1)  # returns when the sums are on the host
    return time.perf_counter() - t0, sums / np.float32(spp)


def adaptive(ctx, tau, max_spp, last):
    passes = []
    t0 = time.perf_counter()
    ctx.adaptive_begin(tau, MIN_SPP, STEP_SPP, max_spp)
    while True:
        p0 = time.perf_counter()
        active, n = ctx.adaptive_pass(SEED, 0, last)
        passes.append({"spp": n, "active_after": active, "s": time.perf_counter() - p0})
        if active == 0:
            break
    sums = ctx.framebuffer_gather([], divisor=1)
    counts, _ = ctx.adaptive_state()
    seconds = time.perf_counter() - t0
    return seconds, sums / counts[..., None].astype(np.float32), counts, passes


def time_to_target(points, target):
    """points: (seconds, rel_mse) of the adaptive renders; log-log interpolation between the two that bracket target"""
    points = sorted(points, key=lambda p: p[1])
    for (t_lo, e_lo), (t_hi, e_hi) in zip(points, points[1:]):
        if e_lo <= target <= e_hi and e_lo > 0 and e_hi > e_lo:
            w = (math.log(target) - math.log(e_lo)) / (math.log(e_hi) - math.log(e_lo))
            return math.exp(math.log(t_lo) + w * (math.log(t_hi) - math.log(t_lo)))
    return None


def run(name, ref_spp, max_spp, repeat):
    w = WORKLOADS[name]
    ctx = load_scene(w["scene"], w["width"], w["height"])
    last = w["last_bounce"]
    pixels = w["width"] * w["height"]
    ctx.framebuffer_clear()
    ctx.framebuffer_render(REF_SEED, 0, ref_spp, 0, last)
    reference = ctx.framebuffer_gather([], divisor=ref_spp)
    uniform(ctx, 16, last)                 # warm-up: module load, path state of the largest wave
    adaptive(ctx, THRESHOLDS[0], max_spp, last)
    out = {"workload": "%s %dx%d PathTracer lastBounce %d" % (w["scene"], w["width"], w["height"], last), "reference_spp": ref_spp,
           "seed": SEED, "reference_seed": REF_SEED, "uniform": [], "adaptive": []}
    for spp in UNIFORM_SPP:
        runs = [uniform(ctx, spp, last) for _ in range(repeat)]
        seconds = min(r[0] for r in runs)
        out["uniform"].append({"spp": spp, "s": seconds, "all_s": [r[0] for r in runs], "rel_mse": rel_mse(runs[0][1], reference),
                               "msamples_per_s": pixels * spp / seconds * 1e-6})
    for tau in THRESHOLDS:
        runs = [adaptive(ctx, tau, max_spp, last) for _ in range(repeat)]
        seconds = min(r[0] for r in runs)
        _, image, counts, passes = runs[0]
        samples = int(counts.sum())
        row = {"tau": tau, "min_spp": MIN_SPP, "step_spp": STEP_SPP, "max_spp": max_spp, "s": seconds, "all_s": [r[0] for r in runs],
               "passes": len(passes), "samples": samples, "mean_spp": samples / pixels, "pixels_at_max": int((counts == max_spp).sum()),
               "rel_mse": rel_mse(image, reference), "msamples_per_s": samples / seconds * 1e-6}
        if tau == 0.1:
            row["pass_wall_s"] = passes
        out["adaptive"].append(row)
    target = next(u for u in out["uniform"] if u["spp"] == 64)
    adaptive_s = time_to_target([(a["s"], a["rel_mse"]) for a in out["adaptive"]], target["rel_mse"])
    out["to_uniform64_rel_mse"] = {"rel_mse": target["rel_mse"], "uniform_s": target["s"], "adaptive_s": adaptive_s,
                                   "adaptive_speedup": None if adaptive_s is None else target["s"] / adaptive_s}
    ctx.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", nargs="+", default=sorted(WORKLOADS), choices=sorted(WORKLOADS))
    ap.add_argument("--ref-spp", type=int, default=4096)
    ap.add_argument("--max-spp", type=int, default=1024)
    ap.add_argument("--repeat", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    name, limit = card()
    print("card: %s, power limit %s" % (name, limit), flush=True)
    for workload in args.workloads:
        result = run(workload, args.ref_spp, args.max_spp, args.repeat)
        result["card"], result["power_limit"] = name, limit
        print(json.dumps(result), flush=True)
        if args.out:
            os.makedirs(args.out, exist_ok=True)
            with open(os.path.join(args.out, "adaptive_%s.json" % workload), "w") as f:
                json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
