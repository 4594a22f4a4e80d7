"""Does denoising pay?  Uniform renders at 4 .. 64 spp, each noisy and denoised (ptc_render_aovs + ptc_denoise), held to a high-spp render.

For each workload: a reference render (--ref-spp, another seed than the renders it judges); uniform renders with the option
"framebuffer_moments" on, timed with a synchronised host clock around clear, render and the read back of sums and second moments,
best of --repeat; the guide pass (ptc_render_aovs over min(spp, 16) samples) and ptc_denoise (default parameters; host copies
included) timed the same way.  rel_mse of every image against the reference (tests/parity.py: mean of (x - r)^2 / (r^2 + 1e-2)),
and for each denoised image the spp at which uniform sampling reaches the same rel_mse (log-log interpolation over the uniform
renders, extended by the 1/spp law beyond 64; null when the denoised error is above the 4-spp error).  A second pass runs ptc_denoise
under torch.profiler with CUDA activities and sums the device time of the filter's kernels (denoisePrepareKernel,
denoiseAtrousKernel) and of aovKernel.  Prints the card's name and power limit and one JSON object per workload; writes them to
--out/r04_denoise_<workload>.json.

    python tools/denoise_bench.py [--workloads cornell-glass dragon] [--out DIR]
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
from pathed_b200._binding import GATHER_MOMENTS  # noqa: E402

WORKLOADS = {
    "cornell-glass": dict(scene="scenes/cornell-glass.json", width=512, height=512, last_bounce=10),
    "dragon": dict(scene="scenes/dragon.json", width=1024, height=1024, last_bounce=10),
}
SPP = [4, 8, 16, 32, 64]
GUIDE_SPP = 16  # what the `pathed` job uses: min(spp, 16)
SEED, REF_SEED = 1, 2
FILTER_KERNELS = ("denoisePrepareKernel", "denoiseAtrousKernel")


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        limit = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                               text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = "unknown"
    return name, limit


def render(ctx, spp, last):
    t0 = time.perf_counter()
    ctx.framebuffer_clear()
    ctx.framebuffer_render(SEED, 0, spp, 0, last)
    sums = ctx.framebuffer_gather([], divisor=1)  # returns when the sums are on the host
    moments = ctx.framebuffer_gather([], 1, GATHER_MOMENTS)
    return time.perf_counter() - t0, sums, moments


def timed(fn, repeat):
    runs = []
    for _ in range(repeat):
        t0 = time.perf_counter()
        out = fn()
        runs.append(time.perf_counter() - t0)
    return min(runs), runs, out


def spp_for(uniform, target):
    """the spp at which uniform sampling reaches rel_mse `target` (log-log between the two renders that bracket it; 1/spp beyond)"""
    pts = sorted((u["spp"], u["rel_mse"]) for u in uniform)
    if target > pts[0][1]:
        return None
    for (s0, e0), (s1, e1) in zip(pts, pts[1:]):
        if e1 <= target <= e0 and e0 > e1 > 0:
            w = (math.log(e0) - math.log(target)) / (math.log(e0) - math.log(e1))
            return math.exp(math.log(s0) + w * (math.log(s1) - math.log(s0)))
    s, e = pts[-1]
    return s * e / target


def kernel_ms(ctx, sums, moments, spp, aovs, aov_spp, out_dir, name):
    """device time of the filter's kernels and of aovKernel in one profiled ptc_denoise / ptc_render_aovs (a run of its own)"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        ctx.denoise(sums, moments, spp, aovs, aov_spp)
        ctx.render_aovs(SEED, 0, aov_spp)
        torch.cuda.synchronize()
    per = {}
    for e in prof.key_averages():
        for k in FILTER_KERNELS + ("aovKernel",):
            if k in e.key:
                per[k] = per.get(k, 0.0) + e.device_time_total / 1000.0
    if out_dir:
        prof.export_chrome_trace(os.path.join(out_dir, "r04_denoise_%s_trace.json" % name))
    return per


def run(name, ref_spp, repeat, out_dir):
    w = WORKLOADS[name]
    ctx = load_scene(w["scene"], w["width"], w["height"])
    ctx.set_option("framebuffer_moments", 1)
    last = w["last_bounce"]
    pixels = w["width"] * w["height"]
    reference = ctx.render(REF_SEED, 0, ref_spp, 0, last) / np.float32(ref_spp)
    render(ctx, SPP[-1], last)  # warm-up: module load, path state of the largest wave
    out = {"workload": "%s %dx%d PathTracer lastBounce %d" % (w["scene"], w["width"], w["height"], last), "reference_spp": ref_spp,
           "seed": SEED, "reference_seed": REF_SEED, "guide_spp": "min(spp, %d)" % GUIDE_SPP, "filter": "defaults (PTC_DENOISE_DEFAULTS)",
           "rows": []}
    inputs = {}
    for spp in SPP:
        seconds, runs, (_, sums, moments) = timed(lambda: render(ctx, spp, last), repeat)
        aov_spp = min(spp, GUIDE_SPP)
        guide_s, guide_runs, aovs = timed(lambda: ctx.render_aovs(SEED, 0, aov_spp), repeat)
        denoise_s, denoise_runs, image = timed(lambda: ctx.denoise(sums, moments, spp, aovs, aov_spp), repeat)
        inputs[spp] = (sums, moments, aovs, aov_spp)
        out["rows"].append({"spp": spp, "render_s": seconds, "render_all_s": runs, "guide_s": guide_s, "guide_all_s": guide_runs,
                            "denoise_s": denoise_s, "denoise_all_s": denoise_runs, "msamples_per_s": pixels * spp / seconds * 1e-6,
                            "rel_mse": rel_mse(sums / np.float32(spp), reference), "denoised_rel_mse": rel_mse(image, reference)})
    uniform = [{"spp": r["spp"], "rel_mse": r["rel_mse"]} for r in out["rows"]]
    for r in out["rows"]:
        r["uniform_spp_for_denoised_rel_mse"] = spp_for(uniform, r["denoised_rel_mse"])
    sums, moments, aovs, aov_spp = inputs[16]
    out["kernel_ms_16spp"] = kernel_ms(ctx, sums, moments, 16, aovs, aov_spp, out_dir, name)
    out["filter_kernels_ms_16spp"] = sum(v for k, v in out["kernel_ms_16spp"].items() if k in FILTER_KERNELS)
    ctx.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", nargs="+", default=sorted(WORKLOADS), choices=sorted(WORKLOADS))
    ap.add_argument("--ref-spp", type=int, default=4096)
    ap.add_argument("--repeat", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    name, limit = card()
    print("card: %s, power limit %s" % (name, limit), flush=True)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
    for workload in args.workloads:
        result = run(workload, args.ref_spp, args.repeat, args.out)
        result["card"], result["power_limit"] = name, limit
        print(json.dumps(result), flush=True)
        if args.out:
            with open(os.path.join(args.out, "r04_denoise_%s.json" % workload), "w") as f:
                json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
