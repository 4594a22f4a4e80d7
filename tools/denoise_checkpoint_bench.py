"""What do denoised checkpoints cost?  (a) one denoised image through ptc_denoise (host inputs) against ptc_framebuffer_denoise_begin
+ ptc_framebuffer_gather_end (device inputs), and (b) whole `pathed` jobs with "denoise" against "denoise" + "denoise_checkpoints".

(a) For each workload: a uniform 16-spp render with the option "framebuffer_moments" on and the guides of its first 16 samples.  The
host path gathers sums and moments to the host and renders the guides with ptc_render_aovs once (untimed), then times ptc_denoise
alone; the device path times ptc_framebuffer_denoise_begin + _gather_end from the same render and ptc_framebuffer_guides.  Both with
a synchronised host clock, best of --repeat, default filter parameters; the two images must be the same bytes.  Then each path runs
once under torch.profiler with CUDA activities (a run of its own) and the device time of its filter kernels is summed.
(b) `pathed` jobs (PathTracer, lastBounce 10, wave_spp 64): dragon 1024^2 at 256 spp and cornell-glass 512^2 at 1024 spp, the two
job variants alternating, best of --job-repeat: the process's wall time and its render loop (PATHED_RESULT render_wall_s, which
includes the checkpoints' denoising).  Outputs go to a temporary directory.

Prints the card's name and power limit and one JSON object per workload; writes them to --out/r05_denoise_checkpoints_<workload>.json.

    python tools/denoise_checkpoint_bench.py [--workloads cornell-glass dragon] [--out DIR]
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from pathed_b200 import load_scene  # noqa: E402
from pathed_b200._binding import GATHER_MOMENTS, PKG_DIR  # noqa: E402

WORKLOADS = {
    "cornell-glass": dict(scene="scenes/cornell-glass.json", width=512, height=512, job_spp=1024),
    "dragon": dict(scene="scenes/dragon.json", width=1024, height=1024, job_spp=256),
}
SPP, GUIDE_SPP, SEED, LAST = 16, 16, 1, 10
HOST_KERNELS = ("denoisePrepareKernel", "denoiseAtrousKernel")
DEVICE_KERNELS = ("denoiseGatherKernel", "denoiseAtrousKernel", "denoisePackKernel")


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        limit = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                               text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = "unknown"
    return name, limit


def timed(fn, repeat):
    runs, out = [], None
    for _ in range(repeat):
        t0 = time.perf_counter()
        out = fn()
        runs.append(time.perf_counter() - t0)
    return min(runs), runs, out


def kernel_ms(fn, names):
    """device time per kernel name of one call of fn under torch.profiler"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    per = {}
    for e in prof.key_averages():
        for k in names:
            if k in e.key:
                per[k] = per.get(k, 0.0) + e.device_time_total / 1000.0
    return per


def one_image(w, repeat):
    ctx = load_scene(w["scene"], w["width"], w["height"])
    ctx.set_option("framebuffer_moments", 1)
    ctx.framebuffer_clear()
    ctx.framebuffer_render(SEED, 0, SPP, 0, LAST)
    sums, moments = ctx.framebuffer_gather([], divisor=1), ctx.framebuffer_gather([], 1, GATHER_MOMENTS)
    aovs = ctx.render_aovs(SEED, 0, GUIDE_SPP)
    ctx.framebuffer_guides(SEED, 0, GUIDE_SPP)
    host = lambda: ctx.denoise(sums, moments, SPP, aovs, GUIDE_SPP)
    device = lambda: ctx.framebuffer_denoise([], -1, SPP)
    host(); device()  # warm-up: buffers, module load
    host_s, host_runs, a = timed(host, repeat)
    device_s, device_runs, b = timed(device, repeat)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), "the two paths differ"
    guides_sync_s, guides_sync_runs, _ = timed(lambda: (ctx.framebuffer_guides(SEED, 0, GUIDE_SPP), ctx.framebuffer_gather([], 1)), repeat)
    out = {"ptc_denoise_s": host_s, "ptc_denoise_all_s": host_runs, "framebuffer_denoise_s": device_s, "framebuffer_denoise_all_s": device_runs,
           "framebuffer_guides_and_gather_s": guides_sync_s, "same_bytes": True,
           "ptc_denoise_kernel_ms": kernel_ms(host, HOST_KERNELS), "framebuffer_denoise_kernel_ms": kernel_ms(device, DEVICE_KERNELS)}
    ctx.close()
    return out


def job(w, tmp, checkpoints):
    out_dir = os.path.join(tmp, "out")
    shutil.rmtree(out_dir, ignore_errors=True)
    spec = {"spp": w["job_spp"], "integrator": "PathTracer", "scene": w["scene"], "startBounce": 0, "lastBounce": LAST, "width": w["width"],
            "height": w["height"], "output_directory": out_dir, "output_name": "final", "showUI": False, "force": True, "denoise": True}
    if checkpoints:
        spec["denoise_checkpoints"] = True
    path = os.path.join(tmp, "job.json")
    json.dump(spec, open(path, "w"))
    t0 = time.perf_counter()
    r = subprocess.run([os.path.join(PKG_DIR, "pathed"), path, "--root", ROOT], capture_output=True, text=True)
    wall = time.perf_counter() - t0
    if r.returncode != 0:
        raise RuntimeError(r.stdout + r.stderr)
    result = json.loads(r.stdout.split("PATHED_RESULT ", 1)[1].splitlines()[0])
    files = sorted(f for f in os.listdir(out_dir) if f.startswith("denoised-auto-"))
    return {"wall_s": wall, "render_wall_s": result["render_wall_s"], "denoised_checkpoints": len(files)}


def jobs(w, repeat):
    tmp = tempfile.mkdtemp(prefix="denoise_checkpoint_bench_")
    try:
        job(w, tmp, False)  # warm-up: page cache of the scene files, driver
        runs = {"denoise": [], "denoise_checkpoints": []}
        for _ in range(repeat):
            for key in runs:
                runs[key].append(job(w, tmp, key == "denoise_checkpoints"))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    out = {}
    for key, rs in runs.items():
        out[key] = {"wall_s": min(r["wall_s"] for r in rs), "render_wall_s": min(r["render_wall_s"] for r in rs),
                    "denoised_checkpoints": rs[0]["denoised_checkpoints"], "runs": rs}
    out["overhead_wall_s"] = out["denoise_checkpoints"]["wall_s"] - out["denoise"]["wall_s"]
    out["overhead_render_wall_s"] = out["denoise_checkpoints"]["render_wall_s"] - out["denoise"]["render_wall_s"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", nargs="+", default=sorted(WORKLOADS), choices=sorted(WORKLOADS))
    ap.add_argument("--repeat", type=int, default=5)
    ap.add_argument("--job-repeat", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    name, limit = card()
    print("card: %s, power limit %s" % (name, limit), flush=True)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
    for workload in args.workloads:
        w = WORKLOADS[workload]
        result = {"workload": "%s %dx%d PathTracer lastBounce %d" % (w["scene"], w["width"], w["height"], LAST), "card": name, "power_limit": limit,
                  "image": dict(one_image(w, args.repeat), spp=SPP, guide_spp=GUIDE_SPP),
                  "job": dict(jobs(w, args.job_repeat), spp=w["job_spp"], wave_spp=64)}
        print(json.dumps(result), flush=True)
        if args.out:
            with open(os.path.join(args.out, "r05_denoise_checkpoints_%s.json" % workload), "w") as f:
                json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
