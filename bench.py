#!/usr/bin/env python3
"""Benchmark of the path-tracing hot path (BASELINE.json: Msamples/s and Mrays/s vs the host-CPU Embree path).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload dragon|cornell|...] [--dump-outputs DIR]

Workload (config.workload): scenes/dragon.json, 1024 x 1024, PathTracer, startBounce 0, lastBounce 10 — the
configuration the north-star target is quoted on (">= 100x the reference CPU Msamples/s on dragon.json on 1 B200").
One step = one pass of the hot path over one batch = SPP_PER_STEP samples per pixel over the whole image
(64 spp -> 67.1 M samples = one wave of the wavefront, traced as two part-waves side by side on two streams; 4 steps = the config's 256 spp).  Synthetic data: the dragon mesh and the environment
map are seeded procedural stand-ins (tools/make_assets.py) because the reference's assets/ are not in its repo.

Timed legs (all on the device with CUDA events, >= 3 warm-up steps, barrier + synchronize on both sides):
  value     ptc_render_device: framebuffer resident in HBM, no host traffic in the timed region
  e2e       ptc_render: the reference-facing call with a HOST radianceLookup buffer (H2D + D2H of the fp32
            framebuffer inside the timed region), i.e. what Integrator::run's sampleImage loop would call
  roofline  the extend (closest-hit traversal) kernel: algorithmic bytes per launch from counted node visits and
            triangle tests (SURVEY 8(d)) / mean launch duration measured live with CUDA events on the launch stream, in a
            pass of the same steps with the stages one after the other (in the `value` region launches of the two part-waves
            and the shadow-ray launches run concurrently, so a launch's duration there is not its own);
            `traffic` = DRAM bytes per launch of the same kernel from the ncu capture of THIS build (profiles/traffic.json carries
            the hash of the CUDA sources it was taken from; a capture of another build is reported as null, never scaled)
  cpu_baseline  the UNMODIFIED reference (oracle/_ref/pathed_ref_headless, Embree) on the host cores, bounded sample
L2: every wave streams its path state (67.1 M paths x 237 B = 15.9 GB incl. queues) through each stage, far more than the
126 MB L2, so no stage finds its inputs cached from the previous one; the BVH itself (~55 MB) is meant to be L2-resident.

Multi-GPU (torchrun, one rank per GPU): samples-per-pixel are split across ranks (each rank renders its own sample
indices of every pixel, Philox-keyed by (pixel, sample, bounce)); every rank's framebuffer stays in its HBM and keeps
accumulating, per step one NCCL reduce of a staging copy to rank 0 (pathed_b200.distributed.reduce_cumulative).
Default "weak": per-GPU work is fixed as N grows (spp_per_step samples per pixel per rank and step).  `--scaling strong`:
the step is the whole BASELINE job (dragon: 256 spp, teapot: 1024 spp) split over the ranks.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

WORKLOADS = {
    "dragon": dict(scene="scenes/dragon.json", width=1024, height=1024, last_bounce=10),
    "cornell": dict(scene="scenes/cornell.json", width=512, height=512, last_bounce=10),
    "cornell-glass": dict(scene="scenes/cornell-glass.json", width=512, height=512, last_bounce=10),
    "mis-pbrt": dict(scene="scenes/mis-pbrt.json", width=768, height=512, last_bounce=10),
    "teapot": dict(scene="scenes/teapot.json", width=1920, height=1080, last_bounce=10),
    # SURVEY 8(f) N3: participating medium in a Passthrough container, VolumePathTracer (one-thread-per-path kernel)
    "cornell-medium": dict(scene="scenes/cornell-medium.json", width=512, height=512, last_bounce=10, integrator="VolumePathTracer"),
}
PATH_STATE_BYTES = 237  # per path: 5 x 32 B records (ray and modulation|throughput, current + next; NEE), 4 x 16 B (hit, result x 2, out), 1 B occlusion,
                        # 4 B shadow queue, 4 B per material class queue (2 classes in the dragon scene)
SPP_PER_STEP = 64  # one wave of 2^26 paths at 1024^2: the late bounces' queues stay long enough to fill 148 SMs (profiles/README.md)
REF_SPP_PER_STEP = 1  # the CPU reference does ~0.5 Msamples/s: one spp of 1024^2 is ~2 s
STRONG_JOB_SPP = {"dragon": 256, "teapot": 1024}  # --scaling strong: one step = the whole job BASELINE.json names for the scene


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks and throttle reasons during the timed region"""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                f = [x.strip() for x in out.split(",")]
                if len(f) >= 6:
                    self.samples.append(f)
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        mhz = [float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[2 + i] == "Active" for s in self.samples)]
        return {"sm_mhz": statistics.median(mhz) if mhz else None, "sm_max_mhz": float(self.samples[0][1]), "reasons": reasons}


def run_reference(workload, steps, warmup, spp_per_step=REF_SPP_PER_STEP):
    """Times the UNMODIFIED reference renderer (Embree + PathTracer, OpenMP over the host cores)."""
    binary = os.path.join(ROOT, "oracle", "_ref", "pathed_ref_headless")
    if not os.path.exists(binary):
        return None
    w = WORKLOADS[workload]
    with tempfile.TemporaryDirectory() as tmp:
        def job(name, spp):
            path = os.path.join(tmp, name + ".json")
            json.dump({"spp": spp, "integrator": w.get("integrator", "PathTracer"), "scene": w["scene"], "startBounce": 0, "lastBounce": w["last_bounce"],
                       "output_directory": os.path.join(tmp, name), "showUI": False, "force": True,
                       "width": w["width"], "height": w["height"], "output_name": name}, open(path, "w"))
            return path
        cmd = [binary, "--root", ROOT, job("timed", steps * spp_per_step)]
        if warmup > 0:
            cmd += ["--warmup", job("warmup", warmup * spp_per_step)]
        # torchrun exports OMP_NUM_THREADS=1 to its workers; the reference arm is meant to use every host core
        env = dict(os.environ, OMP_NUM_THREADS=str(os.cpu_count() or 1))
        proc = subprocess.run(cmd, capture_output=True, text=True, env=env)
        if proc.returncode != 0:
            sys.stderr.write(proc.stderr[-4000:])
            raise RuntimeError("pathed_ref_headless exited with %d (stderr above)" % proc.returncode)
        out = proc.stdout
    line = [l for l in out.splitlines() if l.startswith("REF_RESULT")][-1]
    r = json.loads(line[len("REF_RESULT "):])
    r["spp_per_step"] = spp_per_step
    return r


def ensure_reference_inputs():
    """scenes/, assets/ and test_scenes/ are generated (git- and gpurun-ignored): a fresh box has none until
    tools/make_assets.py ran.  Where /root/reference is mounted the compiled reference is (re)built as well."""
    subprocess.check_call([sys.executable, os.path.join(ROOT, "tools", "make_assets.py")], stdout=sys.stderr)
    binary = os.path.join(ROOT, "oracle", "_ref", "pathed_ref_headless")
    if not os.path.exists(binary) and os.path.isdir("/root/reference/src"):
        subprocess.check_call(["bash", os.path.join(ROOT, "oracle", "ref", "build_ref.sh")], stdout=sys.stderr)


def workload_config(args, world):
    """`config` of the JSON line: a pure function of the command line, so that both arms print the same object"""
    w = WORKLOADS[args.workload]
    n_pix = w["width"] * w["height"]
    ppw = args.paths_per_wave or (1 << 27)  # the library's default wave size
    spp_rank = rank_spp(args, world)
    waves = max(1, -(-spp_rank // max(1, ppw // n_pix)))
    if world > 1:
        parallelism = "spp-split x%d (%s) + one NCCL reduce of the fp32 framebuffer per step" % (world, args.scaling)
    else:
        parallelism = "single GPU"
    return {"workload": "%s %dx%d %s lastBounce %d" % (w["scene"], w["width"], w["height"], w.get("integrator", "PathTracer"), w["last_bounce"]),
            "spp_per_step": step_spp(args, world), "spp_per_rank_and_step": spp_rank, "scaling": args.scaling, "parallelism": parallelism,
            "l2": "inputs larger than L2: %.0f MB of path state streamed per wave, %d wave(s) per step" % (min(n_pix * spp_rank, ppw) * PATH_STATE_BYTES / 1e6, waves)}


def rank_spp(args, world):
    if args.scaling == "strong":
        return max(1, step_spp(args, world) // world)
    return args.spp_per_step


def step_spp(args, world):
    """samples per pixel one step adds to the image, over all ranks"""
    if args.scaling == "strong":
        return args.spp_per_step if args.spp_per_step_given else STRONG_JOB_SPP.get(args.workload, 256)
    return args.spp_per_step * world


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return 0
    w = WORKLOADS[args.workload]
    ensure_reference_inputs()
    r = run_reference(args.workload, args.steps, args.warmup)
    if r is None:
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/pathed_ref_headless is not built"}))
        return 0
    value = r["msamples_per_s"]
    sample = "each step = %d spp of %dx%d (a bounded sample of the workload; throughput per sample does not depend on spp): %d spp in %d steps, " \
             "unmodified reference + Embree 3.6.0, %d OpenMP threads" % (r["spp_per_step"], w["width"], w["height"], r["spp"], args.steps, r["threads"])
    print(json.dumps({
        "impl": "reference", "metric": "Msamples/s", "value": value, "unit": "Msamples/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": r["render_wall_s"] * 1e3 / args.steps, "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, world),
        "cpu_baseline": {"value": value, "unit": "Msamples/s", "cores": r["threads"], "kind": "reference", "sample": sample},
        "e2e": {"value": value, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))
    return 0


def source_hash():
    """identifies the build a profile was taken from: sha256 over the CUDA sources"""
    import hashlib
    h = hashlib.sha256()
    d = os.path.join(ROOT, "pathed_b200", "csrc")
    for name in sorted(os.listdir(d)):
        if name.endswith((".cu", ".cuh", ".h")):
            h.update(name.encode())
            h.update(open(os.path.join(d, name), "rb").read())
    return h.hexdigest()[:16]


def profile_facts(workload):
    """ncu-derived per-ray facts of the extend kernel (profiles/traffic.json, written by tools/ncu_traffic.py from a capture of the
    bench command).  Only a capture of THIS build counts; anything else is reported as stale instead of being scaled."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(path):
        return None, "no ncu capture committed"
    t = json.load(open(path))
    if t.get("workload") != workload:
        return None, "the committed ncu capture is of workload %s" % t.get("workload")
    if t.get("source_hash") != source_hash():
        return None, "the committed ncu capture is of another build (%s, this build %s)" % (t.get("source_hash"), source_hash())
    return t, t.get("source")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=16)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="dragon", choices=sorted(WORKLOADS))
    ap.add_argument("--spp-per-step", type=int, default=None)
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: spp-per-step samples per pixel per rank and step; strong: one step = the whole BASELINE job split over the ranks")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--paths-per-wave", type=int, default=0, help="override the library's wave size (paths resident per wave)")
    ap.add_argument("--bvh-builder", type=int, default=1, choices=[0, 1], help="1: device builder (default), 0: host binned-SAH builder")
    ap.add_argument("--lanes", type=int, default=0, help="part-waves traced side by side (ptc_set_option lanes); 0: the library's choice per wave")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps write the framebuffers the timed calls left (cumulative fp32 radiance sums) to DIR/<name>.npy")
    args = ap.parse_args()
    args.spp_per_step_given = args.spp_per_step is not None
    if args.spp_per_step is None:
        args.spp_per_step = SPP_PER_STEP
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    if args.impl == "reference":
        return reference_arm(args)

    import numpy as np
    import torch

    import __graft_entry__
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    distributed = world > 1
    if distributed:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl")
    if rank == 0:
        __graft_entry__.build()
    if distributed:
        dist.barrier()
    torch.cuda.set_device(local_rank)

    from pathed_b200 import load_scene
    w = WORKLOADS[args.workload]
    width, height, last = w["width"], w["height"], w["last_bounce"]
    spp = rank_spp(args, world)          # samples per pixel THIS rank renders per step
    total_spp = spp * world              # samples per pixel one step adds to the image
    t0 = time.time()
    ctx = load_scene(w["scene"], width, height, device=local_rank, options={"bvh_builder": args.bvh_builder},
                     integrator=1 if w.get("integrator") == "VolumePathTracer" else 0)
    build_s = time.time() - t0
    tst0 = ctx.stats()
    if args.paths_per_wave:
        ctx.set_option("paths_per_wave", args.paths_per_wave)
    if args.lanes:
        ctx.set_option("lanes", args.lanes)
    n_pix = width * height
    local = torch.zeros(height * width * 3, dtype=torch.float32, device="cuda")    # this rank's cumulative radianceLookup
    staging = torch.zeros_like(local) if distributed else None                     # what the per-step reduce works on
    stream = torch.cuda.current_stream().cuda_stream
    seed = 0x5EED

    from pathed_b200.distributed import reduce_cumulative, reduce_framebuffer, sample_block

    def step_device(i):
        # global sample indices of this step: [i*world*spp, (i+1)*world*spp); this rank takes its contiguous block
        first, count = sample_block(i, rank, world, spp)
        ctx.render_device(seed, first, count, 0, last, local.data_ptr(), stream)
        if distributed:
            reduce_cumulative(local, staging, dst=0)  # rank 0's staging = the image of every sample rendered so far

    def timed(fn, steps):
        if distributed:
            dist.barrier()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(steps):
            fn(i)
        b.record()
        torch.cuda.synchronize()
        if distributed:
            dist.barrier()
        ms = torch.tensor([a.elapsed_time(b)], device="cuda")
        if distributed:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    # ---- value: device-resident framebuffer
    for i in range(args.warmup):
        step_device(i)
    torch.cuda.synchronize()
    ctx.reset_stats()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ms = timed(lambda i: step_device(i + args.warmup), args.steps)
    st = ctx.stats()
    outputs = {}
    if args.dump_outputs and rank == 0:
        # the caller's radianceLookup after the last timed step: sums of every sample rendered so far (warm-up steps included)
        outputs["radiance_device"] = (staging if distributed else local).view(height, width, 3).cpu().numpy()
    launches = int(st.kernel_launches)
    rays = int(st.closest_rays + st.shadow_rays)
    samples_total = float(n_pix) * total_spp * args.steps
    value = samples_total / (ms * 1e-3) * 1e-6
    # the multi-rank image is checked, not only timed: rank 0's reduced image = mean radiance of every rank's samples
    image_check = None
    if distributed:
        # a sample can be NaN exactly where the reference's is (teapot, 1920x1080, seed 0x5EED: sample 5318 of pixel (402, 922) is NaN in the
        # oracle too -- tools/nan_hunt.py), so the check runs over the finite pixels and reports the others
        mean_local = torch.tensor([float(torch.nan_to_num(local.double(), nan=0.0, posinf=0.0, neginf=0.0).mean())], device="cuda", dtype=torch.float64)
        dist.all_reduce(mean_local, op=dist.ReduceOp.SUM)
        if rank == 0:
            got, want = float(torch.nan_to_num(staging.double(), nan=0.0, posinf=0.0, neginf=0.0).mean()), float(mean_local.item())
            image_check = {"reduced_mean": got, "sum_of_rank_means": want, "spp": (args.steps + args.warmup) * total_spp,
                           "non_finite_values": int((~torch.isfinite(staging)).sum().item())}
            assert abs(got - want) <= 1e-4 * abs(want) + 1e-9, image_check

    # ---- e2e: the reference-facing call with a HOST radianceLookup (accumulated, not overwritten: upload, add, download).
    # N = 1: ptc_render.  N > 1: every rank renders its sample block into a cleared device buffer, one NCCL reduce brings the step's
    # sum to rank 0, which uploads the host accumulator from pinned memory, adds and downloads -- one H2D + one D2H of the
    # framebuffer per step on rank 0, nothing through the host on the other ranks
    # the host radianceLookup lives in page-locked memory (what a binding gets with one cudaHostRegister of the reference's vector):
    # ptc_render then copies from and to it directly instead of through its own staging buffer
    host_accum = torch.zeros((height, width, 3), dtype=torch.float32).pin_memory().numpy()
    fb_bytes = n_pix * 3 * 4
    if distributed:
        stepbuf = torch.zeros_like(local)
        pinned = torch.zeros(height * width * 3, dtype=torch.float32).pin_memory() if rank == 0 else None
        total = torch.zeros_like(local) if rank == 0 else None

    def step_host(i):
        if not distributed:
            ctx.render(seed, sample_block(i, rank, world, spp)[0], spp, 0, last, accum=host_accum)
            return
        stepbuf.zero_()
        first, count = sample_block(i, rank, world, spp)
        ctx.render_device(seed, first, count, 0, last, stepbuf.data_ptr(), stream)
        reduce_framebuffer(stepbuf, dst=0)
        if rank == 0:
            total.copy_(pinned, non_blocking=True)
            total.add_(stepbuf)
            pinned.copy_(total, non_blocking=True)
        torch.cuda.synchronize()

    for i in range(3):
        step_host(i)
    if distributed:
        dist.barrier()
    torch.cuda.synchronize()
    t_start = time.perf_counter()
    e2e_device_ms = 0.0
    for i in range(args.steps):
        step_host(i + 3)
        if not distributed:
            e2e_device_ms += ctx.stats().last_render_ms
    torch.cuda.synchronize()
    e2e_wall_ms = (time.perf_counter() - t_start) * 1e3
    e2e_ms = torch.tensor([max(e2e_wall_ms, e2e_device_ms)], device="cuda")
    if distributed:
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
    e2e_value = samples_total / (float(e2e_ms.item()) * 1e-3) * 1e-6
    sampler.stop_flag = True
    sampler.join(timeout=2)
    if args.dump_outputs and rank == 0:
        outputs["radiance_host"] = (pinned.numpy().reshape(height, width, 3) if distributed else host_accum).copy()
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, array in outputs.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), array)

    # ---- roofline of the dominant kernel (extend), rank 0 only: stage-timed pass, then counted pass (same seed)
    roofline, stages = None, None
    if rank == 0 and w.get("integrator") == "VolumePathTracer":
        # wavefront stages (pathed_b200/csrc/volume_wavefront.cuh): merged probe / continuation traversal, two shadow traversals,
        # logic, one material kernel per class.  Stage times from CUDA events around every launch, traversal work counted by the
        # kernels themselves in a second pass.  The roofline object describes the stage that takes the most time:
        #  traversal: 32 B ray + 2 x 16 B hit records (plain + filtered) + 80 B per inner-node visit + 48 B per triangle test
        #  shading:   the path-state records one vertex moves through the logic and material stages (DESIGN.md section 5):
        #             logic 148 B (result, modulation | throughput, two hit records, two shadow outcomes, NEE term, queue entry) +
        #             material 336 B (queue entry, ray, hit, result, modulation | throughput, 80 B triangle record; next ray, next
        #             modulation | throughput, next result, NEE record, queue entries)
        peak, peak_note = measured_peak()
        ctx.set_option("overlap_shadow", 0)  # stage times are taken with the stages one after the other
        ctx.set_option("stage_timing", 1)
        ctx.reset_stats()
        for i in range(args.steps):
            ctx.render_device(seed, i * world * spp, spp, 0, last, local.data_ptr(), stream)
        tst = ctx.stats()
        ctx.set_option("stage_timing", 0)
        ctx.set_option("count_traversal", 1)
        ctx.reset_stats()
        for i in range(args.steps):
            ctx.render_device(seed, i * world * spp, spp, 0, last, local.data_ptr(), stream)
        cst = ctx.stats()
        ctx.set_option("count_traversal", 0)
        ctx.set_option("overlap_shadow", 1)
        n_rays = max(cst.closest_rays + cst.shadow_rays, 1)
        extend_bytes = 64.0 * cst.closest_rays + 80.0 * cst.extend_inner_visits + 48.0 * cst.extend_triangle_tests
        shade_bytes = (148.0 + 336.0) * cst.closest_rays
        total_stage = tst.extend_ms + tst.shadow_ms + tst.shade_ms + tst.other_ms
        if tst.shade_ms >= tst.extend_ms:
            kernel, nbytes, t_ms, launches_k, units = "volumeLogicKernel + volumeMaterialKernel<class> (shading stages)", shade_bytes, tst.shade_ms, tst.shade_launches, "path vertices"
        else:
            kernel, nbytes, t_ms, launches_k, units = "volumeTraverseKernel<VOL_EXTEND> (probe + continuation ray in one traversal)", extend_bytes, tst.extend_ms, tst.extend_launches, "rays"
        achieved = nbytes / max(t_ms * 1e-3, 1e-12) * 1e-9
        roofline = {"bound": "hbm", "kernel": kernel, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                    "peak_source": peak_note, "bytes_per_unit": nbytes / max(cst.closest_rays, 1), "unit_of_work": units,
                    "units_per_launch": cst.closest_rays / max(launches_k, 1), "ms_per_launch": t_ms / max(launches_k, 1),
                    "inner_visits_per_ray": (cst.extend_inner_visits + cst.shadow_inner_visits) / n_rays,
                    "triangle_tests_per_ray": (cst.extend_triangle_tests + cst.shadow_triangle_tests) / n_rays,
                    "extend_frac": extend_bytes / max(tst.extend_ms * 1e-3, 1e-12) * 1e-9 / peak,
                    "shade_frac": shade_bytes / max(tst.shade_ms * 1e-3, 1e-12) * 1e-9 / peak,
                    "note": "24-triangle scene: 2 node visits and 5 triangle tests per ray, so the traversal stages cost little and the wave is "
                            "bound by the shading stages (Philox, BSDF / light sampling, medium math over dependent loads)"}
        stages = {"extend_ms": tst.extend_ms, "shadow_ms": tst.shadow_ms, "shade_ms": tst.shade_ms, "other_ms": tst.other_ms,
                  "extend_share": tst.extend_ms / max(total_stage, 1e-9), "shade_share": tst.shade_ms / max(total_stage, 1e-9),
                  "extend_grays_per_s": cst.closest_rays / max(tst.extend_ms, 1e-9) * 1e-6,
                  "shadow_grays_per_s": cst.shadow_rays / max(tst.shadow_ms, 1e-9) * 1e-6}
    elif rank == 0:
        peak, peak_note = measured_peak()
        # per-stage times are taken with the stages one after the other (in the timed region above the shadow rays of a bounce are traced
        # on a second stream, concurrently with its extend rays, and the stage times would overlap)
        ctx.set_option("overlap_shadow", 0)
        ctx.set_option("stage_timing", 1)
        ctx.reset_stats()
        for i in range(args.steps):
            ctx.render_device(seed, i * world * spp, spp, 0, last, local.data_ptr(), stream)
        tst = ctx.stats()
        ctx.set_option("stage_timing", 0)
        ctx.set_option("count_traversal", 1)
        ctx.reset_stats()
        count_steps = min(args.steps, 2)
        for i in range(count_steps):
            ctx.render_device(seed, i * world * spp, spp, 0, last, local.data_ptr(), stream)
        cst = ctx.stats()
        ctx.set_option("count_traversal", 0)
        ctx.set_option("overlap_shadow", 1)
        # algorithmic bytes per extend ray: 32 B ray + 16 B hit record + 80 B per inner node + 48 B per triangle test
        per_ray = 32 + 16 + (80.0 * cst.extend_inner_visits + 48.0 * cst.extend_triangle_tests) / max(cst.closest_rays, 1)
        extend_rays_per_launch = tst.closest_rays / max(tst.extend_launches, 1)
        bytes_per_launch = per_ray * extend_rays_per_launch
        ms_per_launch = tst.extend_ms / max(tst.extend_launches, 1)
        achieved = bytes_per_launch / (ms_per_launch * 1e-3) * 1e-9
        facts, facts_source = profile_facts(args.workload)
        traffic = facts["extend_dram_bytes_per_ray"] * extend_rays_per_launch if facts else None
        l2_peak = None
        lpath = os.path.join(ROOT, "profiles", "l2_peak.json")
        if os.path.exists(lpath):
            l2_peak = json.load(open(lpath))
        total_stage = tst.extend_ms + tst.shadow_ms + tst.shade_ms + tst.other_ms
        roofline = {"bound": "hbm", "kernel": "traverseKernel<false> (extend: closest-hit BVH traversal)", "achieved": achieved, "peak": peak,
                    "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_source": facts_source, "peak_source": peak_note,
                    "bytes_per_ray": per_ray, "inner_visits_per_ray": cst.extend_inner_visits / max(cst.closest_rays, 1),
                    "triangle_tests_per_ray": cst.extend_triangle_tests / max(cst.closest_rays, 1),
                    "rays_per_launch": extend_rays_per_launch, "ms_per_launch": ms_per_launch,
                    "limiter": "instruction issue, then L2->L1 bandwidth: the BVH (%.1f MB) is L2-resident, so `achieved` (algorithmic bytes, the contract's "
                               "definition) exceeds the DRAM traffic and the HBM ceiling is not the wall this kernel runs into" % (tst.bvh_bytes / 1e6)}
        if facts:
            roofline["issue_active"] = facts.get("extend_issue_active")
            roofline["lanes_per_instruction"] = facts.get("extend_lanes_per_instruction")
            if l2_peak and facts.get("extend_l2_bytes_per_ray"):
                l2_rate = facts["extend_l2_bytes_per_ray"] * extend_rays_per_launch / (ms_per_launch * 1e-3) * 1e-9
                roofline["l2_gbs"] = l2_rate
                roofline["l2_peak_gbs"] = l2_peak["l2_read_gbs"]
                roofline["l2_frac"] = l2_rate / l2_peak["l2_read_gbs"]
                roofline["l2_peak_source"] = l2_peak.get("source")
        ext_counts, sh_counts = ctx.wave_counts(last + 2)
        stages = {"last_wave_extend_rays": ext_counts, "last_wave_shadow_rays": sh_counts, "extend_ms": tst.extend_ms, "shadow_ms": tst.shadow_ms, "shade_ms": tst.shade_ms, "other_ms": tst.other_ms,
                  "extend_share": tst.extend_ms / max(total_stage, 1e-9), "extend_grays_per_s": tst.closest_rays / max(tst.extend_ms, 1e-9) * 1e-6,
                  "shadow_grays_per_s": tst.shadow_rays / max(tst.shadow_ms, 1e-9) * 1e-6}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        r = run_reference(args.workload, steps=8, warmup=1)
        if r is not None:
            cpu = {"value": r["msamples_per_s"], "unit": "Msamples/s", "cores": r["threads"], "kind": "reference",
                   "sample": "%d spp of %dx%d after 1 warm-up spp, unmodified reference + Embree 3.6.0, %d OpenMP threads, %.1f s"
                             % (r["spp"], width, height, r["threads"], r["render_wall_s"])}

    # the first build of a process also pays for CUDA's lazy module loading (every builder kernel, cub's sort and scan) and the first
    # large allocations; a second scene in the same process shows the builder itself.  Done after everything that is timed: earlier
    # allocations and frees move later ones, and the throughput of the tiny scenes depends on where a handful of hot lines land.
    warm_build_ms = None
    if rank == 0 and not distributed:
        again = load_scene(w["scene"], width, height, device=local_rank, options={"bvh_builder": args.bvh_builder},
                           integrator=1 if w.get("integrator") == "VolumePathTracer" else 0)
        warm_build_ms = again.stats().bvh_build_ms
        again.close()

    if rank == 0:
        line = {
            "metric": "Msamples/s", "value": value, "unit": "Msamples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": workload_config(args, world),
            "setup": {"scene_build_s": build_s,
                      "lanes": args.lanes or "chosen per wave: 4 part-waves side by side for waves of <= 2^25 paths, else 2 (stage / counter passes: 1)",
                      "bvh_build": {"builder": "device (Morton sort + PLOC + wide collapse kernels)" if tst0.bvh_builder else "host binned SAH",
                                    "ms": tst0.bvh_build_ms, "ms_second_build_in_process": warm_build_ms, "triangles": tst0.bvh_triangles, "nodes": tst0.bvh_nodes, "depth": tst0.bvh_depth}},
            "mrays_per_s": rays * world / (ms * 1e-3) * 1e-6, "rays_per_sample": rays / (samples_total / world),
            "e2e": {"value": e2e_value, "unit": "Msamples/s", "h2d_bytes_per_step": fb_bytes, "d2h_bytes_per_step": fb_bytes,
                    "wall_ms_per_step": e2e_wall_ms / args.steps, "device_ms_per_step": (e2e_device_ms / args.steps) if not distributed else None},
            "gpu_launches": launches, "clocks": sampler.summary(), "roofline": roofline, "stages": stages, "cpu_baseline": cpu,
        }
        if image_check:
            line["multi_gpu_image_check"] = image_check
        print(json.dumps(line))
    if distributed:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
