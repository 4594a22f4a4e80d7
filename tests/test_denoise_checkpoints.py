"""GPU tests of device-resident denoising (DESIGN §10, denoised checkpoints): the second moments the checkpoint snapshots keep,
ptc_framebuffer_guides against ptc_render_aovs, ptc_framebuffer_denoise_begin against ptc_denoise on the gathered inputs (byte for
byte), its refusals, and the `pathed` job key "denoise_checkpoints"."""
import json
import os
import subprocess

import numpy as np
import pytest

from parity import half_like_reference

from pathed_b200 import load_scene, read_exr
from pathed_b200._binding import GATHER_MOMENTS, PKG_DIR, REPO_ROOT, VOLUME_PATH_TRACER, PathedError

pytestmark = pytest.mark.gpu

SEED, LAST, GUIDE_SPP = 13, 10, 8
W, H = 24, 16
SETTINGS = {"lanes1": {"lanes": 1}, "default": {}, "small_waves": {"paths_per_wave": 3000}}
INTEGRATORS = {"pt": ("scenes/cornell-glass.json", 0), "vpt": ("scenes/cornell-medium.json", VOLUME_PATH_TRACER)}
PARAMS = {"defaults": {}, "other": {"iterations": 3, "sigma_l": 1.0, "sigma_n": 16.0, "sigma_z": 0.5, "sigma_a": 0.5}, "none": {"iterations": 0}}


def _context(scene="scenes/cornell-glass.json", integrator=0, options=None, moments=True, width=W, height=H):
    if not os.path.exists(os.path.join(REPO_ROOT, scene)):
        pytest.skip(scene + " not generated")
    ctx = load_scene(scene, width, height, integrator=integrator)
    for name, value in dict(options or {}, framebuffer_moments=int(moments)).items():
        ctx.set_option(name, value)
    return ctx


def _same(a, b):
    assert a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def _fresh(ctx, blocks, k, seed=SEED):
    """sums and second moments of `ctx`'s samples below k out of `blocks` [(first, n), ...], rendered from a cleared framebuffer"""
    ctx.framebuffer_clear()
    for first, n in blocks:
        if first < k:
            ctx.framebuffer_render(seed, first, min(n, k - first), 0, LAST)
    return ctx.framebuffer_gather([], divisor=1), ctx.framebuffer_gather([], 1, GATHER_MOMENTS)


# ------------------------------------------------------------------------------------------------ moment snapshots
@pytest.mark.parametrize("setting", sorted(SETTINGS))
@pytest.mark.parametrize("integrator", sorted(INTEGRATORS))
def test_snapshots_keep_the_moments_of_a_render_that_stopped_there(integrator, setting):
    """snapshot i's sums are read with the gather; its moments through the denoise, which must give ptc_denoise's bytes for the
    sums and moments of a fresh render of samples 0 .. k - 1 (a variance that differs changes the filter's weights)"""
    scene, kind = INTEGRATORS[integrator]
    ctx = _context(scene, kind, SETTINGS[setting])
    fresh = _context(scene, kind, SETTINGS[setting])
    aovs = ctx.framebuffer_guides(SEED, 0, GUIDE_SPP, fetch=True)
    counts = [2, 3, 6]
    ctx.framebuffer_clear()
    ctx.framebuffer_render(SEED, 0, 1, 0, LAST)  # the moments carry over from an earlier call
    ctx.framebuffer_render_checkpoints(SEED, 1, 8, 0, LAST, counts)
    for i, k in enumerate(counts):
        S, M = _fresh(fresh, [(0, 9)], k)
        _same(ctx.framebuffer_gather([], 1, i), S)
        _same(ctx.framebuffer_denoise([], i, k), ctx.denoise(S, M, k, aovs, GUIDE_SPP))
        _same(ctx.framebuffer_denoise([], i, k, iterations=1), ctx.denoise(S, M, k, aovs, GUIDE_SPP, iterations=1))
    S, M = _fresh(fresh, [(0, 9)], 9)
    _same(ctx.framebuffer_denoise([], -1, 9), ctx.denoise(S, M, 9, aovs, GUIDE_SPP))


def test_a_context_without_samples_in_the_wave_snapshots_its_current_moments():
    ctx = _context()
    ctx.framebuffer_guides(SEED, 0, GUIDE_SPP)
    ctx.framebuffer_clear()
    ctx.framebuffer_render(SEED, 0, 5, 0, LAST)
    ctx.framebuffer_render_checkpoints(SEED, 5, 0, 0, LAST, [6, 7])
    whole = ctx.framebuffer_denoise([], -1, 5)
    for i in range(2):
        _same(ctx.framebuffer_gather([], 1, i), ctx.framebuffer_gather([], 1))
        _same(ctx.framebuffer_denoise([], i, 5), whole)
    # as the peer of a job's wave: a GPU that got no samples adds its zeros, sums and moments alike
    other = _context()
    other.framebuffer_clear()
    other.framebuffer_render_checkpoints(SEED, 5, 0, 0, LAST, [6, 7])
    _same(ctx.framebuffer_denoise([other], 1, 5), whole)


# ------------------------------------------------------------------------------------------------ device denoise = ptc_denoise
def test_framebuffer_guides_equal_render_aovs_from_zero():
    ctx = _context()
    want = ctx.render_aovs(SEED, 3, 7)
    for _ in range(2):  # a call starts from zero: it replaces the previous guides
        got = ctx.framebuffer_guides(SEED, 3, 7, fetch=True)
        for key in want:
            assert np.array_equal(got[key], want[key]), key
    assert ctx.framebuffer_guides(SEED, 0, 4) is None


@pytest.mark.parametrize("params", sorted(PARAMS))
def test_denoise_of_two_contexts_equals_ptc_denoise_of_the_gather(params):
    """a job's wave over samples 0 .. 9 on two contexts (0 .. 4 and 5 .. 9) with checkpoints at 2 and 8"""
    p = PARAMS[params]
    a, b, c = _context(), _context(), _context()
    aovs = a.framebuffer_guides(SEED, 0, GUIDE_SPP, fetch=True)
    for ctx, first in ((a, 0), (b, 5)):
        ctx.framebuffer_clear()
        ctx.framebuffer_render_checkpoints(SEED, first, 5, 0, LAST, [2, 8])
    for snapshot, k, blocks in ((-1, 10, [(0, 5), (5, 5)]), (0, 2, [(0, 5), (5, 5)]), (1, 8, [(0, 5), (5, 5)])):
        (Sa, Ma), (Sb, Mb) = _fresh(c, blocks[:1], k), _fresh(c, blocks[1:], k)
        S, M = Sa + Sb, Ma + Mb  # fp32, root first: the gather's order
        _same(a.framebuffer_gather([b], 1, snapshot), S)
        _same(a.framebuffer_denoise([b], snapshot, k, **p), a.denoise(S, M, k, aovs, GUIDE_SPP, **p))
    # tickets: several in flight, fetched in any order
    t = [a.framebuffer_denoise_begin([b], s, k, **p) for s, k in ((1, 8), (-1, 10))]
    _same(a.framebuffer_gather_end(t[1]), a.framebuffer_denoise([b], -1, 10, **p))
    _same(a.framebuffer_gather_end(t[0]), a.framebuffer_denoise([b], 1, 8, **p))


def test_denoise_of_an_adaptive_root_uses_its_counts_and_moments():
    ctx = _context(moments=False)
    aovs = ctx.framebuffer_guides(SEED, 0, GUIDE_SPP, fetch=True)
    ctx.adaptive_begin(0.1, 4, 4, 16)
    while True:
        active, _ = ctx.adaptive_pass(SEED, 0, LAST)
        S = ctx.framebuffer_gather([], divisor=1)
        counts, M = ctx.adaptive_state()
        for p in PARAMS.values():
            _same(ctx.framebuffer_denoise([], -1, 0, **p), ctx.denoise(S, M, counts, aovs, GUIDE_SPP, **p))
        if not active:
            break


# ------------------------------------------------------------------------------------------------ refusals
def _status(code, fn, *args, **kw):
    with pytest.raises(PathedError, match="status %d" % code):
        fn(*args, **kw)


INVALID, STATE = -1, -3


def test_refusals():
    ctx = _context()
    ctx.framebuffer_clear()
    ctx.framebuffer_render_checkpoints(SEED, 0, 4, 0, LAST, [2])
    _status(STATE, ctx.framebuffer_denoise, [], -1, 4)  # no guides yet
    _status(INVALID, ctx.framebuffer_guides, SEED, 0, 0)
    ctx.framebuffer_guides(SEED, 0, GUIDE_SPP)
    ctx.framebuffer_denoise([], -1, 4)
    ctx.framebuffer_denoise([], 0, 2)
    for bad in ({"iterations": 11}, {"sigma_l": 0.0}, {"sigma_n": -1.0}, {"eps": float("nan")}):
        _status(INVALID, ctx.framebuffer_denoise, [], -1, 4, **bad)
    _status(INVALID, ctx.framebuffer_denoise, [], -1, 1)  # one sample: no variance
    _status(STATE, ctx.framebuffer_denoise, [], 1, 4)  # snapshot 1 was never rendered
    # moments that miss samples: the option off for a render, of the framebuffer and of the snapshots written then
    ctx.set_option("framebuffer_moments", 0)
    ctx.framebuffer_render_checkpoints(SEED, 4, 2, 0, LAST, [5])
    _status(STATE, ctx.framebuffer_denoise, [], -1, 6)
    _status(STATE, ctx.framebuffer_denoise, [], 0, 5)
    # a peer without moments
    ctx.set_option("framebuffer_moments", 1)
    ctx.framebuffer_clear()
    ctx.framebuffer_render(SEED, 0, 4, 0, LAST)
    peer = _context(moments=False)
    peer.framebuffer_clear()
    peer.framebuffer_render(SEED, 4, 2, 0, LAST)
    _status(STATE, ctx.framebuffer_denoise, [peer], -1, 6)
    # an adaptive root before its first pass, and its snapshots
    ctx.adaptive_begin(0.1, 4, 4, 8)
    _status(STATE, ctx.framebuffer_denoise, [], -1, 0)
    ctx.adaptive_pass(SEED, 0, LAST)
    ctx.framebuffer_denoise([], -1, 0)
    _status(STATE, ctx.framebuffer_denoise, [], 0, 0)
    # guides of another resolution
    ctx.set_camera((0, 1, 4), (0, 1, 0), (0, 1, 0), 40.0, W + 8, H)
    ctx.framebuffer_clear()
    ctx.framebuffer_render(SEED, 0, 4, 0, LAST)
    _status(STATE, ctx.framebuffer_denoise, [], -1, 4)
    ctx.framebuffer_guides(SEED, 0, GUIDE_SPP)
    assert ctx.framebuffer_denoise([], -1, 4).shape == (H, W + 8, 3)
    _status(STATE, ctx.framebuffer_denoise, [], 0, 2)  # the snapshot is of the old resolution
    _status(STATE, ctx.framebuffer_gather, [], 1, 0)
    ctx.framebuffer_clear()
    ctx.framebuffer_render_checkpoints(SEED, 0, 4, 0, LAST, [2])  # new snapshots of the new size
    fresh = _context(width=W + 8, height=H)
    fresh.set_camera((0, 1, 4), (0, 1, 0), (0, 1, 0), 40.0, W + 8, H)
    S, M = _fresh(fresh, [(0, 4)], 2)
    _same(ctx.framebuffer_denoise([], 0, 2), ctx.denoise(S, M, 2, ctx.render_aovs(SEED, 0, GUIDE_SPP), GUIDE_SPP))
    # the same number of pixels in another shape
    ctx.set_camera((0, 1, 4), (0, 1, 0), (0, 1, 0), 40.0, H, W + 8)
    ctx.framebuffer_clear()
    ctx.framebuffer_render(SEED, 0, 4, 0, LAST)
    _status(STATE, ctx.framebuffer_denoise, [], -1, 4)


# ------------------------------------------------------------------------------------------------ the job key
JOB_SEED = 0x5EED


def _run_job(tmp_path, **over):
    job = {"spp": 16, "integrator": "PathTracer", "scene": "scenes/cornell-glass.json", "startBounce": 0, "lastBounce": 10,
           "output_directory": str(tmp_path / "out"), "output_name": "final", "showUI": False, "force": True, "width": 48, "height": 40,
           "wave_spp": 5, "denoise": True}
    job.update(over)
    os.makedirs(str(tmp_path), exist_ok=True)
    path = str(tmp_path / "job.json")
    json.dump(job, open(path, "w"))
    r = subprocess.run([os.path.join(PKG_DIR, "pathed"), path, "--root", REPO_ROOT], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    return str(tmp_path / "out")


def _check_job(tmp_path, expected, **over):
    """expected: spp -> the denoised image (row 0 = bottom) of the checkpoint of that many samples"""
    out = _run_job(tmp_path / "checkpoints", denoise_checkpoints=True, **over)
    plain = _run_job(tmp_path / "plain", **over)
    files = sorted(f for f in os.listdir(out) if f.startswith("denoised-auto-"))
    assert files == ["denoised-auto-%05dspp.exr" % k for k in sorted(expected)]
    for k, image in expected.items():
        got = read_exr(os.path.join(out, "denoised-auto-%05dspp.exr" % k))[..., :3]
        assert np.array_equal(got, half_like_reference(image[::-1])), k
    latest = open(os.path.join(out, "denoised-auto-%05dspp.exr" % max(expected)), "rb").read()
    assert open(os.path.join(out, "denoised-auto.exr"), "rb").read() == latest
    kept = lambda d: {f: open(os.path.join(d, f), "rb").read() for f in os.listdir(d)
                      if f in ("final.exr", "denoised.exr", "albedo.exr", "normal.exr") or f.startswith("auto")}
    images = kept(out)
    assert len(images) > 4 and images == kept(plain)  # the checkpoints add files and change none


def test_cli_denoise_checkpoints_job(tmp_path):
    ctx = _context(width=48, height=40)
    aovs = ctx.render_aovs(JOB_SEED, 0, 16)
    expected = {}
    for k in (2, 4, 8, 16):
        S, M = _fresh(ctx, [(0, 16)], k, JOB_SEED)
        expected[k] = ctx.denoise(S, M, k, aovs, 16)
    _check_job(tmp_path, expected)


def test_cli_denoise_checkpoints_adaptive_job(tmp_path):
    ctx = _context(width=48, height=40, moments=False)
    aovs = ctx.render_aovs(JOB_SEED, 0, 16)
    ctx.adaptive_begin(0.1, 4, 4, 32)
    expected = {}
    while True:
        active, n = ctx.adaptive_pass(JOB_SEED, 0, LAST)
        if (n & (n - 1)) == 0:
            counts, M = ctx.adaptive_state()
            expected[n] = ctx.denoise(ctx.framebuffer_gather([], divisor=1), M, counts, aovs, 16)
        if not active:
            break
    _check_job(tmp_path, expected, spp=32, adaptive_threshold=0.1, adaptive_min_spp=4, adaptive_step_spp=4)


def test_cli_denoise_checkpoints_job_on_two_gpus(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    ctx = _context(width=48, height=40)
    aovs = ctx.render_aovs(JOB_SEED, 0, 16)
    # the job's split: waves of wave_spp per GPU, each wave cut into two contiguous halves
    blocks = ([], [])
    for first in range(0, 16, 10):
        end = min(first + 10, 16)
        per = (end - first + 1) // 2
        blocks[0].append((first, per)); blocks[1].append((first + per, end - first - per))
    expected = {}
    for k in (2, 4, 8, 16):
        (Sa, Ma), (Sb, Mb) = _fresh(ctx, blocks[0], k, JOB_SEED), _fresh(ctx, blocks[1], k, JOB_SEED)
        expected[k] = ctx.denoise(Sa + Sb, Ma + Mb, k, aovs, 16)
    _check_job(tmp_path, expected, gpus=2)
