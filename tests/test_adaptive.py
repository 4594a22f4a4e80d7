"""GPU tests of adaptive sampling (ptc_adaptive_begin / _pass / _state and the `pathed` job keys): each pixel stops once the estimated
relMSE term of its mean meets tau^2.  A path's random stream is keyed by (pixel, sample) and the resolve adds a pixel's samples in sample
order, so an adaptive framebuffer is, pixel by pixel, bit for bit the framebuffer of a fixed render with that pixel's sample count."""
import json
import os
import re
import subprocess

import numpy as np
import pytest

from parity import half_like_reference, rel_mse

from pathed_b200 import load_scene, read_exr
from pathed_b200._binding import PKG_DIR, REPO_ROOT, VOLUME_PATH_TRACER, PathedError

pytestmark = pytest.mark.gpu

SEED, LAST = 11, 10
MIN, STEP, MAX = 4, 3, 17  # passes end at 4, 7, 10, 13, 16, 17: the last one is ragged
PASS_ENDS = [4, 7, 10, 13, 16, 17]

SCENES = {
    "cornell_glass": ("scenes/cornell-glass.json", 0, {}),
    "mis": ("scenes/mis-pbrt.json", 0, {}),
    "instanced": ("scenes/instanced.json", 0, {}),
    "cornell_medium": ("scenes/cornell-medium.json", VOLUME_PATH_TRACER, {}),
    "cornell_medium_megakernel": ("scenes/cornell-medium.json", VOLUME_PATH_TRACER, {"volume_megakernel": 1}),
}
# lanes 1, the per-wave default, and a paths_per_wave that splits every pass of a 48 x 48 image into several waves
SETTINGS = {"lanes1": {"lanes": 1}, "default": {}, "small_waves": {"paths_per_wave": 3000}}


def _context(scene, width, height, integrator, options):
    if not os.path.exists(os.path.join(REPO_ROOT, scene)):
        pytest.skip(scene + " not generated")
    ctx = load_scene(scene, width, height, integrator=integrator)
    for name, value in options.items():
        ctx.set_option(name, value)
    return ctx


def _adaptive_render(ctx, tau, lo=MIN, step=STEP, hi=MAX, seed=SEED, last=LAST):
    ctx.adaptive_begin(tau, lo, step, hi)
    passes = []
    while True:
        active, n = ctx.adaptive_pass(seed, 0, last)
        passes.append((active, n))
        if active == 0:
            break
    counts, m2 = ctx.adaptive_state()
    return ctx.framebuffer_gather([], divisor=1), counts, m2, passes


@pytest.mark.parametrize("setting", sorted(SETTINGS))
@pytest.mark.parametrize("name", sorted(SCENES))
def test_adaptive_sums_equal_fixed_renders_pixel_by_pixel(name, setting):
    scene, integrator, options = SCENES[name]
    ctx = _context(scene, 48, 48, integrator, dict(options, **SETTINGS[setting]))
    # a threshold that leaves both pixels that stopped early and pixels that ran to MAX (the scenes differ in noise)
    for tau in (0.1, 0.05, 0.2, 0.4):
        ctx.reset_stats()
        sums, counts, m2, passes = _adaptive_render(ctx, tau)
        if counts.min() < MAX and counts.max() == MAX:
            break
    assert counts.min() < MAX and counts.max() == MAX, (name, np.unique(counts))
    assert [n for _, n in passes] == PASS_ENDS[:len(passes)] and passes[-1] == (0, MAX)
    assert set(np.unique(counts)) <= set(PASS_ENDS)
    assert ctx.stats().samples == int(counts.sum())  # the samples actually traced
    for n in np.unique(counts):
        mask = counts == n
        want = ctx.render(SEED, 0, int(n), 0, LAST)  # from zero into a host buffer: the framebuffer stays the adaptive one
        assert np.array_equal(sums[mask], want[mask], equal_nan=True), (name, setting, n)
    assert np.isfinite(sums).all() and sums.mean() > 0


def test_min_equal_to_max_is_one_fixed_pass():
    ctx = _context("scenes/cornell-glass.json", 48, 40, 0, {})
    sums, counts, _, passes = _adaptive_render(ctx, 0.1, lo=8, step=3, hi=8)
    assert passes == [(0, 8)] and (counts == 8).all()
    assert np.array_equal(sums, ctx.render(SEED, 0, 8, 0, LAST), equal_nan=True)


def _criterion(S, M, n, tau):
    """the stopping test in numpy, in the device's fp64 operation order; (stop, distance to the boundary relative to it)"""
    S = S.astype(np.float64); M = M.astype(np.float64)
    mean = S / n
    sq = mean * mean
    var = (M - n * sq) / (n - 1.0)
    var = np.where(var < 0.0, 0.0, var)
    tau2 = np.float64(np.float32(tau)) ** 2
    lhs, rhs = var / n, tau2 * (sq + 1e-2)
    with np.errstate(invalid="ignore"):
        stop = (np.isfinite(mean) & np.isfinite(var) & (lhs <= rhs)).all(-1)
        margin = np.where(np.isfinite(lhs), np.abs(lhs - rhs) / rhs, np.inf).min(-1)
    return stop, margin


def test_moments_and_stopping_decision_match_single_sample_renders():
    ctx = _context("scenes/cornell-glass.json", 16, 16, 0, {})
    singles = [ctx.render(SEED, s, 1, 0, LAST) for s in range(MAX)]  # from zero: the sample values themselves
    S, M = np.zeros_like(singles[0]), np.zeros_like(singles[0])
    running = {}
    for s, x in enumerate(singles):  # fp32, in sample order, product and sum rounded separately like the accumulate kernel
        S = S + x
        M = M + x * x
        running[s + 1] = (S.copy(), M.copy())
    for tau in (0.1, 0.05, 0.2, 0.4):
        sums, counts, m2, _ = _adaptive_render(ctx, tau)
        if counts.min() < MAX and counts.max() == MAX:
            break
    assert counts.min() < MAX and counts.max() == MAX, np.unique(counts)
    assert set(np.unique(counts)) <= set(PASS_ENDS)
    want_S = np.zeros_like(sums); want_M = np.zeros_like(m2)
    for n in np.unique(counts):
        mask = counts == n
        want_S[mask], want_M[mask] = running[int(n)][0][mask], running[int(n)][1][mask]
    assert np.array_equal(sums, want_S, equal_nan=True)
    assert np.allclose(m2, want_M, rtol=1e-6, atol=0, equal_nan=True)
    TIE = 1e-9  # a pixel this close to the boundary may fall either way
    for n in PASS_ENDS[:-1]:
        stop, margin = _criterion(*running[n], n, tau)
        clear = margin > TIE
        stopped_here, still_going = counts == n, counts > n
        assert stop[stopped_here & clear].all(), n     # it stopped at n: the test held there
        assert not stop[still_going & clear].any(), n  # it went on past n: the test failed there


def test_error_target_against_a_converged_render():
    tau, lo, step, hi = 0.1, 16, 16, 1024
    ctx = _context("scenes/cornell-glass.json", 128, 128, 0, {})
    reference = ctx.render(SEED + 1, 0, 4096, 0, LAST) / np.float32(4096)
    sums, counts, _, passes = _adaptive_render(ctx, tau, lo, step, hi)
    image = sums / counts[..., None].astype(np.float32)
    err = rel_mse(image, reference)
    mean_spp = float(counts.mean())
    assert err <= 2 * tau * tau, (err, mean_spp, len(passes))
    assert lo < mean_spp < hi, mean_spp


def test_adaptive_state_errors_and_framebuffer_ownership():
    ctx = _context("scenes/cornell.json", 32, 24, 0, {})
    for args in [(0.0, 4, 4, 16), (-0.1, 4, 4, 16), (float("nan"), 4, 4, 16), (0.1, 1, 4, 16), (0.1, 4, 0, 16), (0.1, 8, 4, 7)]:
        with pytest.raises(PathedError, match="status -1"):
            ctx.adaptive_begin(*args)
    with pytest.raises(PathedError, match="status -3"):
        ctx.adaptive_pass(SEED, 0, LAST)
    with pytest.raises(PathedError, match="status -3"):
        ctx.adaptive_state()
    ctx.adaptive_begin(0.1, 4, 4, 8)
    ctx.adaptive_pass(SEED, 0, LAST)
    with pytest.raises(PathedError, match="status -3"):
        ctx.framebuffer_render(SEED, 0, 1, 0, LAST)
    with pytest.raises(PathedError, match="status -3"):
        ctx.framebuffer_render_checkpoints(SEED, 0, 2, 0, LAST, [1])
    while ctx.adaptive_pass(SEED, 0, LAST)[0]:
        pass
    assert ctx.adaptive_pass(SEED, 0, LAST) == (0, ctx.adaptive_state()[0].max())  # done: a no-op
    ctx.framebuffer_clear()  # the framebuffer is a plain one again
    ctx.framebuffer_render(SEED, 0, 2, 0, LAST)
    assert np.array_equal(ctx.framebuffer_gather([], divisor=1), ctx.render(SEED, 0, 2, 0, LAST))
    with pytest.raises(PathedError, match="status -3"):
        ctx.adaptive_pass(SEED, 0, LAST)


def read_exr_float_channel(path):
    """the one FLOAT channel of an uncompressed scanline EXR (adaptive-spp.exr), top scanline first"""
    b = open(path, "rb").read()
    assert b[:4] == b"\x76\x2f\x31\x01"
    pos, attrs = 8, {}
    while b[pos] != 0:
        end = b.index(b"\0", pos); name = b[pos:end].decode(); pos = end + 1
        end = b.index(b"\0", pos); pos = end + 1
        size = int.from_bytes(b[pos:pos + 4], "little"); pos += 4
        attrs[name] = b[pos:pos + size]; pos += size
    pos += 1
    x0, y0, x1, y1 = np.frombuffer(attrs["dataWindow"], np.int32)
    w, h = int(x1 - x0 + 1), int(y1 - y0 + 1)
    channel = attrs["channels"]
    assert channel.count(b"\0") >= 1 and channel.split(b"\0")[0] == b"Y" and len(channel) == 2 + 16 + 1  # one channel
    assert int.from_bytes(channel[2:6], "little") == 2 and attrs["compression"] == b"\0"  # FLOAT, uncompressed
    image = np.zeros((h, w), np.float32)
    for offset in np.frombuffer(b, np.uint64, h, pos):
        o = int(offset)
        y = int.from_bytes(b[o:o + 4], "little", signed=True)
        image[y - y0] = np.frombuffer(b, np.float32, w, o + 8)
    return image


def _run_job(tmp_path, **over):
    job = {"spp": 32, "integrator": "PathTracer", "scene": "scenes/cornell-glass.json", "startBounce": 0, "lastBounce": 10,
           "output_directory": str(tmp_path / "out"), "output_name": "final", "showUI": False, "force": True, "width": 48, "height": 40,
           "adaptive_threshold": 0.1, "adaptive_min_spp": 4, "adaptive_step_spp": 4}
    job.update(over)
    os.makedirs(str(tmp_path), exist_ok=True)
    path = str(tmp_path / "job.json")
    json.dump(job, open(path, "w"))
    r = subprocess.run([os.path.join(PKG_DIR, "pathed"), path, "--root", REPO_ROOT], capture_output=True, text=True)
    return job, r


def test_cli_adaptive_job(tmp_path):
    job, r = _run_job(tmp_path)
    assert r.returncode == 0, r.stdout + r.stderr
    out = str(tmp_path / "out")
    ends = [int(m) for m in re.findall(r"adaptive pass \d+: (\d+)/32 spp, \d+ pixels active", r.stdout)]
    assert ends and ends[0] == 4 and ends == sorted(ends) and "sample: " not in r.stdout
    for n in (4, 8, 16, 32):  # the checkpoints are the passes that end at a power of two
        assert os.path.exists(os.path.join(out, "auto-%05dspp.exr" % n)) == (n in ends), n
    for name in ("final.exr", "auto.exr", "adaptive-spp.exr", "report.json"):
        assert os.path.exists(os.path.join(out, name)), name
    counts = read_exr_float_channel(os.path.join(out, "adaptive-spp.exr"))[::-1].astype(np.uint32)  # row 0 = bottom
    assert counts.shape == (40, 48) and counts.max() == ends[-1] and set(np.unique(counts)) <= set(ends)
    result = json.loads(r.stdout.split("PATHED_RESULT ")[1].splitlines()[0])
    assert result["samples"] == int(counts.sum())
    ctx = load_scene(job["scene"], job["width"], job["height"])
    want = np.zeros((40, 48, 3), np.float32)
    for n in np.unique(counts):
        mask = counts == n
        want[mask] = (ctx.render(0x5EED, 0, int(n), 0, 10) / np.float32(n))[mask]
    assert np.array_equal(read_exr(os.path.join(out, "final.exr"))[..., :3], half_like_reference(want[::-1]))
