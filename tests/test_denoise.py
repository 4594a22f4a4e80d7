"""GPU tests of denoising (DESIGN §10): the first-hit guide buffers of ptc_render_aovs rebuilt from the probe entry points, the
second moments of the framebuffer renders and their gather, the filter of ptc_denoise against the numpy restatement below, its
effect on the error, and the `pathed` job key "denoise"."""
import ctypes
import json
import os
import subprocess

import numpy as np
import pytest

from parity import half_like_reference, rel_mse

from pathed_b200 import load_scene, read_exr
from pathed_b200._binding import (GATHER_MOMENTS, LAMBERTIAN, OREN_NAYAR, PKG_DIR, PLASTIC, REPO_ROOT, VOLUME_PATH_TRACER, DenoiseDesc,
                                  DenoiseInput, PathedError, SceneFile, load_image_rgb8)

pytestmark = pytest.mark.gpu

SEED, LAST = 13, 10
f32 = np.float32


def _context(scene, width, height, integrator=0, options=None):
    if not os.path.exists(os.path.join(REPO_ROOT, scene)):
        pytest.skip(scene + " not generated")
    ctx = load_scene(scene, width, height, integrator=integrator)
    for name, value in (options or {}).items():
        ctx.set_option(name, value)
    return ctx


# ------------------------------------------------------------------------------------------------ guide buffers
def _textures(scene):
    """texture id -> texels (h, w, 3) uint8: the parser registers each file once, in the order the scene names them"""
    paths = []

    def walk(node):
        if isinstance(node, dict):
            for key, value in node.items():
                if key == "texture" and isinstance(value, str) and value not in paths:
                    paths.append(value)
                walk(value)
        elif isinstance(node, list):
            for value in node:
                walk(value)
    walk(json.load(open(os.path.join(REPO_ROOT, scene))))
    return [load_image_rgb8(os.path.join(REPO_ROOT, p)) for p in paths]


# pow(c / 255, 2.2) in fp32, rounded from fp64 (the library tabulates it with the host's powf)
GAMMA = np.power((np.arange(256, dtype=np.float32) / f32(255)).astype(np.float64), np.float64(f32(2.2))).astype(np.float32)


def _round_half_away(x):
    t = np.trunc(x)
    return (t + np.where(np.abs(x - t) >= 0.5, np.sign(x), 0)).astype(np.int64)


def _albedo(desc, textures, uv):
    """lambertAlbedo (shading.cuh) for one material over hits with texture coordinates uv [n, 2], fp32"""
    n = len(uv)
    if desc.type not in (LAMBERTIAN, OREN_NAYAR, PLASTIC):
        return np.ones((n, 3), np.float32)
    u, v = uv[:, 0], uv[:, 1]
    if desc.albedo_kind == 2:
        tex = textures[desc.texture]
        th, tw = tex.shape[:2]
        uu = u - np.floor(u).astype(np.int32).astype(np.float32)
        vv = f32(1) - (v - np.floor(v).astype(np.int32).astype(np.float32))
        x = _round_half_away(uu * f32(tw - 1)); y = _round_half_away(vv * f32(th - 1))
        return GAMMA[tex[y, x]]
    if desc.albedo_kind == 1:
        ui = np.floor(u * f32(desc.checker_resolution[0])).astype(np.int64)
        vi = np.floor(v * f32(desc.checker_resolution[1])).astype(np.int64)
        same = np.fmod(ui, 2) == np.fmod(vi, 2)
        return np.where(same[:, None], np.array(desc.checker_on, np.float32), np.array(desc.checker_off, np.float32))
    return np.broadcast_to(np.array(desc.diffuse, np.float32), (n, 3)).copy()


def _guide_restatement(ctx, scene_file, textures, seed, first, n_spp):
    h, w = ctx.height, ctx.width
    pixels = np.arange(h * w, dtype=np.uint32)
    row, col = (pixels // w).astype(np.float32), (pixels % w).astype(np.float32)
    albedo = np.zeros((h * w, 3), np.float32); normal = np.zeros((h * w, 3), np.float32)
    depth = np.zeros(h * w, np.float32); hits = np.zeros(h * w, np.uint32)
    materials = {}
    for s in range(first, first + n_spp):
        streams = np.stack([pixels, np.full_like(pixels, s), np.zeros_like(pixels)], 1)
        u = ctx.uniforms(seed, streams, 2)
        jx, jy = u[:, 0] - f32(0.5), u[:, 1] - f32(0.5)
        isect = ctx.intersect_full(ctx.camera_rays(np.stack([row + jy, col + jx], 1)))
        hit = isect["hit"] != 0
        a = np.zeros((h * w, 3), np.float32)
        for m in np.unique(isect["material"][hit]):
            sel = hit & (isect["material"] == m)
            if m not in materials:
                materials[m] = scene_file.material(int(m))
            a[sel] = _albedo(materials[m], textures, isect["uv"][sel])
        albedo = albedo + a
        normal = normal + np.where(hit[:, None], isect["shading_normal"], f32(0))
        depth = depth + np.where(hit, isect["t"], f32(0))
        hits = hits + hit.astype(np.uint32)
    return {"albedo": albedo.reshape(h, w, 3), "normal": normal.reshape(h, w, 3), "depth": depth.reshape(h, w), "hits": hits.reshape(h, w)}


GUIDE_SCENES = {
    "cornell": ("scenes/cornell.json", 0),
    "textured": ("scenes/textured.json", 0),
    "mis": ("scenes/mis-pbrt.json", 0),
    "instanced": ("scenes/instanced.json", 0),
    "cornell_medium_pt": ("scenes/cornell-medium.json", 0),
    "cornell_medium_vpt": ("scenes/cornell-medium.json", VOLUME_PATH_TRACER),
}


@pytest.mark.parametrize("name", sorted(GUIDE_SCENES))
def test_guide_buffers_equal_the_first_hits_rebuilt_from_the_probes(name):
    scene, integrator = GUIDE_SCENES[name]
    W, H, N = 24, 16, 8
    ctx = _context(scene, W, H, integrator)
    got = ctx.render_aovs(SEED, 0, N)
    want = _guide_restatement(ctx, SceneFile(scene, W, H), _textures(scene), SEED, 0, N)
    assert got["hits"].sum() > 0
    for key in ("normal", "depth", "hits"):
        assert np.array_equal(got[key], want[key]), (name, key)
    if name == "textured":  # numpy's pow may differ by one ulp from the table the library computed at commit time
        diff = np.abs(got["albedo"].astype(np.float64) - want["albedo"])
        assert (diff <= N * np.spacing(np.maximum(np.abs(want["albedo"]), f32(1e-30)))).all()
        assert np.mean(got["albedo"] == want["albedo"]) > 0.99
    else:
        assert np.array_equal(got["albedo"], want["albedo"]), name
    # a call adds to what it is given: two halves give the bytes of the whole
    halves = ctx.render_aovs(SEED, N, N, ctx.render_aovs(SEED, 0, N))
    whole = ctx.render_aovs(SEED, 0, 2 * N)
    for key in whole:
        assert np.array_equal(halves[key], whole[key]), (name, key)


# ------------------------------------------------------------------------------------------------ second moments
SETTINGS = {"lanes1": {"lanes": 1}, "default": {}, "small_waves": {"paths_per_wave": 3000}}


@pytest.mark.parametrize("setting", sorted(SETTINGS))
def test_framebuffer_moments_leave_the_sums_alone_and_equal_the_squares(setting):
    N = 9
    ctx = _context("scenes/cornell-glass.json", 24, 16, 0, SETTINGS[setting])
    ctx.framebuffer_clear()
    ctx.framebuffer_render(SEED, 0, N, 0, LAST)
    plain = ctx.framebuffer_gather([], divisor=1)
    with pytest.raises(PathedError, match="status -3"):
        ctx.framebuffer_gather([], 1, GATHER_MOMENTS)
    ctx.set_option("framebuffer_moments", 1)
    ctx.framebuffer_clear()
    ctx.framebuffer_render(SEED, 0, 4, 0, LAST)
    ctx.framebuffer_render_checkpoints(SEED, 4, N - 4, 0, LAST, [6])
    assert np.array_equal(ctx.framebuffer_gather([], divisor=1), plain)
    moments = ctx.framebuffer_gather([], 1, GATHER_MOMENTS)
    singles = [ctx.render(SEED, s, 1, 0, LAST) for s in range(N)]
    want = np.zeros_like(plain)
    for x in singles:
        want = want + x * x
    assert np.allclose(moments, want, rtol=1e-6, atol=0)
    ctx.framebuffer_clear()  # zeroes the moments too
    assert not ctx.framebuffer_gather([], 1, GATHER_MOMENTS).any()


def test_a_context_without_samples_has_zero_moments_to_gather():
    """a multi-GPU job can leave a GPU without samples in every wave: its moments are the zeros of the clear"""
    a = _context("scenes/cornell-glass.json", 24, 16, 0, {"framebuffer_moments": 1})
    b = _context("scenes/cornell-glass.json", 24, 16, 0, {"framebuffer_moments": 1})
    for ctx in (a, b):
        ctx.framebuffer_clear()
    a.framebuffer_render_checkpoints(SEED, 0, 6, 0, LAST, [4])
    b.framebuffer_render_checkpoints(SEED, 6, 0, 0, LAST, [4])
    alone = a.framebuffer_gather([], 1, GATHER_MOMENTS)
    assert alone.any() and np.array_equal(a.framebuffer_gather([b], 1, GATHER_MOMENTS), alone)
    assert not b.framebuffer_gather([], 1, GATHER_MOMENTS).any()


def test_moments_that_miss_samples_are_refused():
    ctx = _context("scenes/cornell-glass.json", 24, 16, 0, {"framebuffer_moments": 1})
    ctx.framebuffer_clear()
    ctx.framebuffer_render(SEED, 0, 3, 0, LAST)
    ctx.set_option("framebuffer_moments", 0)  # switched off: later renders would not add to them
    with pytest.raises(PathedError, match="status -3"):
        ctx.framebuffer_gather([], 1, GATHER_MOMENTS)
    ctx.framebuffer_render(SEED, 3, 2, 0, LAST)
    ctx.set_option("framebuffer_moments", 1)  # back on in the middle of an accumulation: samples 3, 4 are missing
    ctx.framebuffer_render(SEED, 5, 2, 0, LAST)
    with pytest.raises(PathedError, match="status -3"):
        ctx.framebuffer_gather([], 1, GATHER_MOMENTS)
    ctx.framebuffer_clear()  # complete again from here
    ctx.framebuffer_render(SEED, 0, 2, 0, LAST)
    want = ctx.render(SEED, 0, 1, 0, LAST) ** 2 + ctx.render(SEED, 1, 1, 0, LAST) ** 2
    assert np.allclose(ctx.framebuffer_gather([], 1, GATHER_MOMENTS), want, rtol=1e-6, atol=0)


def test_gather_of_moments_sums_contexts_and_reads_adaptive_renders():
    a = _context("scenes/cornell-glass.json", 24, 16, 0, {"framebuffer_moments": 1})
    b = _context("scenes/cornell-glass.json", 24, 16, 0, {"framebuffer_moments": 1})
    for ctx, first in ((a, 0), (b, 5)):
        ctx.framebuffer_clear()
        ctx.framebuffer_render(SEED, first, 5, 0, LAST)
    ma, mb = a.framebuffer_gather([], 1, GATHER_MOMENTS), b.framebuffer_gather([], 1, GATHER_MOMENTS)
    assert np.array_equal(a.framebuffer_gather([b], 1, GATHER_MOMENTS), ma + mb)
    c = _context("scenes/cornell-glass.json", 24, 16)
    c.adaptive_begin(0.1, 4, 4, 12)
    while c.adaptive_pass(SEED, 0, LAST)[0]:
        pass
    assert np.array_equal(c.framebuffer_gather([], 1, GATHER_MOMENTS), c.adaptive_state()[1])
    c.framebuffer_clear()  # a plain framebuffer without the option: no moments
    with pytest.raises(PathedError, match="status -3"):
        c.framebuffer_gather([], 1, GATHER_MOMENTS)


# ------------------------------------------------------------------------------------------------ the filter, restated
K3 = [f32(0.25), f32(0.5), f32(0.25)]
K5 = [f32(1 / 16), f32(0.25), f32(0.375), f32(0.25), f32(1 / 16)]


def _shift(a, oy, ox, fill):
    """b[y, x] = a[y + oy, x + ox] where that is inside the image, else fill; and the mask of the inside"""
    h, w = a.shape[:2]
    b = np.full_like(a, fill)
    inside = np.zeros((h, w), bool)
    ys, yd = (slice(oy, h), slice(0, h - oy)) if oy >= 0 else (slice(0, h + oy), slice(-oy, h))
    xs, xd = (slice(ox, w), slice(0, w - ox)) if ox >= 0 else (slice(0, w + ox), slice(-ox, w))
    if yd.stop > yd.start and xd.stop > xd.start:
        b[yd, xd] = a[ys, xs]
        inside[yd, xd] = True
    return b, inside


def _lum(c):
    return (f32(0.2126) * c[..., 0] + f32(0.7152) * c[..., 1]) + f32(0.0722) * c[..., 2]


def denoise_restatement(S, M, counts, aovs, aov_spp, iterations=5, sigma_l=4.0, sigma_n=128.0, sigma_z=1.0, sigma_a=0.1, eps=1e-6):
    """DESIGN §10 in numpy, fp32, every operation rounded on its own in the kernel's order"""
    sigma_l, sigma_n, sigma_z, sigma_a, eps = (f32(x) for x in (sigma_l, sigma_n, sigma_z, sigma_a, eps))
    with np.errstate(all="ignore"):
        n = np.asarray(counts, np.float32)
        if n.ndim == 0:
            n = np.full(S.shape[:2], n, np.float32)
        c = S / n[..., None]
        var = (M - n[..., None] * (c * c)) / (n[..., None] - f32(1))
        var = np.where(var < 0, f32(0), var)
        v = ((var[..., 0] + var[..., 1]) + var[..., 2]) / (f32(3) * n)
        a = aovs["albedo"] / f32(aov_spp)
        N = aovs["normal"]
        len2 = (N[..., 0] * N[..., 0] + N[..., 1] * N[..., 1]) + N[..., 2] * N[..., 2]
        length = np.where(len2 > 0, np.sqrt(len2), f32(0))
        N = np.where(length[..., None] > 0, N / length[..., None], f32(0))
        z = aovs["depth"] / np.maximum(aovs["hits"], 1).astype(np.float32)
        zeroN = (N == 0).all(-1)
        for i in range(iterations):
            h = 2 ** i
            finite = np.isfinite(c).all(-1) & np.isfinite(v)
            vs = np.zeros_like(v); ks = np.zeros_like(v)
            for dy in (-1, 0, 1):
                for dx in (-1, 0, 1):
                    vq, inside = _shift(v, dy, dx, 0)
                    ok = inside & _shift(finite, dy, dx, False)[0]
                    k = K3[dx + 1] * K3[dy + 1]
                    vs = np.where(ok, vs + k * vq, vs); ks = np.where(ok, ks + k, ks)
            vt = vs / ks
            lp = _lum(c)
            denom_l = sigma_l * np.sqrt(vt) + eps
            step_z = sigma_z * f32(h)
            sw = np.zeros_like(v); sc = np.zeros_like(c); sv = np.zeros_like(v)
            for dy in (-2, -1, 0, 1, 2):
                for dx in (-2, -1, 0, 1, 2):
                    cq, inside = _shift(c, h * dy, h * dx, 0)
                    vq = _shift(v, h * dy, h * dx, 0)[0]
                    ok = inside & _shift(finite, h * dy, h * dx, False)[0]
                    aq, zq = _shift(a, h * dy, h * dx, 0)[0], _shift(z, h * dy, h * dx, 0)[0]
                    Nq, zeroNq = _shift(N, h * dy, h * dx, 0)[0], _shift(zeroN, h * dy, h * dx, True)[0]
                    dot = (N[..., 0] * Nq[..., 0] + N[..., 1] * Nq[..., 1]) + N[..., 2] * Nq[..., 2]
                    g = np.power(np.maximum(f32(0), dot), sigma_n)
                    g = np.where(zeroN | zeroNq, np.where(zeroN & zeroNq, f32(1), f32(0)), g)
                    dl = np.abs(lp - _lum(cq)) / denom_l
                    da = ((np.abs(a[..., 0] - aq[..., 0]) + np.abs(a[..., 1] - aq[..., 1])) + np.abs(a[..., 2] - aq[..., 2])) / sigma_a
                    dz = np.abs(z - zq) / (step_z * np.maximum(np.maximum(z, zq), eps))
                    w = ((K5[dx + 2] * K5[dy + 2]) * np.exp(((-dl) - da) - dz)) * g
                    sw = np.where(ok, sw + w, sw)
                    sc = np.where(ok[..., None], sc + w[..., None] * cq, sc)
                    sv = np.where(ok, sv + (w * w) * vq, sv)
            c = np.where(finite[..., None], sc / sw[..., None], c)
            v = np.where(finite, sv / (sw * sw), v)
    return c


def _synthetic(seed, h=28, w=40, uniform_spp=None):
    rng = np.random.default_rng(seed)
    counts = np.full((h, w), uniform_spp, np.uint32) if uniform_spp else rng.integers(2, 40, (h, w)).astype(np.uint32)
    n = counts.astype(np.float32)[..., None]
    mean = (rng.random((h, w, 3)) * 2).astype(np.float32)
    mean[:, : w // 2] *= f32(0.2)  # two regions of different brightness
    S = (mean * n).astype(np.float32)
    M = (S * mean * f32(1.3) + rng.random((h, w, 3)).astype(np.float32) * n * f32(0.1)).astype(np.float32)
    S[3, 5, 1] = np.nan; M[10, 20, 0] = np.inf; S[h - 1, w - 1, 2] = np.inf  # non-finite pixels
    aov_spp = 8
    hits = rng.integers(0, aov_spp + 1, (h, w)).astype(np.uint32)
    hits[:, -6:] = 0  # a region of misses
    frac = hits.astype(np.float32)[..., None]
    dirs = rng.normal(size=(h, w, 3)).astype(np.float32)
    dirs[h // 2:] = np.array([0, 1, 0], np.float32) + f32(0.05) * dirs[h // 2:]
    aovs = {"albedo": (rng.random((h, w, 3)).astype(np.float32) * frac).astype(np.float32),
            "normal": (dirs * frac).astype(np.float32),
            "depth": ((f32(2) + rng.random((h, w)).astype(np.float32)) * frac[..., 0]).astype(np.float32),
            "hits": hits}
    return S, M, counts, aovs, aov_spp


def _close(got, want):
    scale = np.maximum(np.abs(want), 1e-6)
    both = ~np.isfinite(want)
    assert np.array_equal(np.isfinite(got), np.isfinite(want))
    assert np.array_equal(got[both], want[both], equal_nan=True)
    err = np.abs(got[~both].astype(np.float64) - want[~both]) / scale[~both]
    assert err.max() <= 1e-5, err.max()


def _synthetic_context(h=28, w=40):
    return _context("scenes/cornell.json", w, h)  # the filter takes only the image size from the context


@pytest.mark.parametrize("params", [{}, {"iterations": 3, "sigma_l": 1.0, "sigma_n": 16.0, "sigma_z": 0.5, "sigma_a": 0.5},
                                    {"iterations": 10}])
@pytest.mark.parametrize("per_pixel", [True, False])
def test_filter_equals_its_restatement_on_synthetic_inputs(params, per_pixel):
    S, M, counts, aovs, aov_spp = _synthetic(5, uniform_spp=None if per_pixel else 7)
    ctx = _synthetic_context()
    arg = counts if per_pixel else 7
    got = ctx.denoise(S, M, arg, aovs, aov_spp, **params)
    _close(got, denoise_restatement(S, M, arg, aovs, aov_spp, **params))
    assert np.array_equal(got.view(np.uint32), ctx.denoise(S, M, arg, aovs, aov_spp, **params).view(np.uint32))  # same bytes
    raw = S / (counts[..., None].astype(np.float32) if per_pixel else f32(7))
    nonfinite = ~np.isfinite(raw).all(-1) | ~np.isfinite(M).all(-1)  # (a finite S with an infinite M has an infinite variance)
    assert np.array_equal(got[nonfinite], raw[nonfinite], equal_nan=True)  # non-finite pixels pass through
    assert np.isfinite(got[~nonfinite]).all()


def test_zero_iterations_and_a_constant_image():
    S, M, counts, aovs, aov_spp = _synthetic(6)
    ctx = _synthetic_context()
    assert np.array_equal(ctx.denoise(S, M, counts, aovs, aov_spp, iterations=0), S / counts[..., None].astype(np.float32), equal_nan=True)
    n = counts[..., None].astype(np.float32)
    colour = np.array([0.5, 0.25, 0.125], np.float32)
    S = (colour * n).astype(np.float32); M = (colour * colour * n).astype(np.float32)  # zero variance, exactly
    out = ctx.denoise(S, M, counts, aovs, aov_spp)
    assert np.array_equal(out, np.broadcast_to(colour, out.shape))


def test_filter_on_a_real_render():
    ctx = _context("scenes/cornell-glass.json", 64, 64, 0, {"framebuffer_moments": 1})
    ctx.framebuffer_clear()
    ctx.framebuffer_render(SEED, 0, 16, 0, LAST)
    S, M = ctx.framebuffer_gather([], divisor=1), ctx.framebuffer_gather([], 1, GATHER_MOMENTS)
    aovs = ctx.render_aovs(SEED, 0, 8)
    _close(ctx.denoise(S, M, 16, aovs, 8), denoise_restatement(S, M, 16, aovs, 8))


def test_bad_descriptors_and_inputs_raise():
    S, M, counts, aovs, aov_spp = _synthetic(7)
    ctx = _synthetic_context()
    for bad in ({"iterations": 11}, {"sigma_l": 0.0}, {"sigma_z": -1.0}, {"sigma_a": float("nan")}, {"eps": 0.0}, {"sigma_n": -1.0},
                {"sigma_l": float("inf")}):
        with pytest.raises(PathedError, match="status -1"):
            ctx.denoise(S, M, counts, aovs, aov_spp, **bad)
    with pytest.raises(TypeError):
        ctx.denoise(S, M, counts, aovs, aov_spp, sigma=1.0)
    with pytest.raises(PathedError, match="status -1"):
        ctx.denoise(S, M, 1, aovs, aov_spp)  # one sample: no variance
    one = counts.copy(); one[4, 4] = 1
    with pytest.raises(PathedError, match="status -1"):
        ctx.denoise(S, M, one, aovs, aov_spp)
    with pytest.raises(PathedError, match="status -1"):
        ctx.denoise(S, M, counts, aovs, 0)
    desc, out = DenoiseDesc(5, 4.0, 128.0, 1.0, 0.1, 1e-6), np.zeros(S.shape, np.float32)
    with pytest.raises(PathedError, match="status -1"):  # no inputs at all
        ctx._call("denoise", ctypes.byref(desc), ctypes.byref(DenoiseInput()), out.ctypes.data_as(ctypes.c_void_p))
    with pytest.raises(PathedError, match="status -1"):
        ctx._call("denoise", None, ctypes.byref(DenoiseInput()), out.ctypes.data_as(ctypes.c_void_p))


# ------------------------------------------------------------------------------------------------ quality
def test_denoising_halves_the_error_of_a_16_spp_render():
    ctx = _context("scenes/cornell-glass.json", 128, 128, 0, {"framebuffer_moments": 1})
    reference = ctx.render(SEED + 1, 0, 4096, 0, LAST) / f32(4096)
    aovs = ctx.render_aovs(SEED, 0, 16)
    ctx.framebuffer_clear()
    ctx.framebuffer_render(SEED, 0, 16, 0, LAST)
    S, M = ctx.framebuffer_gather([], divisor=1), ctx.framebuffer_gather([], 1, GATHER_MOMENTS)
    noisy, denoised = rel_mse(S / f32(16), reference), rel_mse(ctx.denoise(S, M, 16, aovs, 16), reference)
    assert denoised <= 0.5 * noisy, (noisy, denoised)
    ctx.adaptive_begin(0.1, 4, 4, 16)
    while ctx.adaptive_pass(SEED, 0, LAST)[0]:
        pass
    S = ctx.framebuffer_gather([], divisor=1)
    counts, M = ctx.adaptive_state()
    noisy = rel_mse(S / counts[..., None].astype(np.float32), reference)
    denoised = rel_mse(ctx.denoise(S, M, counts, aovs, 16), reference)
    assert denoised <= 0.5 * noisy, (noisy, denoised)


# ------------------------------------------------------------------------------------------------ the job key
def _run_job(tmp_path, **over):
    job = {"spp": 16, "integrator": "PathTracer", "scene": "scenes/cornell-glass.json", "startBounce": 0, "lastBounce": 10,
           "output_directory": str(tmp_path / "out"), "output_name": "final", "showUI": False, "force": True, "width": 48, "height": 40,
           "wave_spp": 5}
    job.update(over)
    os.makedirs(str(tmp_path), exist_ok=True)
    path = str(tmp_path / "job.json")
    json.dump(job, open(path, "w"))
    r = subprocess.run([os.path.join(PKG_DIR, "pathed"), path, "--root", REPO_ROOT], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    return job, str(tmp_path / "out")


def _images(out):
    return {f: open(os.path.join(out, f), "rb").read() for f in os.listdir(out) if f == "final.exr" or f.startswith("auto-")}


def _check_job(tmp_path, expected, **over):
    job, out = _run_job(tmp_path / "denoised", denoise=True, **over)
    _, plain = _run_job(tmp_path / "plain", **over)
    images = _images(out)
    assert images and images == _images(plain)  # denoising adds files and changes none
    assert not os.path.exists(os.path.join(plain, "denoised.exr"))
    got = read_exr(os.path.join(out, "denoised.exr"))[..., :3]
    assert np.array_equal(got, half_like_reference(expected["denoised"][::-1]))
    aov_spp = min(job["spp"], 16)
    assert np.array_equal(read_exr(os.path.join(out, "albedo.exr"))[..., :3], (expected["aovs"]["albedo"] / f32(aov_spp))[::-1])
    assert np.array_equal(read_exr(os.path.join(out, "normal.exr"))[..., :3], (expected["aovs"]["normal"] / f32(aov_spp))[::-1])


def test_cli_denoise_job(tmp_path):
    ctx = _context("scenes/cornell-glass.json", 48, 40, 0, {"framebuffer_moments": 1})
    ctx.framebuffer_clear()
    ctx.framebuffer_render(0x5EED, 0, 16, 0, 10)
    S, M = ctx.framebuffer_gather([], divisor=1), ctx.framebuffer_gather([], 1, GATHER_MOMENTS)
    aovs = ctx.render_aovs(0x5EED, 0, 16)
    _check_job(tmp_path, {"denoised": ctx.denoise(S, M, 16, aovs, 16), "aovs": aovs})


def test_cli_denoise_job_on_two_gpus(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    a = _context("scenes/cornell-glass.json", 48, 40, 0, {"framebuffer_moments": 1})
    b = a.replicate(1)
    b.set_option("framebuffer_moments", 1)
    for ctx in (a, b):
        ctx.framebuffer_clear()
    # the job's split: waves of wave_spp per GPU, each wave cut into two contiguous halves
    for first in range(0, 16, 10):
        end = min(first + 10, 16)
        per = (end - first + 1) // 2
        a.framebuffer_render(0x5EED, first, per, 0, 10)
        b.framebuffer_render(0x5EED, first + per, end - first - per, 0, 10)
    S, M = a.framebuffer_gather([b], divisor=1), a.framebuffer_gather([b], 1, GATHER_MOMENTS)
    aovs = a.render_aovs(0x5EED, 0, 16)
    _check_job(tmp_path, {"denoised": a.denoise(S, M, 16, aovs, 16), "aovs": aovs}, gpus=2)


def test_cli_denoise_adaptive_job(tmp_path):
    ctx = _context("scenes/cornell-glass.json", 48, 40)
    ctx.adaptive_begin(0.1, 4, 4, 32)
    while ctx.adaptive_pass(0x5EED, 0, 10)[0]:
        pass
    S = ctx.framebuffer_gather([], divisor=1)
    counts, M = ctx.adaptive_state()
    aovs = ctx.render_aovs(0x5EED, 0, 16)
    _check_job(tmp_path, {"denoised": ctx.denoise(S, M, counts, aovs, 16), "aovs": aovs}, spp=32, adaptive_threshold=0.1,
               adaptive_min_spp=4, adaptive_step_spp=4)
