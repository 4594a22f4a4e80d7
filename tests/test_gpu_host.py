"""GPU tests (pytest -m gpu) of the C++ host API and the context-owned framebuffer: the `pathed` command-line renderer run on a
job.json like the reference's binary, Scene::testIntersect / testOcclusion, and the peer-memory reduce + resolve."""
import json
import os
import subprocess

import numpy as np
import pytest

from parity import half_like_reference

from pathed_b200 import SceneFile, load_scene, read_exr, scene_query
from pathed_b200._binding import PKG_DIR, REPO_ROOT, rays_array

pytestmark = pytest.mark.gpu


def _run_job(tmp_path, **over):
    job = {"spp": 8, "integrator": "PathTracer", "scene": "scenes/cornell.json", "startBounce": 0, "lastBounce": 10,
           "output_directory": str(tmp_path / "out"), "output_name": "final", "showUI": False, "force": True, "width": 48, "height": 40}
    job.update(over)
    os.makedirs(str(tmp_path), exist_ok=True)
    path = str(tmp_path / "job.json")
    json.dump(job, open(path, "w"))
    r = subprocess.run([os.path.join(PKG_DIR, "pathed"), path, "--root", REPO_ROOT], capture_output=True, text=True)
    return job, r


def test_cli_renders_a_job_like_the_reference_binary(tmp_path):
    job, r = _run_job(tmp_path)
    assert r.returncode == 0, r.stdout + r.stderr
    out = str(tmp_path / "out")
    # src/integrator.cpp:87-92 checkpoints at every power of two; app/main.cpp:115 saves <output_name>.exr at the end
    for name in ["report.json", "auto.exr", "final.exr"] + ["auto-%05dspp.exr" % s for s in (1, 2, 4, 8)]:
        assert os.path.exists(os.path.join(out, name)), name
    assert json.load(open(os.path.join(out, "report.json")))["scene"] == job["scene"]
    assert "sample: 8/8" in r.stdout and "PATHED_RESULT" in r.stdout
    ctx = load_scene(job["scene"], job["width"], job["height"])
    assert r.stdout.count("sample: ") == 1  # ONE wave of 8 spp: the checkpoints inside it are snapshots, not wave ends
    for spp in (1, 2, 4, 8):
        want = half_like_reference((ctx.render(0x5EED, 0, spp, 0, 10) / np.float32(spp))[::-1])
        got = read_exr(os.path.join(out, "auto-%05dspp.exr" % spp))[..., :3]
        assert np.array_equal(got, want), spp  # same Philox streams, same accumulation order: bit-exact after HALF
    assert np.array_equal(read_exr(os.path.join(out, "final.exr")), read_exr(os.path.join(out, "auto.exr")))


def test_cli_wave_size_and_seed_keys(tmp_path):
    _, a = _run_job(tmp_path, spp=6, wave_spp=1, seed=7)
    assert a.returncode == 0, a.stdout
    assert [l for l in a.stdout.splitlines() if "sample: " in l][-1].split("sample: ")[1].startswith("6/6")
    assert a.stdout.count("sample: ") == 6  # one wave per spp, like the reference
    got = read_exr(str(tmp_path / "out" / "final.exr"))[..., :3]
    ctx = load_scene("scenes/cornell.json", 48, 40)
    want = half_like_reference((ctx.render(7, 0, 6, 0, 10) / np.float32(6))[::-1])
    assert np.array_equal(got, want)


def test_cli_rejects_what_the_reference_rejects(tmp_path):
    _, r = _run_job(tmp_path, integrator="BDPT")
    assert r.returncode == 1 and "Unimplemented" in r.stdout
    _, r = _run_job(tmp_path, scene="scenes/does-not-exist.json")
    assert r.returncode == 1


def test_cli_volume_path_tracer_job(tmp_path):
    """SURVEY N3: job.json with "integrator": "VolumePathTracer" on the medium scene = ptc_set_integrator + ptc_render"""
    from pathed_b200._binding import VOLUME_PATH_TRACER
    job, r = _run_job(tmp_path, integrator="VolumePathTracer", scene="scenes/cornell-medium.json", spp=4)
    assert r.returncode == 0, r.stdout + r.stderr
    got = read_exr(str(tmp_path / "out" / "final.exr"))[..., :3]
    ctx = load_scene(job["scene"], job["width"], job["height"], integrator=VOLUME_PATH_TRACER)
    want = half_like_reference((ctx.render(0x5EED, 0, 4, 0, 10) / np.float32(4))[::-1])
    assert np.array_equal(got, want)
    assert want.mean() > 0.01


def test_scene_queries_through_the_host_api():
    sf = SceneFile("scenes/cornell.json", 32, 32)
    ctx = sf.feed(__import__("pathed_b200").create_context(0))
    cam = ctx.camera_rays(np.array([[16.0, 16.0], [3.0, 29.0]], np.float32))
    full = ctx.intersect_full(cam)
    for i in range(2):
        q = scene_query(sf, cam["origin"][i], cam["direction"][i], 0.5 * float(full["t"][i]))
        assert q["hit"] and q["t"] == full["t"][i] and q["material"] == int(full["material"][i])
        assert np.array_equal(np.float32(q["point"]), full["point"][i]) and np.array_equal(np.float32(q["normal"]), full["normal"][i])
        assert not q["occluded"]  # the segment ends half way to the first surface
        assert scene_query(sf, cam["origin"][i], cam["direction"][i], 2.0 * float(full["t"][i]))["occluded"]
    miss = scene_query(sf, (0, 1, 10), (0, 0, 1), 5.0)
    assert not miss["hit"] and not miss["occluded"]


def test_framebuffer_gather_sums_contexts_and_resolves():
    """two contexts (same device here; peer devices on a multi-GPU box) each render half of the samples into their own HBM
    framebuffer; one kernel sums them and divides by the sample count"""
    a = load_scene("scenes/cornell-glass.json", 40, 40)
    b = load_scene("scenes/cornell-glass.json", 40, 40)
    a.framebuffer_clear(); b.framebuffer_clear()
    a.framebuffer_render(5, 0, 4, 0, 10)
    b.framebuffer_render(5, 4, 4, 0, 10)
    got = a.framebuffer_gather([b], divisor=8)
    want = load_scene("scenes/cornell-glass.json", 40, 40).render(5, 0, 8, 0, 10) / np.float32(8)
    assert np.allclose(got, want, rtol=2e-6, atol=1e-7)
    sums = a.framebuffer_gather([], divisor=1)
    assert np.array_equal(sums, load_scene("scenes/cornell-glass.json", 40, 40).render(5, 0, 4, 0, 10))
    a.framebuffer_clear()
    assert not a.framebuffer_gather([], divisor=1).any()


@pytest.mark.parametrize("lanes", [1, 3])
def test_checkpoint_snapshots_equal_renders_that_stopped_there(lanes):
    """ptc_framebuffer_render_checkpoints: the K7 resolve keeps the running sums after 1, 2, 4, 8 of a 12-sample wave -- the very
    floats of renders that ended there (src/integrator.cpp:87-92 without ending waves at the checkpoints); with the samples split
    over two contexts a checkpoint is the sum of both contexts' snapshots, also where it lies outside a context's block.
    lanes = 3: the wave is traced as three part-waves of 4 samples (ptc_set_option("lanes")), the checkpoints fall inside and between them"""
    def fresh():
        ctx = load_scene("scenes/cornell-glass.json", 40, 40)
        ctx.set_option("lanes", lanes)
        return ctx
    counts = [1, 2, 4, 8]
    a = fresh()
    a.framebuffer_clear()
    a.framebuffer_render_checkpoints(5, 0, 12, 0, 10, counts)
    tickets = [a.framebuffer_gather_begin([], snapshot=i, divisor=1) for i in range(len(counts))] + [a.framebuffer_gather_begin([], divisor=1)]
    images = [a.framebuffer_gather_end(t) for t in tickets]  # all in flight at once, collected afterwards
    for c, image in zip(counts + [12], images):
        assert np.array_equal(image, fresh().render(5, 0, c, 0, 10)), c
    # a second wave on top: snapshots before / inside / after the wave's samples
    a.framebuffer_render_checkpoints(5, 12, 6, 0, 10, [8, 16, 32])
    got = [a.framebuffer_gather_end(a.framebuffer_gather_begin([], snapshot=i, divisor=1)) for i in range(3)]
    assert np.array_equal(got[0], images[-1]) and np.array_equal(got[1], fresh().render(5, 0, 16, 0, 10)) and np.array_equal(got[2], fresh().render(5, 0, 18, 0, 10))
    # two contexts, blocks [0, 6) and [6, 12): checkpoint 4 lies before b's block, 8 inside it, 16 behind both
    a, b = fresh(), fresh()
    a.framebuffer_clear(); b.framebuffer_clear()
    a.framebuffer_render_checkpoints(5, 0, 6, 0, 10, [4, 8, 16])
    b.framebuffer_render_checkpoints(5, 6, 6, 0, 10, [4, 8, 16])
    four, eight, sixteen = [a.framebuffer_gather_end(a.framebuffer_gather_begin([b], snapshot=i, divisor=1)) for i in range(3)]
    assert np.array_equal(four, fresh().render(5, 0, 4, 0, 10))
    assert np.allclose(eight, fresh().render(5, 0, 8, 0, 10), rtol=2e-6, atol=1e-7)
    assert np.array_equal(sixteen, a.framebuffer_gather([b], divisor=1))
    b.framebuffer_render_checkpoints(5, 12, 0, 0, 10, [4])  # no samples in this wave: the snapshot is the framebuffer as it stands
    assert np.array_equal(b.framebuffer_gather_end(b.framebuffer_gather_begin([], snapshot=0, divisor=1)), b.framebuffer_gather([], divisor=1))


@pytest.mark.parametrize("scene", ["scenes/cornell-glass.json", "scenes/textured.json", "test_scenes/environment_map_sampling.json", "scenes/instanced.json", "scenes/cornell-medium.json"])
def test_replicated_context_renders_what_the_original_renders(scene):
    """ptc_replicate (SURVEY 8(e): build once, broadcast): the copy -- on the last device of the box, which is the same device on a
    one-GPU box -- owns rebased copies of BVH, shading records, textures, environment tables and media, and renders bit-identically"""
    import torch
    from pathed_b200._binding import VOLUME_PATH_TRACER
    if not os.path.exists(os.path.join(REPO_ROOT, scene)):
        pytest.skip(scene + " not generated")
    volume = "medium" in scene
    a = load_scene(scene, 48, 40, integrator=VOLUME_PATH_TRACER if volume else 0)
    b = a.replicate(torch.cuda.device_count() - 1)
    want = a.render(3, 0, 4, 0, 6)
    a.close()  # the copy does not depend on the original's memory
    assert b.num_lights() > 0 and np.array_equal(b.render(3, 0, 4, 0, 6), want) and want.mean() > 0
    cam = b.camera_rays(np.array([[20.0, 24.0]], np.float32))
    assert b.intersect_full(cam)["hit"][0] == 1


def test_multi_gpu_job_matches_single_gpu(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    _, one = _run_job(tmp_path / "a", spp=8)
    _, two = _run_job(tmp_path / "b", spp=8, gpus=2)
    assert one.returncode == 0 and two.returncode == 0, two.stdout
    x = read_exr(str(tmp_path / "a" / "out" / "final.exr")); y = read_exr(str(tmp_path / "b" / "out" / "final.exr"))
    assert np.allclose(x, y, rtol=2e-3, atol=1e-4)  # HALF output of sums that differ in the last fp32 bit


REF_CUDA = os.path.join(REPO_ROOT, "oracle", "_ref", "pathed_ref_cuda")
REF_CUDA_GOLDEN = os.path.join(REPO_ROOT, "tests", "golden", "reference_binding.json")


def image_digest(a):
    """sha256 of an image's fp32 bytes: the comparisons below are bit for bit, so a digest stores as much as the image"""
    import hashlib
    return hashlib.sha256(np.ascontiguousarray(a, np.float32).tobytes()).hexdigest()


@pytest.mark.parametrize("scene,integrator,width,height", [
    ("scenes/cornell.json", "PathTracer", 48, 40), ("scenes/cornell-glass.json", "PathTracer", 48, 40), ("scenes/mis-pbrt.json", "PathTracer", 60, 40),
    ("scenes/teapot.json", "PathTracer", 64, 36), ("scenes/textured.json", "PathTracer", 48, 40), ("scenes/instanced.json", "PathTracer", 48, 36),
    ("test_scenes/environment_map_sampling.json", "PathTracer", 48, 36), ("scenes/cornell-medium.json", "VolumePathTracer", 40, 40)])
def test_reference_tree_bound_to_the_cuda_library_renders_the_same_image(tmp_path, scene, integrator, width, height):
    """INTEGRATION.md as a binary: the UNMODIFIED reference (its Job, scene / OBJ parsers, Image, Integrator::run) linked against the
    Embree-API shim + libpathed_cuda (oracle/ref/cuda_main.cpp) and the repository's own host layer must feed the same geometry,
    materials, lights and camera -- the final images are equal bit for bit (same Philox streams), and so are the checkpoint files.
    The reference tree is not part of this repository, so tests/golden/reference_binding.json keeps the SHA-256 digests of what the
    binding writes for these jobs (Image::m_raw, final.exr, auto-00004spp.exr); the repository's render and `pathed` are held to them
    everywhere, and to the binary itself where oracle/_ref/pathed_ref_cuda is built."""
    if not os.path.exists(os.path.join(REPO_ROOT, scene)):
        pytest.skip(scene + " not generated")
    job, ours = _run_job(tmp_path / "ours", scene=scene, integrator=integrator, width=width, height=height, spp=4, wave_spp=1)
    assert ours.returncode == 0, ours.stdout + ours.stderr
    ctx = load_scene(scene, width, height, integrator=1 if integrator == "VolumePathTracer" else 0)
    want = (ctx.render(0x5EED, 0, 4, 0, 10) / np.float32(4))[::-1]         # the repository's host layer + the same library
    stored = json.load(open(REF_CUDA_GOLDEN))["%s %s %dx%d" % (scene, integrator, width, height)]
    assert want.mean() > 0 and image_digest(want) == stored["image"], (float(want.mean()), stored["mean"])
    for name in ("final.exr", "auto-00004spp.exr"):
        assert image_digest(read_exr(str(tmp_path / "ours" / "out" / name))) == stored[name], name
    if not os.path.exists(REF_CUDA):
        return
    job["output_directory"] = str(tmp_path / "ref" / "out")
    os.makedirs(str(tmp_path / "ref"), exist_ok=True)
    path = str(tmp_path / "ref" / "job.json")
    json.dump(job, open(path, "w"))
    raw = str(tmp_path / "ref" / "image.f32")
    r = subprocess.run([REF_CUDA, "--root", REPO_ROOT, path, "--raw", raw], capture_output=True, text=True)
    assert r.returncode == 0 and "REF_CUDA_RESULT" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
    got = np.fromfile(raw, np.float32).reshape(height, width, 3)          # Image::m_raw of the reference's Image, top scanline first
    assert np.array_equal(got, want)
    for name in ("final.exr", "auto-00004spp.exr"):                         # the reference's tinyexr writer against this repository's
        a = read_exr(str(tmp_path / "ref" / "out" / name)); b = read_exr(str(tmp_path / "ours" / "out" / name))
        assert np.array_equal(a, b), name
