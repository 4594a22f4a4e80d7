"""CPU tests of the C++ host API (pathed_b200/host/pathed.hpp): Job, BounceController, Image behave like the reference's
(/root/reference/include/job.h, src/job.cpp, src/bounce_controller.cpp, src/image.cpp)."""
import json
import os
import subprocess

import numpy as np
import pytest

from parity import half_like_reference

from pathed_b200 import PathedError, bounce_controller, image_save, job_describe, read_exr
from pathed_b200._binding import PKG_DIR, REPO_ROOT


def _job(tmp_path, **over):
    job = {"spp": 4, "integrator": "PathTracer", "scene": "scenes/cornell.json", "startBounce": 0, "lastBounce": 10,
           "output_directory": str(tmp_path / "out"), "output_name": "final", "showUI": False, "force": True, "width": 32, "height": 24}
    job.update(over)
    for k in [k for k, v in job.items() if v is None]:
        del job[k]
    path = str(tmp_path / "job.json")
    json.dump(job, open(path, "w"))
    return path


def test_job_accessors_and_defaults(tmp_path):
    d = job_describe(_job(tmp_path))
    assert (d["width"], d["height"], d["spp"], d["startBounce"], d["lastBounce"]) == (32, 24, 4, 0, 10)
    assert d["output_directory"].endswith("/out/") and d["output_name"] == "final" and d["scene"] == "scenes/cornell.json"
    assert d["showUI"] is False and d["force"] is True and d["integrator_status"] == "ok"
    assert (d["gpus"], d["seed"], d["wave_spp"]) == (1, 0x5EED, 64)
    # spp <= 0 means "until stopped" (include/job.h:27-33); force defaults to false when absent
    d = job_describe(_job(tmp_path, spp=0, force=None, gpus=4, seed=99, lastBounce=-1))
    assert d["spp"] == 9999999 and d["force"] is False and d["gpus"] == 4 and d["seed"] == 99 and d["lastBounce"] == -1


def test_job_unknown_integrator_is_unimplemented(tmp_path):
    # src/job.cpp:96: throw "Unimplemented"; the research integrators are outside the accelerated path
    for name in ("BDPT", "LightTracer", "NoSuchThing"):
        assert job_describe(_job(tmp_path, integrator=name))["integrator_status"] == "Unimplemented"
    # SURVEY N3: "VolumePathTracer" (src/job.cpp:71-72) is built
    assert job_describe(_job(tmp_path, integrator="VolumePathTracer"))["integrator_status"] == "ok"


def test_job_missing_keys_raise(tmp_path):
    with pytest.raises(PathedError):
        job_describe(_job(tmp_path, startBounce=None))
    with pytest.raises(PathedError):
        job_describe(str(tmp_path / "nope.json"))


def test_bounce_controller_windows():
    # src/bounce_controller.cpp:14-25
    assert bounce_controller(0, 10, 0)[:2] == (True, False)
    assert bounce_controller(0, 10, 10)[:2] == (True, False)
    assert bounce_controller(0, 10, 11)[:2] == (False, True)
    assert bounce_controller(2, 3, 1)[:2] == (False, False)
    assert bounce_controller(2, -1, 1000)[:2] == (True, False)
    assert bounce_controller(2, 3, 0)[2] == (1, 2)
    assert bounce_controller(0, 0, 0)[2] == (0, 0)
    assert bounce_controller(0, -1, 0)[2] == (0, -1)


def test_image_layout_exr_and_preview(tmp_path):
    """src/image.cpp: raw stored flipped (row 0 = bottom scanline), EXR = HALF B,G,R, checkpoint name <stem>-%05dspp.exr,
    preview = min(v^(1/2.2), 1) * 255 truncated"""
    rng = np.random.default_rng(3)
    rgb = (rng.random((6, 5, 3)) * 2).astype(np.float32)
    rgb[0, 0] = (0.25, 0.5, 4.0)
    out = str(tmp_path)
    preview = image_save(out, "auto", rgb, 8, "preview.bmp")
    for name in ("auto.exr", "auto-00008spp.exr"):
        exr = read_exr(os.path.join(out, name))
        assert exr.shape == (6, 5, 4)
        want = half_like_reference(rgb[::-1])  # top scanline first, HALF as the reference rounds it
        assert np.array_equal(exr[..., :3], want)
    want8 = (np.minimum(np.power(rgb, np.float32(1 / 2.2), dtype=np.float32), 1.0) * 255).astype(np.uint8)
    assert np.abs(preview.astype(int) - want8.astype(int)).max() <= 1
    assert tuple(preview[0, 0]) == (int(0.25 ** (1 / 2.2) * 255), int(0.5 ** (1 / 2.2) * 255), 255)
    bmp = open(os.path.join(out, "preview.bmp"), "rb").read()
    assert bmp[:2] == b"BM" and len(bmp) == 54 + 6 * 16  # 5 px * 3 B padded to 16 B per row
    # stb's BMP puts data row 0 at the top of the picture = the LAST stored row; stored order is B,G,R
    last_row = bmp[54 + 5 * 16:54 + 5 * 16 + 3]
    assert tuple(last_row) == (preview[0, 0, 2], preview[0, 0, 1], preview[0, 0, 0])


def test_cli_fails_loudly_without_gpu(tmp_path):
    # an empty CUDA_VISIBLE_DEVICES hides every device, so the run sees no GPU on a GPU machine as well
    r = subprocess.run([os.path.join(PKG_DIR, "pathed"), _job(tmp_path), "--root", REPO_ROOT], capture_output=True, text=True,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 1 and "Failed to create device" in r.stdout
    assert os.path.exists(str(tmp_path / "out" / "report.json"))  # Job::init ran first, as in app/main.cpp:66-73


def _scene(tmp_path, models, media=None):
    scene = {"sensor": {"lookAt": {"origin": ["0", "0", "5"], "target": ["0", "0", "0"], "up": ["0", "1", "0"]}, "fov": "40"},
             "models": models}
    if media is not None:
        scene["media"] = media
    path = str(tmp_path / "scene.json")
    json.dump(scene, open(path, "w"))
    return path


def test_parser_media_and_internal_medium(tmp_path):
    """parseMedia + `internal_medium` + the passthrough bsdf (src/scene_parser.cpp:202-229, :324-343, :503-514, :593-594) through
    the C++ host parser, fed to the CPU checker: a Passthrough sphere that encloses a medium is skipped by Scene::testOcclusion and
    leaves a volume event; the same sphere with an UNKNOWN medium name gets no medium (the reference's map default-constructs a
    null pointer) and is an ordinary occluder; a later medium with the same name replaces the earlier one."""
    from oracle_binding import oracle_context
    from pathed_b200 import SceneFile
    from pathed_b200._binding import PASSTHROUGH, rays_array
    media = [{"name": "gas", "type": "homogeneous", "sigma_t": ["9", "9", "9"]},
             {"name": "gas", "type": "homogeneous", "sigma_t": ["0.5", "0.5", "0.5"], "sigma_s": ["0.25", "0.25", "0.25"]}]
    ball = lambda medium: {"type": "sphere", "center": ["0", "0", "0"], "radius": "1", "internal_medium": medium, "bsdf": {"type": "passthrough"}}
    rays = rays_array([[0, 0, 5]], [[0, 0, -1]])
    far = np.array([20.0], np.float32)

    sf = SceneFile(_scene(tmp_path, [ball("gas")], media), 8, 8, root=str(tmp_path))
    assert sf.counts() == {"geometries": 1, "triangles": 0, "spheres": 1, "materials": 1} and sf.material(0).type == PASSTHROUGH
    o = sf.feed(oracle_context())
    assert o.occluded(rays, far)[0] == 0                      # the container is not an occluder ...
    occ, ne, et, em = o.occluded_volumetric(rays, far)
    assert occ[0] == 0 and ne[0] == 1 and abs(et[0, 0] - 4.0) < 1e-5 and em[0, 0] == 0   # ... it leaves one event (near side only)
    assert abs(float(o.intersect_full(rays)["t"][0]) - 4.0) < 1e-5                      # Scene::testIntersect does hit it

    o = SceneFile(_scene(tmp_path, [ball("no-such-medium")], media), 8, 8, root=str(tmp_path)).feed(oracle_context())
    assert o.occluded(rays, far)[0] == 1                      # no medium: the filter lets the hit stand
    assert o.occluded_volumetric(rays, far)[1][0] == 0

    with pytest.raises(PathedError):
        SceneFile(_scene(tmp_path, [ball("fog")], [{"name": "fog", "type": "heterogeneous", "filename": "x.vol", "albedo": "1"}]), 8, 8, root=str(tmp_path))


# ---- EXR reader (environment maps): every scanline codec the reference reads through tinyexr for its own assets
EXR_DIR = os.path.join(REPO_ROOT, "tests", "golden", "exr")


@pytest.mark.parametrize("codec", ["none", "rle", "zips", "zip", "piz"])
@pytest.mark.parametrize("kind", ["f32", "f16"])
def test_exr_reader_decodes_every_codec(codec, kind):
    """files written by OpenEXR itself (cv2.imwrite, tests/golden/exr); PIZ is what the reference's test_scenes/1_pixel_test.exr uses"""
    want = np.load(os.path.join(EXR_DIR, "pixels_rgb_f32.npy"))
    if kind == "f16":
        want = half_like_reference(want)
    got = read_exr(os.path.join(EXR_DIR, "%s_%s.exr" % (codec, kind)))
    assert got.shape == want.shape[:2] + (4,)
    assert np.array_equal(got[..., :3], want) and (got[..., 3] == 1).all()


def test_exr_reader_reads_the_reference_one_pixel_fixture():
    """known answer (SURVEY F2) of the reference's test_scenes/1_pixel_test.exr: 1000 x 500 fp32 PIZ, exactly one non-zero texel = 10000
    at row 239, column 753.  tests/golden/exr/one_pixel_piz_f32.exr is that image written by OpenEXR itself (cv2.imwrite, PIZ, FLOAT)."""
    img = read_exr(os.path.join(EXR_DIR, "one_pixel_piz_f32.exr"))
    assert img.shape == (500, 1000, 4)
    lit = np.argwhere(img[..., :3].sum(-1) != 0)
    assert lit.tolist() == [[239, 753]] and img[239, 753, :3].tolist() == [10000.0, 10000.0, 10000.0]


def test_exr_reader_rejects_malformed_blocks(tmp_path):
    """a block header is untrusted input: scanline outside the data window, block sizes beyond the file or the scanlines, negative
    attribute sizes and truncated files raise instead of writing out of bounds"""
    import struct
    data = bytearray(open(os.path.join(EXR_DIR, "none_f32.exr"), "rb").read())
    # locate the offset table: it follows the header's terminating zero byte; block 0 starts at its first entry
    pos = 8
    while data[pos] != 0:
        pos = data.index(0, pos) + 1           # attribute name
        pos = data.index(0, pos) + 1           # attribute type
        size = struct.unpack_from("<i", data, pos)[0]
        pos += 4 + size
    table = pos + 1
    block0 = struct.unpack_from("<Q", data, table)[0]

    def expect_failure(mutated, what):
        path = str(tmp_path / (what + ".exr"))
        open(path, "wb").write(bytes(mutated))
        with pytest.raises(PathedError):
            read_exr(path)

    bad = bytearray(data); struct.pack_into("<i", bad, block0, -30000000); expect_failure(bad, "negative_y")
    bad = bytearray(data); struct.pack_into("<i", bad, block0, 1 << 20); expect_failure(bad, "y_beyond_window")
    bad = bytearray(data); struct.pack_into("<i", bad, block0 + 4, 1 << 30); expect_failure(bad, "huge_block")
    bad = bytearray(data); struct.pack_into("<i", bad, block0 + 4, -5); expect_failure(bad, "negative_block")
    bad = bytearray(data); struct.pack_into("<Q", bad, table, 1 << 40); expect_failure(bad, "offset_outside")
    expect_failure(data[:block0 + 40], "truncated")
    zipped = bytearray(open(os.path.join(EXR_DIR, "zip_f32.exr"), "rb").read())
    expect_failure(zipped[:len(zipped) - 100], "truncated_zip")
    piz = bytearray(open(os.path.join(EXR_DIR, "piz_f32.exr"), "rb").read())
    for k in range(len(piz) - 400, len(piz) - 300):
        piz[k] ^= 0x5A
    path = str(tmp_path / "corrupt_piz.exr")
    open(path, "wb").write(bytes(piz))
    try:  # a corrupted Huffman stream either fails a check or decodes to other pixels; it must not crash
        read_exr(path)
    except PathedError:
        pass


def test_exr_half_rounding_is_the_reference_writers(tmp_path):
    """the reference writes HALF through tinyexr's float_to_half_full (vendor/tinyexr.h:7164-7199): ties round UP (1 + 2^-11 -> 1 + 2^-10,
    where round-to-nearest-even gives 1), float denormals flush to zero, the carry may run into the exponent"""
    rgb = np.zeros((4, 8, 3), np.float32)
    special = [1.0 + 2.0 ** -11, 1.0 + 3 * 2.0 ** -11, 2.0 - 2.0 ** -11, 65519.0, 65520.0, 1e-40, 6e-8, 3e-8, 5.96e-8, 6.1e-5, 0.1, 0.3333333, 1e6, 2.0 ** -14 * (1 + 2.0 ** -11)]
    flat = rgb.reshape(-1)
    flat[:len(special)] = special
    flat[len(special):] = np.random.default_rng(3).random(flat.size - len(special), np.float32) * 4
    image_save(str(tmp_path) + "/", "tie", rgb, 1)
    got = read_exr(str(tmp_path / "tie.exr"))[..., :3][::-1]
    assert np.array_equal(got, half_like_reference(rgb))
    assert got.reshape(-1)[0] == np.float32(1.0 + 2.0 ** -10) and np.float32(special[0]).astype(np.float16) == np.float16(1.0)
    assert got.reshape(-1)[2] == 2.0 and np.isinf(got.reshape(-1)[4]) and got.reshape(-1)[5] == 0.0
