"""CPU tests of the boundary: the product libraries load without a GPU and export every symbol the header declares;
without a CUDA device the library refuses to create a context (no CPU fallback)."""
import ctypes
import os
import re

import numpy as np
import pytest

from pathed_b200._binding import REPO_ROOT, PathedError, SceneFile, cuda_lib, host_lib


def _declared(prefix):
    text = open(os.path.join(REPO_ROOT, "include", "pathed_cuda.h")).read()
    return sorted(set(re.findall(r"\b(%s[a-z_]+)\s*\(" % prefix, text)))


def test_cuda_library_exports_every_declared_symbol():
    lib = cuda_lib()
    names = _declared("ptc_")
    assert len(names) >= 25
    for name in names:
        assert hasattr(lib, name), name


def test_no_cpu_fallback():
    # in a process of its own with an empty CUDA_VISIBLE_DEVICES, which hides every device, so it sees no GPU on a GPU machine as well
    import subprocess
    import sys
    code = ("import sys\nsys.path.insert(0, %r)\nfrom pathed_b200._binding import PathedError, create_context\n"
            "try:\n    create_context(0)\nexcept PathedError:\n    print('refused')\n" % REPO_ROOT)
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout.strip() == "refused", r.stdout + r.stderr


def test_product_does_not_link_the_oracle():
    import subprocess
    for lib in ("libpathed_cuda.so", "libpathed_host.so"):
        out = subprocess.run(["ldd", os.path.join(REPO_ROOT, "pathed_b200", lib)], capture_output=True, text=True).stdout
        assert "oracle" not in out and "embree" not in out


def test_scene_parser_reads_every_config():
    host_lib()
    expect = {"scenes/cornell.json": (1, 36, 0), "scenes/cornell-glass.json": (3, 1112, 0), "scenes/mis-pbrt.json": (10, 12, 5),
              "scenes/teapot.json": (3, None, 0), "scenes/dragon.json": (2, None, 0)}
    for scene, (geoms, tris, spheres) in expect.items():
        c = SceneFile(scene, 32, 32).counts()
        assert c["geometries"] == geoms and c["spheres"] == spheres
        if tris is not None:
            assert c["triangles"] == tris


def test_scene_parser_errors():
    import json, tempfile
    with tempfile.TemporaryDirectory() as tmp:
        bad = {"sensor": {"lookAt": {"origin": ["0", "0", "1"], "target": ["0", "0", "0"], "up": ["0", "1", "0"]}, "fov": "30"},
               "models": [{"type": "sphere", "center": ["0", "0", "0"], "radius": "1", "bsdf": {"type": "velvet"}}]}
        path = os.path.join(tmp, "bad.json")
        json.dump(bad, open(path, "w"))
        with pytest.raises(PathedError, match="Unimplemented material"):
            SceneFile("bad.json", 8, 8, root=tmp)
        with pytest.raises(PathedError):
            SceneFile("missing.json", 8, 8, root=tmp)


def test_obj_material_resolution_and_cornell_lights():
    s = SceneFile("scenes/cornell.json", 8, 8)
    pos, idx, mat = s.geometry(0)
    emit = [tuple(s.material(m).emit) for m in mat]
    lights = [i for i, e in enumerate(emit) if e != (0.0, 0.0, 0.0)]
    assert lights == [34, 35] and emit[34] == (17.0, 12.0, 4.0)  # the two light triangles are registered last
    # negative (relative) face indices and the duplicated quads of the data set
    assert pos.shape == (72, 3) and idx.shape == (36, 3)


def test_exr_round_trip(tmp_path):
    lib = host_lib()
    img = np.random.default_rng(0).random((5, 7, 3)).astype(np.float32) * 100
    path = str(tmp_path / "a.exr").encode()
    assert lib.pth_exr_write_rgb_f32(path, 7, 5, img.ctypes.data_as(ctypes.c_void_p)) == 0
    w, h = ctypes.c_int(), ctypes.c_int()
    out = np.zeros((5, 7, 4), np.float32)
    assert lib.pth_exr_read_rgba(path, out.ctypes.data_as(ctypes.c_void_p), 35, ctypes.byref(w), ctypes.byref(h)) == 0
    assert (w.value, h.value) == (7, 5)
    assert np.array_equal(out[..., :3], img) and (out[..., 3] == 1).all()
