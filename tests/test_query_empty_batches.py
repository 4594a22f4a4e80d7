"""GPU tests (pytest -m gpu) of the host-buffer queries at an empty batch: with n = 0 every query entry point needs no array at all
(null pointers), still runs its kernel on one element of device scratch, and returns PTC_OK."""
import ctypes

import numpy as np
import pytest

from pathed_b200 import load_scene
from pathed_b200._binding import PATH_TRACER, VOLUME_PATH_TRACER

pytestmark = pytest.mark.gpu

u32, zero = ctypes.c_uint32, ctypes.c_uint32(0)

# entry point (without the ptc_ prefix) -> its arguments after the context, for a batch of zero elements
EMPTY = {
    "intersect": (None, zero, None),
    "intersect_instanced": (None, zero, None, None),
    "intersect_full": (None, zero, None),
    "occluded": (None, None, zero, None),
    "occluded_volumetric": (None, None, zero, None, None, None, None),
    "intersect_volumetric": (None, zero, None, None, None, None),
    "camera_rays": (None, zero, None),
    "philox4x32_10": (None, None, zero, None),
    "uniforms": (ctypes.c_uint64(7), None, zero, u32(4), None),
    "bsdf_eval": (zero, None, None, zero, None, None),
    "bsdf_sample": (zero, None, None, zero, None, None, None),
    "light_sample": (None, None, zero, None),
    "light_pdf": (None, zero, None),
    "environment_radiance": (None, zero, None),
    "radiance_replay": (None, None, u32(8), zero, ctypes.c_int(0), ctypes.c_int(-1), None),
}


@pytest.mark.parametrize("scene, integrator", [("scenes/cornell.json", PATH_TRACER), ("scenes/cornell-medium.json", VOLUME_PATH_TRACER)],
                         ids=["PathTracer", "VolumePathTracer"])
def test_every_query_accepts_an_empty_batch(scene, integrator):
    ctx = load_scene(scene, 16, 12, integrator=integrator)
    before = ctx.stats().kernel_launches
    for name, args in EMPTY.items():
        ctx._call(name, *args)  # raises on any status but PTC_OK
    assert ctx.stats().kernel_launches == before + len(EMPTY)  # one kernel per query, on one element of scratch
    # the guide buffers' batch is the samples: none leaves the caller's sums as they are
    aovs = {"albedo": np.full((12, 16, 3), 0.5, np.float32), "normal": np.full((12, 16, 3), -1.0, np.float32),
            "depth": np.full((12, 16), 2.0, np.float32), "hits": np.full((12, 16), 3, np.uint32)}
    kept = {k: v.copy() for k, v in aovs.items()}
    ctx.render_aovs(seed=7, first_sample=0, n_spp=0, aovs=aovs)
    for k in aovs:
        assert np.array_equal(aovs[k], kept[k]), k
