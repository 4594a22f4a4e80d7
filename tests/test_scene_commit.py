"""ptc_replicate copies what ptc_commit built: the replica inherits the source's options, reports the source's BVH facts and
walks the same BVH (placements included) in ptc_count_traversal."""
import ctypes
import os

import numpy as np
import pytest

from pathed_b200 import create_context, load_scene
from pathed_b200._binding import GATHER_MOMENTS, REPO_ROOT, _ptr
from test_instancing import _rays, _two_level_scene

pytestmark = pytest.mark.gpu

BVH_FACTS = ("bvh_nodes", "bvh_triangles", "bvh_depth", "bvh_ploc_iterations", "bvh_builder")


def _last_device():
    import torch
    return torch.cuda.device_count() - 1


def _need(scene):
    if not os.path.exists(os.path.join(REPO_ROOT, scene)):
        pytest.skip(scene + " not generated")


def _count_traversal(ctx, rays):
    inner, tris = ctypes.c_uint64(), ctypes.c_uint64()
    ctx._call("count_traversal", _ptr(rays), ctypes.c_uint32(len(rays)), ctypes.byref(inner), ctypes.byref(tris))
    return inner.value, tris.value


def test_replica_inherits_the_sources_options():
    """framebuffer_moments set on the source holds on the replica from its first framebuffer_clear, as on a fresh context"""
    _need("scenes/cornell-glass.json")
    a = load_scene("scenes/cornell-glass.json", 48, 40, options={"framebuffer_moments": 1})
    b = a.replicate(_last_device())
    for ctx in (a, b):
        ctx.framebuffer_clear()
        ctx.framebuffer_render(0x5EED, 0, 8, 0, 10)
    want = a.framebuffer_gather([], 1, GATHER_MOMENTS)
    assert want.max() > 0 and np.array_equal(b.framebuffer_gather([], 1, GATHER_MOMENTS), want)


@pytest.mark.parametrize("builder", [1, 0])
@pytest.mark.parametrize("scene", ["scenes/cornell-glass.json", "two-level"])
def test_replica_reports_the_sources_bvh_and_traverses_it_alike(scene, builder):
    if scene == "two-level":
        a = create_context(0)
        a.set_option("bvh_builder", builder)
        _two_level_scene(a)
        rays = _rays(4096, 11)
    else:
        _need(scene)
        a = load_scene(scene, 48, 40, options={"bvh_builder": builder})
        rc = np.stack(np.meshgrid(np.arange(40, dtype=np.float32) + 0.5, np.arange(48, dtype=np.float32) + 0.5, indexing="ij"), -1)
        rays = a.camera_rays(rc.reshape(-1, 2))
    b = a.replicate(_last_device())
    sa, sb = a.stats(), b.stats()
    assert sa.bvh_builder == builder and sa.bvh_nodes > 0 and sa.bvh_triangles > 0
    assert [getattr(sb, f) for f in BVH_FACTS] == [getattr(sa, f) for f in BVH_FACTS]
    want = _count_traversal(a, rays)
    assert want[0] > 0 and want[1] > 0 and _count_traversal(b, rays) == want
