"""ctypes bindings of the C ABI (include/pathed_cuda.h) and of the host parsers' C entry points.

`Api(lib, prefix)` wraps any shared library exporting the ABI under a prefix: the product
(`libpathed_cuda.so`, prefix `ptc_`).  Tests reuse the same class for the CPU checker (`orc_`), which
is why the prefix is a parameter; nothing in this package loads the checker.
"""
import ctypes
import os

import numpy as np

c_float_p = ctypes.POINTER(ctypes.c_float)
c_u32_p = ctypes.POINTER(ctypes.c_uint32)
PKG_DIR = os.path.dirname(os.path.abspath(__file__))
REPO_ROOT = os.path.dirname(PKG_DIR)

PTC_INVALID_ID = 0xFFFFFFFF
LAMBERTIAN, OREN_NAYAR, MIRROR, GLASS, MICROFACET, PLASTIC, PASSTHROUGH = range(7)
PATH_TRACER, VOLUME_PATH_TRACER = 0, 1
NO_MEDIUM = 0xFFFFFFFF
MAX_EVENTS = 8
BECKMANN, GGX = 0, 1
GATHER_MOMENTS = -2  # snapshot of framebuffer_gather_begin: the sums of the squared samples


class MaterialDesc(ctypes.Structure):
    _fields_ = [("type", ctypes.c_int32), ("diffuse", ctypes.c_float * 3), ("emit", ctypes.c_float * 3),
                ("sigma", ctypes.c_float), ("ior", ctypes.c_float), ("distribution", ctypes.c_int32),
                ("alpha", ctypes.c_float), ("albedo_kind", ctypes.c_int32), ("checker_on", ctypes.c_float * 3),
                ("checker_off", ctypes.c_float * 3), ("checker_resolution", ctypes.c_float * 2), ("texture", ctypes.c_uint32)]


class AdaptiveDesc(ctypes.Structure):
    _fields_ = [("threshold", ctypes.c_float), ("min_spp", ctypes.c_uint32), ("step_spp", ctypes.c_uint32), ("max_spp", ctypes.c_uint32)]


class DenoiseDesc(ctypes.Structure):
    _fields_ = [("iterations", ctypes.c_uint32), ("sigma_l", ctypes.c_float), ("sigma_n", ctypes.c_float), ("sigma_z", ctypes.c_float),
                ("sigma_a", ctypes.c_float), ("eps", ctypes.c_float)]


DENOISE_DEFAULTS = {"iterations": 5, "sigma_l": 4.0, "sigma_n": 128.0, "sigma_z": 1.0, "sigma_a": 0.1, "eps": 1e-6}  # PTC_DENOISE_DEFAULTS


def _denoise_desc(params):
    unknown = set(params) - set(DENOISE_DEFAULTS)
    if unknown:
        raise TypeError("unknown denoise parameters %s" % sorted(unknown))
    p = dict(DENOISE_DEFAULTS, **params)
    return DenoiseDesc(int(p["iterations"]), *[float(p[k]) for k in ("sigma_l", "sigma_n", "sigma_z", "sigma_a", "eps")])


class DenoiseInput(ctypes.Structure):
    _fields_ = [("sums", ctypes.c_void_p), ("moments", ctypes.c_void_p), ("counts", ctypes.c_void_p), ("spp", ctypes.c_uint32),
                ("albedo_rgb", ctypes.c_void_p), ("normal_xyz", ctypes.c_void_p), ("depth", ctypes.c_void_p), ("hits", ctypes.c_void_p),
                ("aov_spp", ctypes.c_uint32)]


class Stats(ctypes.Structure):
    _fields_ = [(n, ctypes.c_uint64) for n in ("closest_rays", "shadow_rays", "samples", "kernel_launches", "bvh_nodes",
                                               "bvh_triangles", "bvh_bytes", "extend_inner_visits", "extend_triangle_tests",
                                               "shadow_inner_visits", "shadow_triangle_tests", "extend_launches",
                                               "shadow_launches", "shade_launches")] + \
               [(n, ctypes.c_float) for n in ("extend_ms", "shadow_ms", "shade_ms", "other_ms", "last_render_ms", "bvh_build_ms")] + \
               [(n, ctypes.c_uint32) for n in ("bvh_builder", "bvh_depth", "bvh_ploc_iterations")]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


RAY_DTYPE = np.dtype([("origin", np.float32, 3), ("direction", np.float32, 3)])
HIT_DTYPE = np.dtype([("t", np.float32), ("u", np.float32), ("v", np.float32), ("geom_id", np.uint32),
                      ("prim_id", np.uint32), ("ng", np.float32, 3)])
ISECT_DTYPE = np.dtype([("hit", np.int32), ("t", np.float32), ("point", np.float32, 3), ("wo", np.float32, 3),
                        ("normal", np.float32, 3), ("shading_normal", np.float32, 3), ("uv", np.float32, 2),
                        ("material", np.uint32)])
LIGHT_SAMPLE_DTYPE = np.dtype([("point", np.float32, 3), ("normal", np.float32, 3), ("inv_pdf", np.float32),
                               ("measure", np.int32), ("solid_angle_pdf", np.float32), ("emit", np.float32, 3)])
assert RAY_DTYPE.itemsize == 24 and HIT_DTYPE.itemsize == 32 and ISECT_DTYPE.itemsize == 68 and LIGHT_SAMPLE_DTYPE.itemsize == 48


class SceneSink(ctypes.Structure):
    _fields_ = [("ctx", ctypes.c_void_p), ("add_material", ctypes.c_void_p), ("add_triangle_mesh", ctypes.c_void_p),
                ("add_sphere", ctypes.c_void_p), ("set_environment", ctypes.c_void_p), ("set_camera", ctypes.c_void_p),
                ("commit", ctypes.c_void_p), ("add_texture", ctypes.c_void_p), ("add_medium", ctypes.c_void_p),
                ("set_internal_medium", ctypes.c_void_p), ("begin_instance", ctypes.c_void_p), ("end_instance", ctypes.c_void_p),
                ("add_instance", ctypes.c_void_p)]


class PathedError(RuntimeError):
    pass


def _ptr(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def rays_array(origins, directions):
    origins = np.asarray(origins, np.float32).reshape(-1, 3)
    directions = np.asarray(directions, np.float32).reshape(-1, 3)
    rays = np.zeros(len(origins), RAY_DTYPE)
    rays["origin"] = origins
    rays["direction"] = directions
    return rays


class Api:
    """One context of a library exporting the pathed_cuda.h ABI under `prefix`."""

    def __init__(self, lib, prefix, device=0):
        self.lib, self.prefix = lib, prefix
        self.ctx = ctypes.c_void_p()
        fn = self._fn("create")
        fn.restype = ctypes.c_int
        rc = fn(ctypes.c_int(device), ctypes.byref(self.ctx))
        if rc != 0 or not self.ctx:
            raise PathedError("%screate failed with status %d (no CUDA device? the product has no CPU fallback)" % (prefix, rc))
        self._fn("last_error").restype = ctypes.c_char_p
        self.width = self.height = 0

    def _fn(self, name):
        return getattr(self.lib, self.prefix + name)

    def replicate(self, device):
        """ptc_replicate: a committed context copied to another GPU (peer copies of the finished device data, no second build)"""
        other = Api.__new__(Api)
        other.lib, other.prefix, other.ctx = self.lib, self.prefix, ctypes.c_void_p()
        other.width, other.height = self.width, self.height
        self._call("replicate", ctypes.c_int(device), ctypes.byref(other.ctx))
        return other

    def _call(self, name, *args):
        fn = self._fn(name)
        fn.restype = ctypes.c_int
        rc = fn(self.ctx, *args)
        if rc != 0:
            raise PathedError("%s%s: status %d: %s" % (self.prefix, name, rc, self._fn("last_error")(self.ctx).decode()))

    def close(self):
        if self.ctx:
            fn = self._fn("destroy")
            fn.restype = None
            fn(self.ctx)
            self.ctx = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def sink(self):
        addr = lambda name: ctypes.cast(self._fn(name), ctypes.c_void_p).value
        return SceneSink(self.ctx.value, addr("add_material"), addr("add_triangle_mesh"), addr("add_sphere"),
                         addr("set_environment"), addr("set_camera"), addr("commit"), addr("add_texture"), addr("add_medium"),
                         addr("set_internal_medium"), addr("begin_instance"), addr("end_instance"), addr("add_instance"))

    # ---- scene description
    def add_texture(self, rgb):
        """rgb: uint8 array (height, width, 3), row 0 = top of the image (what stbi_load returns)."""
        rgb = np.ascontiguousarray(rgb, np.uint8)
        assert rgb.ndim == 3 and rgb.shape[2] == 3
        out = ctypes.c_uint32()
        self._call("add_texture", _ptr(rgb), ctypes.c_int(rgb.shape[1]), ctypes.c_int(rgb.shape[0]), ctypes.byref(out))
        return out.value

    def add_material(self, desc):
        out = ctypes.c_uint32()
        self._call("add_material", ctypes.byref(desc), ctypes.byref(out))
        return out.value

    def add_medium(self, sigma_t, sigma_s=(0.0, 0.0, 0.0)):
        st = (ctypes.c_float * 3)(*[float(x) for x in sigma_t]); ss = (ctypes.c_float * 3)(*[float(x) for x in sigma_s])
        out = ctypes.c_uint32()
        self._call("add_medium", st, ss, ctypes.byref(out))
        return out.value

    def set_internal_medium(self, geom_id, medium_id):
        self._call("set_internal_medium", ctypes.c_uint32(geom_id), ctypes.c_uint32(medium_id))

    # ---- hierarchical instancing (SURVEY 8(f) N4)
    def begin_instance(self):
        out = ctypes.c_uint32()
        self._call("begin_instance", ctypes.byref(out))
        return out.value

    def end_instance(self):
        self._call("end_instance")

    def add_instance(self, instance_scene, local_to_world):
        """local_to_world: 4x4 (row, column) matrix; passed column-major like rtcSetGeometryTransform takes it"""
        m = np.ascontiguousarray(np.asarray(local_to_world, np.float32).reshape(4, 4).T)
        out = ctypes.c_uint32()
        self._call("add_instance", ctypes.c_uint32(instance_scene), _ptr(m), ctypes.byref(out))
        return out.value

    def intersect_instanced(self, rays):
        hits = np.zeros(len(rays), HIT_DTYPE)
        inst = np.zeros((len(rays), 2), np.uint32)
        self._call("intersect_instanced", _ptr(rays), ctypes.c_uint32(len(rays)), _ptr(hits), _ptr(inst))
        return hits, inst

    def set_integrator(self, integrator):
        self._call("set_integrator", ctypes.c_int(integrator))

    def add_triangle_mesh(self, positions, normals, uvs, indices, material_of_tri):
        positions = np.ascontiguousarray(positions, np.float32).reshape(-1, 3)
        nv = len(positions)
        normals = np.zeros((nv, 3), np.float32) if normals is None else np.ascontiguousarray(normals, np.float32)
        uvs = np.zeros((nv, 2), np.float32) if uvs is None else np.ascontiguousarray(uvs, np.float32)
        indices = np.ascontiguousarray(indices, np.uint32).reshape(-1, 3)
        mats = np.ascontiguousarray(np.broadcast_to(np.asarray(material_of_tri, np.uint32), (len(indices),)))
        out = ctypes.c_uint32()
        self._call("add_triangle_mesh", _ptr(positions), _ptr(normals), _ptr(uvs), ctypes.c_uint32(nv), _ptr(indices),
                   _ptr(mats), ctypes.c_uint32(len(indices)), ctypes.byref(out))
        return out.value

    def add_sphere(self, center, radius, material):
        cr = (ctypes.c_float * 4)(center[0], center[1], center[2], radius)
        out = ctypes.c_uint32()
        self._call("add_sphere", cr, ctypes.c_uint32(material), ctypes.byref(out))
        return out.value

    def set_environment(self, rgba, scale=1.0, map_to_world=None, world_to_map=None):
        rgba = np.ascontiguousarray(rgba, np.float32)
        h, w, _ = rgba.shape
        m = np.ascontiguousarray(np.eye(4) if map_to_world is None else map_to_world, np.float32)
        inv = np.ascontiguousarray(np.linalg.inv(m) if world_to_map is None else world_to_map, np.float32)
        self._call("set_environment", _ptr(rgba), ctypes.c_int(w), ctypes.c_int(h), ctypes.c_float(scale), _ptr(m), _ptr(inv))

    def set_camera(self, origin, target, up, vfov, width, height, flip=False):
        f3 = lambda v: (ctypes.c_float * 3)(*[float(x) for x in v])
        self._call("set_camera", f3(origin), f3(target), f3(up), ctypes.c_float(vfov), ctypes.c_int(width),
                   ctypes.c_int(height), ctypes.c_int(1 if flip else 0))
        self.width, self.height = width, height

    def commit(self):
        self._call("commit")

    # ---- hot path
    def render(self, seed, first_sample, n_spp, start_bounce, last_bounce, accum=None):
        if accum is None:
            accum = np.zeros((self.height, self.width, 3), np.float32)
        assert accum.dtype == np.float32 and accum.flags.c_contiguous and accum.size == 3 * self.width * self.height
        self._call("render", ctypes.c_uint64(seed), ctypes.c_uint32(first_sample), ctypes.c_uint32(n_spp),
                   ctypes.c_int(start_bounce), ctypes.c_int(last_bounce), _ptr(accum))
        return accum

    def render_device(self, seed, first_sample, n_spp, start_bounce, last_bounce, accum_ptr, stream=0):
        self._call("render_device", ctypes.c_uint64(seed), ctypes.c_uint32(first_sample), ctypes.c_uint32(n_spp),
                   ctypes.c_int(start_bounce), ctypes.c_int(last_bounce), ctypes.c_void_p(accum_ptr), ctypes.c_void_p(stream))

    def resolve_device(self, accum_ptr, out_ptr, spp, stream=0):
        self._call("resolve_device", ctypes.c_void_p(accum_ptr), ctypes.c_void_p(out_ptr), ctypes.c_uint32(spp), ctypes.c_void_p(stream))

    # ---- context-owned device framebuffer (Integrator::run's radianceLookup kept in HBM)
    def framebuffer_clear(self):
        self._call("framebuffer_clear")

    def framebuffer_render(self, seed, first_sample, n_spp, start_bounce, last_bounce):
        self._call("framebuffer_render", ctypes.c_uint64(seed), ctypes.c_uint32(first_sample), ctypes.c_uint32(n_spp),
                   ctypes.c_int(start_bounce), ctypes.c_int(last_bounce))

    def framebuffer_gather(self, peers=(), divisor=1, snapshot=-1):
        """snapshot -1: the framebuffers; GATHER_MOMENTS (-2): the second moments (use divisor 1); i >= 0: checkpoint snapshot i"""
        if snapshot != -1:
            return self.framebuffer_gather_end(self.framebuffer_gather_begin(peers, snapshot, divisor))
        out = np.zeros((self.height, self.width, 3), np.float32)
        arr = (ctypes.c_void_p * max(len(peers), 1))(*[p.ctx.value for p in peers])
        self._call("framebuffer_gather", arr, ctypes.c_uint32(len(peers)), ctypes.c_uint32(divisor), _ptr(out))
        return out

    def framebuffer_render_checkpoints(self, seed, first_sample, n_spp, start_bounce, last_bounce, sample_counts):
        counts = np.ascontiguousarray(sample_counts, np.uint32)
        self._call("framebuffer_render_checkpoints", ctypes.c_uint64(seed), ctypes.c_uint32(first_sample), ctypes.c_uint32(n_spp),
                   ctypes.c_int(start_bounce), ctypes.c_int(last_bounce), _ptr(counts), ctypes.c_uint32(len(counts)))

    def framebuffer_gather_begin(self, peers=(), snapshot=-1, divisor=1):
        arr = (ctypes.c_void_p * max(len(peers), 1))(*[p.ctx.value for p in peers])
        ticket = ctypes.c_uint32(0)
        self._call("framebuffer_gather_begin", arr, ctypes.c_uint32(len(peers)), ctypes.c_int(snapshot), ctypes.c_uint32(divisor), ctypes.byref(ticket))
        return ticket.value

    def framebuffer_gather_end(self, ticket):
        out = np.zeros((self.height, self.width, 3), np.float32)
        self._call("framebuffer_gather_end", ctypes.c_uint32(ticket), _ptr(out))
        return out

    # ---- adaptive sampling (ptc_adaptive_*): passes into the context's framebuffer until every pixel meets the relMSE target
    def adaptive_begin(self, threshold, min_spp, step_spp, max_spp):
        desc = AdaptiveDesc(float(threshold), int(min_spp), int(step_spp), int(max_spp))
        self._call("adaptive_begin", ctypes.byref(desc))

    def adaptive_pass(self, seed, start_bounce, last_bounce):
        """one pass; returns (pixels still active, samples per active pixel after the pass)"""
        active, spp = ctypes.c_uint32(), ctypes.c_uint32()
        self._call("adaptive_pass", ctypes.c_uint64(seed), ctypes.c_int(start_bounce), ctypes.c_int(last_bounce), ctypes.byref(active), ctypes.byref(spp))
        return active.value, spp.value

    def adaptive_state(self):
        """(samples per pixel [h, w] uint32, per-channel sums of squared samples [h, w, 3] fp32), row 0 = bottom like the sums"""
        counts = np.zeros((self.height, self.width), np.uint32)
        m2 = np.zeros((self.height, self.width, 3), np.float32)
        self._call("adaptive_state", _ptr(counts), _ptr(m2))
        return counts, m2

    # ---- denoising (ptc_render_aovs, ptc_denoise, ptc_framebuffer_guides, ptc_framebuffer_denoise_begin; DESIGN §10)
    def render_aovs(self, seed, first_sample, n_spp, aovs=None):
        """first-hit guide buffers of samples first_sample .. first_sample + n_spp - 1, added into `aovs` (a dict like the one returned;
        None: zeros): albedo [h, w, 3], normal [h, w, 3], depth [h, w] fp32 sums and hits [h, w] uint32, row 0 = bottom"""
        h, w = self.height, self.width
        if aovs is None:
            aovs = {"albedo": np.zeros((h, w, 3), np.float32), "normal": np.zeros((h, w, 3), np.float32),
                    "depth": np.zeros((h, w), np.float32), "hits": np.zeros((h, w), np.uint32)}
        for name, dtype, size in (("albedo", np.float32, 3 * h * w), ("normal", np.float32, 3 * h * w), ("depth", np.float32, h * w),
                                  ("hits", np.uint32, h * w)):
            a = aovs[name]
            assert a.dtype == dtype and a.flags.c_contiguous and a.size == size, name
        self._call("render_aovs", ctypes.c_uint64(seed), ctypes.c_uint32(first_sample), ctypes.c_uint32(n_spp), _ptr(aovs["albedo"]),
                   _ptr(aovs["normal"]), _ptr(aovs["depth"]), _ptr(aovs["hits"]))
        return aovs

    def denoise(self, sums, moments, counts_or_spp, aovs, aov_spp, **params):
        """ptc_denoise: the denoised mean colour [h, w, 3].  counts_or_spp: per-pixel sample counts [h, w] or one spp for every pixel;
        params: iterations, sigma_l, sigma_n, sigma_z, sigma_a, eps (DENOISE_DEFAULTS for the ones not given)"""
        desc = _denoise_desc(params)
        n = 3 * self.width * self.height
        f32 = lambda a, size: np.ascontiguousarray(a, np.float32).reshape(size)
        keep = {"sums": f32(sums, n), "moments": f32(moments, n), "albedo": f32(aovs["albedo"], n), "normal": f32(aovs["normal"], n),
                "depth": f32(aovs["depth"], n // 3), "hits": np.ascontiguousarray(aovs["hits"], np.uint32).reshape(n // 3)}
        inp = DenoiseInput()
        inp.sums, inp.moments = keep["sums"].ctypes.data, keep["moments"].ctypes.data
        if np.ndim(counts_or_spp) == 0:
            inp.counts, inp.spp = None, int(counts_or_spp)
        else:
            keep["counts"] = np.ascontiguousarray(counts_or_spp, np.uint32).reshape(n // 3)
            inp.counts, inp.spp = keep["counts"].ctypes.data, 0
        inp.albedo_rgb, inp.normal_xyz = keep["albedo"].ctypes.data, keep["normal"].ctypes.data
        inp.depth, inp.hits, inp.aov_spp = keep["depth"].ctypes.data, keep["hits"].ctypes.data, int(aov_spp)
        out = np.zeros((self.height, self.width, 3), np.float32)
        self._call("denoise", ctypes.byref(desc), ctypes.byref(inp), _ptr(out))
        return out

    def framebuffer_guides(self, seed, first_sample, n_spp, fetch=False):
        """ptc_framebuffer_guides: the guides of samples first_sample .. first_sample + n_spp - 1, from zero, kept on the device for
        framebuffer_denoise_begin; fetch=True also returns their sums (a dict like render_aovs's), else None"""
        if not fetch:
            self._call("framebuffer_guides", ctypes.c_uint64(seed), ctypes.c_uint32(first_sample), ctypes.c_uint32(n_spp), None, None, None, None)
            return None
        h, w = self.height, self.width
        aovs = {"albedo": np.zeros((h, w, 3), np.float32), "normal": np.zeros((h, w, 3), np.float32),
                "depth": np.zeros((h, w), np.float32), "hits": np.zeros((h, w), np.uint32)}
        self._call("framebuffer_guides", ctypes.c_uint64(seed), ctypes.c_uint32(first_sample), ctypes.c_uint32(n_spp), _ptr(aovs["albedo"]),
                   _ptr(aovs["normal"]), _ptr(aovs["depth"]), _ptr(aovs["hits"]))
        return aovs

    def framebuffer_denoise_begin(self, peers=(), snapshot=-1, spp=0, **params):
        """ptc_framebuffer_denoise_begin: enqueues the denoise of snapshot `snapshot` (-1: the framebuffers) of this context + peers
        with the guides of framebuffer_guides; spp = the image's samples per pixel (ignored on an adaptive render).  Returns the
        ticket for framebuffer_gather_end.  params as for denoise"""
        desc = _denoise_desc(params)
        arr = (ctypes.c_void_p * max(len(peers), 1))(*[p.ctx.value for p in peers])
        ticket = ctypes.c_uint32(0)
        self._call("framebuffer_denoise_begin", arr, ctypes.c_uint32(len(peers)), ctypes.c_int(snapshot), ctypes.c_uint32(spp),
                   ctypes.byref(desc), ctypes.byref(ticket))
        return ticket.value

    def framebuffer_denoise(self, peers=(), snapshot=-1, spp=0, **params):
        """framebuffer_denoise_begin, then framebuffer_gather_end: the denoised mean colour [h, w, 3]"""
        return self.framebuffer_gather_end(self.framebuffer_denoise_begin(peers, snapshot, spp, **params))

    # ---- random streams (known-answer tests)
    def philox(self, counters, keys):
        counters = np.ascontiguousarray(counters, np.uint32).reshape(-1, 4); keys = np.ascontiguousarray(keys, np.uint32).reshape(-1, 2)
        out = np.zeros_like(counters)
        self._call("philox4x32_10", _ptr(counters), _ptr(keys), ctypes.c_uint32(len(counters)), _ptr(out))
        return out

    def uniforms(self, seed, streams, draws):
        streams = np.ascontiguousarray(streams, np.uint32).reshape(-1, 3)
        out = np.zeros((len(streams), draws), np.float32)
        self._call("uniforms", ctypes.c_uint64(seed), _ptr(streams), ctypes.c_uint32(len(streams)), ctypes.c_uint32(draws), _ptr(out))
        return out

    # ---- queries
    def intersect(self, rays):
        hits = np.zeros(len(rays), HIT_DTYPE)
        self._call("intersect", _ptr(rays), ctypes.c_uint32(len(rays)), _ptr(hits))
        return hits

    def intersect_full(self, rays):
        out = np.zeros(len(rays), ISECT_DTYPE)
        self._call("intersect_full", _ptr(rays), ctypes.c_uint32(len(rays)), _ptr(out))
        return out

    def occluded(self, rays, max_t):
        max_t = np.ascontiguousarray(max_t, np.float32)
        out = np.zeros(len(rays), np.uint8)
        self._call("occluded", _ptr(rays), _ptr(max_t), ctypes.c_uint32(len(rays)), _ptr(out))
        return out

    def occluded_volumetric(self, rays, max_t):
        """Scene::testVolumetricOcclusion: (occluded, n_events, event_t[n, MAX_EVENTS], event_medium[n, MAX_EVENTS])"""
        max_t = np.ascontiguousarray(max_t, np.float32)
        n = len(rays)
        occ = np.zeros(n, np.uint8); ne = np.zeros(n, np.uint32)
        et = np.zeros((n, MAX_EVENTS), np.float32); em = np.zeros((n, MAX_EVENTS), np.uint32)
        self._call("occluded_volumetric", _ptr(rays), _ptr(max_t), ctypes.c_uint32(n), _ptr(occ), _ptr(ne), _ptr(et), _ptr(em))
        return occ, ne, et, em

    def intersect_volumetric(self, rays):
        """Scene::testVolumetricIntersect: (isects, n_events, event_t, event_medium)"""
        n = len(rays)
        out = np.zeros(n, ISECT_DTYPE); ne = np.zeros(n, np.uint32)
        et = np.zeros((n, MAX_EVENTS), np.float32); em = np.zeros((n, MAX_EVENTS), np.uint32)
        self._call("intersect_volumetric", _ptr(rays), ctypes.c_uint32(n), _ptr(out), _ptr(ne), _ptr(et), _ptr(em))
        return out, ne, et, em

    def intersect_device(self, rays_ptr, n, hits_ptr, stream=0):
        self._call("intersect_device", ctypes.c_void_p(rays_ptr), ctypes.c_uint32(n), ctypes.c_void_p(hits_ptr), ctypes.c_void_p(stream))

    def occluded_device(self, rays_ptr, max_t_ptr, n, out_ptr, stream=0):
        self._call("occluded_device", ctypes.c_void_p(rays_ptr), ctypes.c_void_p(max_t_ptr), ctypes.c_uint32(n),
                   ctypes.c_void_p(out_ptr), ctypes.c_void_p(stream))

    def camera_rays(self, row_col):
        row_col = np.ascontiguousarray(row_col, np.float32).reshape(-1, 2)
        rays = np.zeros(len(row_col), RAY_DTYPE)
        self._call("camera_rays", _ptr(row_col), ctypes.c_uint32(len(row_col)), _ptr(rays))
        return rays

    def bsdf_eval(self, material, isects, wi):
        wi = np.ascontiguousarray(wi, np.float32)
        f = np.zeros((len(isects), 3), np.float32)
        pdf = np.zeros(len(isects), np.float32)
        self._call("bsdf_eval", ctypes.c_uint32(material), _ptr(isects), _ptr(wi), ctypes.c_uint32(len(isects)), _ptr(f), _ptr(pdf))
        return f, pdf

    def bsdf_sample(self, material, isects, xi):
        xi = np.ascontiguousarray(xi, np.float32)
        n = len(isects)
        wi = np.zeros((n, 3), np.float32); pdf = np.zeros(n, np.float32); thr = np.zeros((n, 3), np.float32)
        self._call("bsdf_sample", ctypes.c_uint32(material), _ptr(isects), _ptr(xi), ctypes.c_uint32(n), _ptr(wi), _ptr(pdf), _ptr(thr))
        return wi, pdf, thr

    def light_sample(self, ref_points, xi):
        ref_points = np.ascontiguousarray(ref_points, np.float32).reshape(-1, 3)
        xi = np.ascontiguousarray(xi, np.float32)
        out = np.zeros(len(ref_points), LIGHT_SAMPLE_DTYPE)
        self._call("light_sample", _ptr(ref_points), _ptr(xi), ctypes.c_uint32(len(ref_points)), _ptr(out))
        return out

    def light_pdf(self, rays):
        out = np.zeros(len(rays), np.float32)
        self._call("light_pdf", _ptr(rays), ctypes.c_uint32(len(rays)), _ptr(out))
        return out

    def environment_radiance(self, directions):
        directions = np.ascontiguousarray(directions, np.float32).reshape(-1, 3)
        out = np.zeros((len(directions), 3), np.float32)
        self._call("environment_radiance", _ptr(directions), ctypes.c_uint32(len(directions)), _ptr(out))
        return out

    def radiance_replay(self, rays, xi, start_bounce, last_bounce):
        xi = np.ascontiguousarray(xi, np.float32).reshape(len(rays), -1)
        out = np.zeros((len(rays), 3), np.float32)
        self._call("radiance_replay", _ptr(rays), _ptr(xi), ctypes.c_uint32(xi.shape[1]), ctypes.c_uint32(len(rays)),
                   ctypes.c_int(start_bounce), ctypes.c_int(last_bounce), _ptr(out))
        return out

    def num_lights(self):
        out = ctypes.c_uint32()
        self._call("num_lights", ctypes.byref(out))
        return out.value

    def stats(self):
        out = Stats()
        self._call("get_stats", ctypes.byref(out))
        return out

    def wave_counts(self, n=12):
        e = (ctypes.c_uint32 * n)(); s = (ctypes.c_uint32 * n)()
        self._call("get_wave_counts", e, s, ctypes.c_uint32(n))
        return list(e), list(s)

    def reset_stats(self):
        self._call("reset_stats")

    def reserve_paths(self, n_paths):
        self._call("reserve_paths", ctypes.c_uint64(n_paths))

    def set_option(self, name, value):
        self._call("set_option", name.encode(), ctypes.c_int64(value))


_host_lib = None


def host_lib():
    global _host_lib
    if _host_lib is None:
        path = os.path.join(PKG_DIR, "libpathed_host.so")
        if not os.path.exists(path):
            raise PathedError("libpathed_host.so is not built; run `python -c 'import __graft_entry__ as g; g.build()'`")
        _host_lib = ctypes.CDLL(path)
    return _host_lib


class SceneFile:
    """A scene JSON parsed by the C++ host layer (pathed_b200/host/scene_parser.cpp)."""

    def __init__(self, scene_json, width, height, root=REPO_ROOT):
        lib = host_lib()
        self.handle = ctypes.c_void_p()
        err = ctypes.create_string_buffer(512)
        rc = lib.pth_scene_load(scene_json.encode(), root.encode(), ctypes.c_int(width), ctypes.c_int(height),
                                ctypes.byref(self.handle), err, ctypes.c_int(512))
        if rc != 0:
            raise PathedError("parseScene(%s): %s" % (scene_json, err.value.decode()))
        self.width, self.height = width, height

    def feed(self, api):
        sink = api.sink()
        lib = host_lib()
        lib.pth_scene_feed.restype = ctypes.c_int
        rc = lib.pth_scene_feed(self.handle, ctypes.byref(sink))
        if rc != 0:
            raise PathedError("feeding scene failed: status %d: %s" % (rc, api._fn("last_error")(api.ctx).decode()))
        api.width, api.height = self.width, self.height
        return api

    def counts(self):
        g, t, s, m = (ctypes.c_uint32() for _ in range(4))
        host_lib().pth_scene_counts(self.handle, ctypes.byref(g), ctypes.byref(t), ctypes.byref(s), ctypes.byref(m))
        return {"geometries": g.value, "triangles": t.value, "spheres": s.value, "materials": m.value}

    def geometry(self, geom):
        pos, idx, mat = ctypes.POINTER(ctypes.c_float)(), ctypes.POINTER(ctypes.c_uint32)(), ctypes.POINTER(ctypes.c_uint32)()
        nv, nt = ctypes.c_uint32(), ctypes.c_uint32()
        rc = host_lib().pth_scene_geometry(self.handle, ctypes.c_uint32(geom), ctypes.byref(pos), ctypes.byref(nv),
                                           ctypes.byref(idx), ctypes.byref(mat), ctypes.byref(nt))
        if rc != 0:
            return None
        return (np.ctypeslib.as_array(pos, (nv.value, 3)).copy(), np.ctypeslib.as_array(idx, (nt.value, 3)).copy(),
                np.ctypeslib.as_array(mat, (nt.value,)).copy())

    def material(self, i):
        d = MaterialDesc()
        if host_lib().pth_scene_material(self.handle, ctypes.c_uint32(i), ctypes.byref(d)) != 0:
            raise IndexError(i)
        return d

    def close(self):
        if self.handle:
            host_lib().pth_scene_free(self.handle)
            self.handle = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def load_image_rgb8(path):
    """The C++ host layer's Texture::load decode (pathed_b200/host/image_loader.cpp): uint8 array (height, width, 3)."""
    lib = host_lib()
    w, h = ctypes.c_int(), ctypes.c_int()
    err = ctypes.create_string_buffer(512)
    lib.pth_image_load_rgb8.restype = ctypes.c_int
    if lib.pth_image_load_rgb8(path.encode(), None, ctypes.c_size_t(0), ctypes.byref(w), ctypes.byref(h), err, ctypes.c_int(512)) != 0:
        raise PathedError(err.value.decode())
    out = np.zeros((h.value, w.value, 3), np.uint8)
    lib.pth_image_load_rgb8(path.encode(), _ptr(out), ctypes.c_size_t(out.nbytes), ctypes.byref(w), ctypes.byref(h), err, ctypes.c_int(512))
    return out


def job_describe(job_path):
    """Every accessor of the C++ Job (pathed_b200/host/job.cpp) for a job file, as a dict."""
    import json
    out, err = ctypes.create_string_buffer(4096), ctypes.create_string_buffer(512)
    rc = host_lib().pth_job_describe(job_path.encode(), out, ctypes.c_int(4096), err, ctypes.c_int(512))
    if rc != 0:
        raise PathedError("Job(%s): %s" % (job_path, err.value.decode()))
    return json.loads(out.value.decode())


def bounce_controller(start, last, bounce):
    """(checkCounts, checkDone, copyAfterBounce window) of the C++ BounceController."""
    a, b = ctypes.c_int(), ctypes.c_int()
    bits = host_lib().pth_bounce_controller(ctypes.c_int(start), ctypes.c_int(last), ctypes.c_int(bounce), ctypes.byref(a), ctypes.byref(b))
    return bool(bits & 1), bool(bits & 2), (a.value, b.value)


def image_save(output_directory, stem, rgb, spp, bmp_name=""):
    """Image::set per pixel (row 0 = bottom), setSpp, saveCheckpoint(stem), write(bmp); returns the 8-bit preview."""
    rgb = np.ascontiguousarray(rgb, np.float32)
    h, w, _ = rgb.shape
    preview = np.zeros((h, w, 3), np.uint8)
    rc = host_lib().pth_image_save(output_directory.encode(), stem.encode(), bmp_name.encode(), ctypes.c_int(w), ctypes.c_int(h),
                                   ctypes.c_int(spp), _ptr(rgb), _ptr(preview))
    if rc != 0:
        raise PathedError("Image::save failed")
    return preview


def read_exr(path):
    """RGBA fp32, top scanline first (pathed_b200/host/exr_io.cpp)."""
    lib = host_lib()
    w, h = ctypes.c_int(), ctypes.c_int()
    if lib.pth_exr_read_rgba(path.encode(), None, ctypes.c_int(0), ctypes.byref(w), ctypes.byref(h)) != 0:
        raise PathedError("cannot read " + path)
    out = np.zeros((h.value, w.value, 4), np.float32)
    lib.pth_exr_read_rgba(path.encode(), _ptr(out), ctypes.c_int(w.value * h.value), ctypes.byref(w), ctypes.byref(h))
    return out


def scene_query(scene_file, origin, direction, max_t):
    """Scene::testIntersect + Scene::testOcclusion of the C++ host layer for one ray (needs a GPU)."""
    o = (ctypes.c_float * 3)(*origin); d = (ctypes.c_float * 3)(*direction)
    out = (ctypes.c_float * 14)(); occ = ctypes.c_int(); err = ctypes.create_string_buffer(512)
    rc = host_lib().pth_scene_query(scene_file.handle, o, d, ctypes.c_float(max_t), out, ctypes.byref(occ), err, ctypes.c_int(512))
    if rc != 0:
        raise PathedError(err.value.decode())
    v = list(out)
    return {"hit": v[0] != 0, "t": v[1], "point": v[2:5], "normal": v[5:8], "shading_normal": v[8:11], "uv": v[11:13],
            "material": int(v[13]), "occluded": occ.value != 0}


_cuda_lib = None


def cuda_lib():
    """The product library.  Fails loudly when it is missing: there is no CPU fallback."""
    global _cuda_lib
    if _cuda_lib is None:
        path = os.path.join(PKG_DIR, "libpathed_cuda.so")
        if not os.path.exists(path):
            raise PathedError("libpathed_cuda.so is not built; run `python -c 'import __graft_entry__ as g; g.build()'`")
        _cuda_lib = ctypes.CDLL(path)
    return _cuda_lib


def create_context(device=0):
    return Api(cuda_lib(), "ptc_", device)


def load_scene(scene_json, width, height, device=0, root=REPO_ROOT, options=None, integrator=PATH_TRACER):
    """parseScene + upload: the Python spelling of what app/main.cpp does before Integrator::run.
    options: ptc_set_option pairs applied before the commit (e.g. {"bvh_builder": 0} for the host SAH builder)."""
    api = create_context(device)
    for name, value in (options or {}).items():
        api.set_option(name, value)
    SceneFile(scene_json, width, height, root).feed(api)
    api.set_integrator(integrator)
    return api
