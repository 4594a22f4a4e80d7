/*
 * pathed_cuda.h — C ABI of the B200-native replacement for Pathed's surface path-tracing hot path.
 *
 * This is the drop-in boundary (SURVEY.md §8(b)).  Pathed has no plugin loader; the seams a
 * maintainer binds are (1) the Embree `rtc*` build/query calls, (2) `Material` / `Light` /
 * `Camera` construction and (3) `Integrator::sampleImage`.  Every entry point below names the
 * reference interface it replaces (paths relative to the reference repo root).
 *
 * Conventions
 *  - plain pointers and sizes only; all input pointers are HOST memory unless the name says
 *    `_device`; inputs are copied during the call (caller keeps ownership);
 *  - every call returns PTC_OK (0) or a negative status; `ptc_last_error` gives the text;
 *    no C++ exception crosses the ABI (the reference's `exit(1)` / `throw` sites map to statuses);
 *  - one context drives ONE GPU and is not thread-safe; multi-GPU = one context per process/GPU;
 *  - there is no CPU fallback: without a CUDA device `ptc_create` fails.
 */
#ifndef PATHED_CUDA_H
#define PATHED_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ptc_ctx ptc_ctx;

enum {
    PTC_OK = 0,
    PTC_ERR_INVALID = -1, /* bad argument (the reference would assert / throw std::runtime_error) */
    PTC_ERR_CUDA = -2,    /* CUDA runtime failure */
    PTC_ERR_STATE = -3,   /* call order violated (e.g. render before commit) */
    PTC_ERR_NOMEM = -4
};

#define PTC_INVALID_ID 0xFFFFFFFFu /* = RTC_INVALID_GEOMETRY_ID */

/* Material types on the hot path (src/scene_parser.cpp:parseMaterial, :604-700). */
enum {
    PTC_LAMBERTIAN = 0, /* src/lambertian.cpp */
    PTC_OREN_NAYAR = 1, /* src/oren_nayar.cpp */
    PTC_MIRROR = 2,     /* src/mirror.cpp */
    PTC_GLASS = 3,      /* src/glass.cpp */
    PTC_MICROFACET = 4, /* src/microfacet.cpp */
    PTC_PLASTIC = 5,    /* src/plastic.cpp */
    PTC_PASSTHROUGH = 6 /* src/passthrough.cpp: the container material of participating media (isContainer, isDelta) */
};
/* Job::integrator (src/job.cpp:66-75) */
enum { PTC_INTEGRATOR_PATH_TRACER = 0 /* src/path_tracer.cpp */, PTC_INTEGRATOR_VOLUME_PATH_TRACER = 1 /* src/volume_path_tracer.cpp */ };
#define PTC_NO_MEDIUM 0xFFFFFFFFu
/* volume events kept per ray by the volumetric queries (the reference's std::vector<VolumeEvent>, include/volume_event.h);
 * the reference only ever distinguishes 0, 1, 2 and "more" events (src/volume_helper.cpp:42-63, :80-120) */
#define PTC_MAX_EVENTS 8
enum { PTC_BECKMANN = 0 /* src/beckmann.cpp */, PTC_GGX = 1 /* src/ggx.cpp */ };
enum { PTC_ALBEDO_CONSTANT = 0, PTC_ALBEDO_CHECKERBOARD = 1 /* src/checkerboard.cpp */, PTC_ALBEDO_TEXTURE = 2 /* src/texture.cpp */ };

/* Flat form of what the reference's Material constructors receive
 * (include/lambertian.h, oren_nayar.h, glass.h, microfacet.h, plastic.h, checkerboard.h). */
typedef struct ptc_material_desc {
    int32_t type;
    float diffuse[3];     /* Lambertian / OrenNayar / Plastic diffuseReflectance */
    float emit[3];        /* Material::m_emit (Lambertian only in the reference's parser) */
    float sigma;          /* OrenNayar */
    float ior;            /* Glass (reference default 1.4, src/glass.cpp:16-18) */
    int32_t distribution; /* Microfacet / Plastic: PTC_BECKMANN | PTC_GGX */
    float alpha;
    int32_t albedo_kind;  /* Lambertian: constant colour or checkerboard */
    float checker_on[3];
    float checker_off[3];
    float checker_resolution[2];
    uint32_t texture;     /* albedo_kind == PTC_ALBEDO_TEXTURE (Lambertian, Plastic's diffuse lobe): id from ptc_add_texture */
} ptc_material_desc;

/* Ray as Scene::testIntersect / testOcclusion take it (include/ray.h): origin + direction.
 * tnear = 1e-3 and tfar = 1e5 (closest hit) / maxT - 1e-3 (occlusion) are applied inside,
 * exactly as src/scene.cpp:102-103 and :366-367 do. */
typedef struct ptc_ray {
    float origin[3];
    float direction[3];
} ptc_ray;

/* Raw hit record = the RTCHit fields the reference reads (src/scene.cpp:115-176). */
typedef struct ptc_hit {
    float t; /* ray.tfar after rtcIntersect1; 1e5 on a miss */
    float u, v;
    uint32_t geom_id; /* PTC_INVALID_ID on a miss */
    uint32_t prim_id;
    float ng[3]; /* unnormalised geometric normal */
} ptc_hit;

/* Processed intersection = the reference's `Intersection` (include/intersection.h:13-24). */
typedef struct ptc_isect {
    int32_t hit;
    float t;
    float point[3];
    float wo[3];
    float normal[3];
    float shading_normal[3];
    float uv[2];
    uint32_t material; /* id returned by ptc_add_material */
} ptc_isect;

/* Result of Light::sample / Scene::sampleDirectLights (include/shape.h:15-20, include/scene.h:46-81). */
typedef struct ptc_light_sample_t {
    float point[3];
    float normal[3];
    float inv_pdf;
    int32_t measure; /* 0 = solid angle, 1 = area */
    float solid_angle_pdf; /* LightSample::solidAnglePDF(reference point) */
    float emit[3];         /* light->emit(lightWo) toward the reference point */
} ptc_light_sample_t;

typedef struct ptc_stats {
    uint64_t closest_rays; /* rays traced by the extend stage (one per vertex: the MIS probe and the
                              continuation ray of src/path_tracer.cpp:44 / :175 are the same ray) */
    uint64_t shadow_rays;
    uint64_t samples;
    uint64_t kernel_launches;
    uint64_t bvh_nodes;
    uint64_t bvh_triangles;
    uint64_t bvh_bytes;
    /* traversal work counters, filled while option "count_traversal" is on (same code path as the scalar
     * reference traversal of ptc_count_traversal; SURVEY.md 8(d): algorithmic bytes per ray) */
    uint64_t extend_inner_visits, extend_triangle_tests;
    uint64_t shadow_inner_visits, shadow_triangle_tests;
    /* per-stage device time (CUDA events on the launching stream), filled while option "stage_timing" is on */
    uint64_t extend_launches, shadow_launches, shade_launches;
    float extend_ms, shadow_ms, shade_ms, other_ms;
    float last_render_ms; /* device time of the last ptc_render call (CUDA events, copies included) */
    /* BVH build of ptc_commit (rtcCommitScene, src/scene.cpp:39): wall time of the build incl. its synchronisations,
     * builder used (1 = device: Morton sort + PLOC clustering + wide collapse in kernels, 0 = host binned SAH) */
    float bvh_build_ms;
    uint32_t bvh_builder, bvh_depth, bvh_ploc_iterations;
} ptc_stats;

/* ---- lifetime ----------------------------------------------------------------------------- */
/* replaces rtcNewDevice + rtcNewScene (app/main.cpp:46-56) */
int ptc_create(int device_ordinal, ptc_ctx **out);
void ptc_destroy(ptc_ctx *ctx); /* rtcReleaseScene / rtcReleaseDevice (app/main.cpp:122-123) */
const char *ptc_last_error(ptc_ctx *ctx);

/* ---- scene description (geometry sink = the rtc* build API) -------------------------------- */
/* replaces GeometryParser::processRTCGeometry (src/geometry_parser.cpp:5-97) and the mesh half of
 * Quad::parse (src/quad.cpp:34-150): vertices float3, per-vertex normal float3 (zeros = none, Q3),
 * per-vertex uv float2, indices uint3; material_of_tri = RTCManager's primID -> Surface -> Material
 * (src/rtc_manager.cpp:64-69).  geom ids are handed out sequentially in call order, like
 * rtcAttachGeometry. */
int ptc_add_triangle_mesh(ptc_ctx *ctx, const float *positions, const float *normals, const float *uvs,
                          uint32_t n_vertices, const uint32_t *indices, const uint32_t *material_of_tri,
                          uint32_t n_triangles, uint32_t *geom_id_out);
/* replaces Sphere::create (src/sphere.cpp:16-48): RTC_GEOMETRY_TYPE_SPHERE_POINT, one item */
int ptc_add_sphere(ptc_ctx *ctx, const float center_radius[4], uint32_t material, uint32_t *geom_id_out);
/* ---- hierarchical instancing (SURVEY 8(f) N4), up to RTC_MAX_INSTANCE_LEVEL_COUNT = 2 levels.
 * ptc_begin_instance .. ptc_end_instance replace parseInstance (src/scene_parser.cpp:231-249: rtcNewScene + parseObjects into it +
 * rtcCommitScene): triangle meshes added in between belong to the new instance scene, with geometry ids counting from 0 inside it
 * (the reference's quads, spheres and PLY meshes attach to the global scene even there -- src/quad.cpp:149, src/sphere.cpp:46,
 * src/ply_parser.cpp:143 -- and leave its surface tables inconsistent, so anything but a triangle mesh is refused).  Definitions
 * nest like the parser's recursion does; ptc_end_instance returns to the enclosing scene.
 * ptc_add_instance replaces parseInstanced (:449-492: rtcNewGeometry(RTC_GEOMETRY_TYPE_INSTANCE), rtcSetGeometryInstancedScene,
 * rtcSetGeometryTransform with a column-major 4x4 local-to-world matrix, rtcAttachGeometry): the placement takes the next geometry
 * id of the scene being described (the root scene outside a begin/end pair).  As in the reference, a hit on an instance keeps
 * Ng, the interpolated normal and uv in the instance's LOCAL space (src/scene.cpp:122-219 never transforms them back), t in world
 * units, and only root-scene surfaces become lights (src/scene_parser.cpp:173-182). */
int ptc_begin_instance(ptc_ctx *ctx, uint32_t *instance_scene_out);
int ptc_end_instance(ptc_ctx *ctx);
int ptc_add_instance(ptc_ctx *ctx, uint32_t instance_scene, const float local_to_world_column_major[16], uint32_t *geom_id_out);
/* rtcIntersect1 including RTCHit::instID: inst_ids[2 * i + level] = geometry id of the placement at that level (PTC_INVALID_ID:
 * none); geom_id / prim_id of the hit are those of the mesh inside the innermost instance scene (src/rtc_manager.cpp:37-54) */
int ptc_intersect_instanced(ptc_ctx *ctx, const ptc_ray *rays, uint32_t n, ptc_hit *hits, uint32_t *inst_ids);
/* replaces Texture::load (src/texture.cpp:12-32): the 8-bit RGB texels stbi_load(..., 3) returns, row 0 = top of the
 * image, width * height * 3 bytes.  Texture::lookup (:34-49: wrap, flip v, nearest texel, pow(c / 255, 2.2)) runs on the
 * device.  Register textures before the materials that name them. */
int ptc_add_texture(ptc_ctx *ctx, const uint8_t *rgb, int width, int height, uint32_t *texture_id_out);
/* replaces the Material subclass constructors */
int ptc_add_material(ptc_ctx *ctx, const ptc_material_desc *desc, uint32_t *material_id_out);
/* replaces HomogeneousMedium::HomogeneousMedium (src/homogeneous_medium.cpp:7-11) as parseMedia builds it
 * (src/scene_parser.cpp:202-229): sigma_t and sigma_s per channel (sigma_s defaults to 0 in the parser) */
int ptc_add_medium(ptc_ctx *ctx, const float sigma_t[3], const float sigma_s[3], uint32_t *medium_id_out);
/* replaces the `internal_medium` argument of Surface::Surface (include/surface.h:18-30) as the parsers pass it for every
 * surface of an obj / ply / sphere model (src/scene_parser.cpp:324-343, :370-381, :503-514): all primitives of geometry
 * `geom_id` enclose `medium_id`.  A Passthrough surface WITH a medium is skipped by the volumetric queries and by
 * Scene::testOcclusion, and leaves a volume event instead (the occlusion filter, src/scene.cpp:42-84). */
int ptc_set_internal_medium(ptc_ctx *ctx, uint32_t geom_id, uint32_t medium_id);
/* replaces Job::integrator (src/job.cpp:66-75): which L() ptc_render / ptc_framebuffer_render / ptc_radiance_replay run.
 * May be changed between renders. */
int ptc_set_integrator(ptc_ctx *ctx, int integrator);
/* replaces EnvironmentLight::EnvironmentLight (src/environment_light.cpp:14-54): RGBA fp32 lat-long
 * texels as tinyexr's LoadEXR returns them, scale, and both 4x4 row-major matrices of `mapToWorld` */
int ptc_set_environment(ptc_ctx *ctx, const float *rgba, int width, int height, float scale,
                        const float map_to_world[16], const float world_to_map[16]);
/* replaces Camera::Camera (src/camera.cpp:13-30): look-at + vertical fov in radians + resolution */
int ptc_set_camera(ptc_ctx *ctx, const float origin[3], const float target[3], const float up[3],
                   float vertical_fov, int width, int height, int flip_handedness);
/* replaces Scene::Scene -> rtcCommitScene (src/scene.cpp:26-40) and the light list of parseScene
 * (src/scene_parser.cpp:173-190): builds the BVH, the light table (emissive surfaces in registration
 * order, environment light last) and the environment CDFs; uploads everything */
int ptc_commit(ptc_ctx *ctx);

/* ---- hot path ------------------------------------------------------------------------------ */
/* replaces n_spp iterations of SampleIntegrator::sampleImage (src/sample_integrator.cpp:80-113):
 * adds, for every pixel, the radiance of samples first_sample .. first_sample+n_spp-1 into
 * accum_rgb (HOST, 3*W*H floats, index 3*(row*W+col)+c, row 0 = bottom; `+=` like radianceLookup).
 * start_bounce / last_bounce = BounceController (src/bounce_controller.cpp:14-25; -1 = unbounded,
 * capped at PTC_MAX_BOUNCES).  seed keys the Philox streams (pixel, sample, bounce).
 * The upload of accum_rgb overlaps the first wave of kernels.  A page-locked accum_rgb (cudaHostRegister of the vector the
 * reference keeps for the whole render, or cudaHostAlloc) is copied from and to directly; pageable memory goes through a staging
 * buffer of the context (two more host copies of the framebuffer per call). */
int ptc_render(ptc_ctx *ctx, uint64_t seed, uint32_t first_sample, uint32_t n_spp, int start_bounce,
               int last_bounce, float *accum_rgb);
/* optional: allocates the per-path state for waves of up to n_paths paths (clamped to "paths_per_wave") NOW instead of inside the
 * first render call.  Needs no scene: a renderer knows resolution and sample count from its job file (src/job.cpp:25-60) and can call
 * this -- from another thread -- while it parses the scene; 16 GB of cudaMalloc cost ~0.1 s of the first wave otherwise. */
int ptc_reserve_paths(ptc_ctx *ctx, uint64_t n_paths);
/* same, accumulating into a DEVICE buffer on `cuda_stream` (a cudaStream_t; NULL = default stream);
 * asynchronous: returns after enqueueing.  Used for multi-GPU (NCCL reduce of the buffer) */
int ptc_render_device(ptc_ctx *ctx, uint64_t seed, uint32_t first_sample, uint32_t n_spp, int start_bounce,
                      int last_bounce, float *accum_rgb_device, void *cuda_stream);
/* K7 resolve: out[i] = accum[i] / spp on the device (src/integrator.cpp:74-85) */
int ptc_resolve_device(ptc_ctx *ctx, const float *accum_rgb_device, float *out_rgb_device, uint32_t spp,
                       void *cuda_stream);
#define PTC_MAX_BOUNCES 64

/* SURVEY 8(e), "the BVH is built once and broadcast": a committed context copied to another GPU.  The new context owns copies of
 * everything ptc_commit put on the device (BVH, shading records, material / light tables, environment map and its sampling
 * tables, textures), made with peer copies over NVLink -- no second parse, feed or build (replaces calling the whole
 * Scene::Scene / rtcCommitScene sequence of src/scene.cpp, src/rtc_manager.cpp once per device).  Options are inherited. */
int ptc_replicate(ptc_ctx *src, int device, ptc_ctx **out);

/* ---- context-owned device framebuffer: Integrator::run's radianceLookup kept in HBM ----------- */
/* `std::vector<float> radianceLookup(3*W*H)` zero-filled (src/integrator.cpp:37-40) */
int ptc_framebuffer_clear(ptc_ctx *ctx);
/* ptc_render into the context's framebuffer; asynchronous on the context's stream, no host traffic */
int ptc_framebuffer_render(ptc_ctx *ctx, uint64_t seed, uint32_t first_sample, uint32_t n_spp, int start_bounce,
                           int last_bounce);
/* K7 + the multi-GPU reduce in ONE kernel on `root`'s device: out = (root's framebuffer + every peer context's
 * framebuffer, read through NVLink peer mappings) / divisor, i.e. `radianceLookup[i] / (i + 1)` of
 * src/integrator.cpp:74-85 over the spp split of SURVEY 8(e).  Waits for all contexts' pending renders,
 * copies the result to out_rgb_host (3*W*H floats) and returns when it is there.  divisor = 1 gives the raw sums.
 * peers may be NULL when n_peers = 0; at most PTC_MAX_PEERS peers. */
int ptc_framebuffer_gather(ptc_ctx *root, ptc_ctx *const *peers, uint32_t n_peers, uint32_t divisor, float *out_rgb_host);
#define PTC_MAX_PEERS 15
/* ptc_framebuffer_render that also keeps the images the reference checkpoints (src/integrator.cpp:87-92: `auto-%05dspp.exr` after
 * 1, 2, 4, ... samples) WITHOUT ending a wave there: snapshot i = this context's sums over the samples it has rendered with a
 * global index below sample_counts[i] (ascending; at most PTC_MAX_CHECKPOINTS).  The K7 resolve writes the copies while it adds
 * the wave's samples in order, so a snapshot holds exactly the floats a render that stopped there would hold.  Snapshots stay
 * valid until the context's next framebuffer render. */
int ptc_framebuffer_render_checkpoints(ptc_ctx *ctx, uint64_t seed, uint32_t first_sample, uint32_t n_spp, int start_bounce,
                                       int last_bounce, const uint32_t *sample_counts, uint32_t n_counts);
#define PTC_MAX_CHECKPOINTS 32
/* ptc_framebuffer_gather in two halves, so that the host enqueues the next wave before it waits for this one's image
 * (src/integrator.cpp:42-105 alternates render and host work; here they overlap).  begin: enqueues reduce + resolve of the
 * framebuffers (snapshot < 0) or of snapshot `snapshot` of every context and the copy to a pinned host buffer; later renders
 * on any of the contexts are ordered after the reads.  end: waits for that copy and hands the image out. */
int ptc_framebuffer_gather_begin(ptc_ctx *root, ptc_ctx *const *peers, uint32_t n_peers, int snapshot, uint32_t divisor,
                                 uint32_t *ticket);
int ptc_framebuffer_gather_end(ptc_ctx *root, uint32_t ticket, float *out_rgb_host);

/* ---- adaptive sampling: each pixel stops once its estimated relative error meets a target ------------------------------ */
/* A render is a sequence of passes into the context's framebuffer.  Pass 1 gives every pixel samples 0 .. min_spp - 1; each later
 * pass gives every pixel still ACTIVE the next min(step_spp, max_spp - n) samples, so all active pixels share one count n.  After a
 * pass pixel p stops when, for every channel c, var_c / n <= threshold^2 * (mean_c^2 + 1e-2), with mean_c = S_c / n, var_c =
 * max(0, (M_c - n mean_c^2) / (n - 1)), S the framebuffer's sum and M the sum of the squared samples, evaluated in fp64: the
 * expected per-pixel term of the relMSE metric (x - r)^2 / (r^2 + 1e-2) (SURVEY 8(d)) is at most threshold^2.  A non-finite
 * estimate never stops a pixel (a NaN sample keeps it going to max_spp); every pixel stops at max_spp.
 * A path's random stream is keyed by (pixel, sample index) and the resolve adds a pixel's samples in sample order, so pixel p of
 * the adaptive framebuffer holds exactly, bit for bit, what ptc_render(seed, 0, n_p, ...) accumulates there from zero.
 * Device memory: 24 bytes per pixel besides the framebuffer (second moments 3 x fp32, count, two pixel-list entries). */
typedef struct ptc_adaptive_desc {
    float threshold;   /* tau > 0: the relMSE target is tau^2 */
    uint32_t min_spp;  /* >= 2: samples of the first pass */
    uint32_t step_spp; /* >= 1: samples per later pass */
    uint32_t max_spp;  /* >= min_spp */
} ptc_adaptive_desc;
/* clears the framebuffer, the second moments and the counts; every pixel active.  PTC_ERR_INVALID for a bad descriptor.
 * Until the next ptc_framebuffer_clear the framebuffer belongs to the adaptive render: ptc_framebuffer_render* return
 * PTC_ERR_STATE (ptc_render, ptc_render_device and ptc_framebuffer_gather work as usual; the gather with divisor 1 reads the sums) */
int ptc_adaptive_begin(ptc_ctx *ctx, const ptc_adaptive_desc *desc);
/* one pass on the context's stream, returns when the stopping test is done (one host synchronisation per pass): active_out =
 * pixels still active (0: the render is complete and further calls are no-ops), spp_out = the samples the active pixels hold
 * after the pass.  Either pointer may be NULL.  PTC_ERR_STATE before ptc_adaptive_begin.  ptc_stats.samples counts the samples traced. */
int ptc_adaptive_pass(ptc_ctx *ctx, uint64_t seed, int start_bounce, int last_bounce, uint32_t *active_out, uint32_t *spp_out);
/* spp_per_pixel (W*H) = the samples each pixel holds so far, second_moment_rgb (3*W*H) = per-channel sums of the squared samples;
 * index row*W + col, row 0 = bottom, like the framebuffer.  Either may be NULL.  PTC_ERR_STATE before ptc_adaptive_begin. */
int ptc_adaptive_state(ptc_ctx *ctx, uint32_t *spp_per_pixel, float *second_moment_rgb);

/* ---- denoising: first-hit guide buffers and a variance-guided a-trous filter (DESIGN §10) ------------------------------ */
/* snapshot argument of ptc_framebuffer_gather_begin: sum the second-moment buffers of root + peers instead of the framebuffers
 * (a context's adaptive render's moments, else its option "framebuffer_moments" buffer; use divisor 1).  PTC_ERR_STATE for a
 * context whose moments do not cover every sample of its framebuffer: the option must be on at ptc_framebuffer_clear and at every
 * framebuffer render since (a context that rendered no samples has zero moments). */
#define PTC_GATHER_MOMENTS (-2)
/* Adds into the host buffers (index row*W + col, row 0 = bottom, `+=` like ptc_render), for every pixel and every sample s in
 * first_sample .. first_sample + n_spp - 1, in sample order and in fp32, what the first hit of the path tracer's camera ray for
 * (seed, pixel, s) sees -- the same two Philox draws of vertex 0 jitter cameraRay(row + jy, col + jx), the closest hit is
 * Scene::testIntersect's (ptc_intersect_full):
 *   albedo_rgb (3*W*H): Lambertian / OrenNayar / Plastic: the diffuse colour, checkerboard or texture the BSDF uses; Mirror,
 *                       Glass, Microfacet, Passthrough: (1, 1, 1); a miss: 0
 *   normal_xyz (3*W*H): the shading normal, unflipped (in an instance's local space for instanced geometry); a miss: 0
 *   depth      (W*H):   the hit distance t; a miss: 0
 *   hits       (W*H):   +1 per sample that hits.
 * The same for both integrators; draws no random numbers of the paths and leaves the framebuffer alone. */
int ptc_render_aovs(ptc_ctx *ctx, uint64_t seed, uint32_t first_sample, uint32_t n_spp, float *albedo_rgb, float *normal_xyz,
                    float *depth, uint32_t *hits);
/* the spatial filter of SVGF (Schied et al., HPG 2017) with an albedo edge-stopping term; the formula is in DESIGN §10 */
typedef struct ptc_denoise_desc {
    uint32_t iterations; /* a-trous levels, steps 1, 2, 4, ...: 0 .. 10 (0 returns S / n) */
    float sigma_l;       /* > 0: luminance, in units of the blurred standard deviation of the mean */
    float sigma_n;       /* >= 0: exponent of the normal term */
    float sigma_z;       /* > 0: relative depth difference per unit of the step */
    float sigma_a;       /* > 0: L1 albedo difference */
    float eps;           /* > 0 */
} ptc_denoise_desc;
#define PTC_DENOISE_DEFAULTS {5u, 4.f, 128.f, 1.f, 0.1f, 1e-6f}
typedef struct ptc_denoise_input {
    const float *sums;       /* 3*W*H: sums of the samples (the framebuffer) */
    const float *moments;    /* 3*W*H: sums of the squared samples */
    const uint32_t *counts;  /* W*H samples per pixel (adaptive renders), or NULL: every pixel has `spp` */
    uint32_t spp;
    const float *albedo_rgb, *normal_xyz, *depth; /* ptc_render_aovs over aov_spp samples */
    const uint32_t *hits;
    uint32_t aov_spp;
} ptc_denoise_input;
/* out_rgb (3*W*H) = the denoised mean colour; W, H from the context's camera; all pointers are host pointers.  Runs on the
 * context's device and returns when the output is on the host.  Deterministic: two calls give the same bytes.  PTC_ERR_INVALID
 * for a bad descriptor, a missing input, a pixel with fewer than 2 samples or aov_spp == 0. */
int ptc_denoise(ptc_ctx *ctx, const ptc_denoise_desc *desc, const ptc_denoise_input *in, float *out_rgb);
/* Device-resident denoising of the contexts' own images.  With option "framebuffer_moments" on, ptc_framebuffer_render_checkpoints
 * also keeps the second moments of every snapshot (12 B per pixel per snapshot, next to the snapshot's sums); a snapshot's moments
 * count as complete under the rule of PTC_GATHER_MOMENTS at the time it was written.
 * ptc_framebuffer_guides: ptc_render_aovs into context-owned device buffers, from zero (replaces the previous call's guides); the
 * guide records for ptc_framebuffer_denoise_begin are built here.  Any host pointer may be NULL; non-NULL ones receive the sums
 * (like ptc_render_aovs from zeroed buffers).  Asynchronous on the context's stream unless a host pointer is given.
 * PTC_ERR_INVALID for n_spp == 0. */
int ptc_framebuffer_guides(ptc_ctx *ctx, uint64_t seed, uint32_t first_sample, uint32_t n_spp, float *albedo_rgb, float *normal_xyz,
                           float *depth, uint32_t *hits);
/* ptc_denoise of snapshot `snapshot` (< 0: the framebuffers) of root + peers, summed as ptc_framebuffer_gather_begin sums them, with
 * their second moments summed the same way and the root's device guides (aov_spp = the n_spp of ptc_framebuffer_guides); spp =
 * samples per pixel of that image (ignored on a root that holds an adaptive render: its per-pixel counts are used).  Enqueues only;
 * the image (3*W*H) is fetched with ptc_framebuffer_gather_end(root, ticket, out).  Same bytes as ptc_denoise on the gathered inputs.
 * PTC_ERR_INVALID: a bad descriptor or arguments, spp < 2 on a uniform image.  PTC_ERR_STATE: no guides on the root or guides of
 * another resolution, a snapshot that was not rendered (or any snapshot of an adaptive root), moments that do not cover every sample
 * of a context, an adaptive root before its first pass. */
int ptc_framebuffer_denoise_begin(ptc_ctx *root, ptc_ctx *const *peers, uint32_t n_peers, int snapshot, uint32_t spp,
                                  const ptc_denoise_desc *desc, uint32_t *ticket);

/* ---- the random streams on their own (known-answer tests; need no scene) ---------------------- */
/* Philox4x32-10, the generator that replaces RandomGenerator (src/random_generator.cpp:4-11) and std::rand (src/camera.cpp:51-52)
 * on the device: out[4i..4i+3] = philox(counter = counters[4i..4i+3], key = keys[2i..2i+1]) */
int ptc_philox4x32_10(ptc_ctx *ctx, const uint32_t *counters, const uint32_t *keys, uint32_t n, uint32_t *out);
/* the first `draws` uniform floats in [0, 1) a path draws at a vertex: stream i = (pixel, sample, bounce) = streams[3i..3i+2] under
 * `seed`, out[i * draws + d] = draw d (counter = (pixel, sample, bounce, d / 4), lane d % 4, top 24 bits) */
int ptc_uniforms(ptc_ctx *ctx, uint64_t seed, const uint32_t *streams, uint32_t n_streams, uint32_t draws, float *out);

/* ---- ray queries (keep Scene::testIntersect / testOcclusion alive for CPU integrators; parity) */
int ptc_intersect(ptc_ctx *ctx, const ptc_ray *rays, uint32_t n, ptc_hit *hits);        /* rtcIntersect1 */
int ptc_intersect_full(ptc_ctx *ctx, const ptc_ray *rays, uint32_t n, ptc_isect *out);  /* Scene::testIntersect */
int ptc_occluded(ptc_ctx *ctx, const ptc_ray *rays, const float *max_t, uint32_t n, uint8_t *occluded); /* Scene::testOcclusion */
/* Scene::testVolumetricOcclusion (src/scene.cpp:383-424): occlusion with container surfaces filtered out; n_events[i] = number
 * of distinct volume events on an unoccluded ray, event_t / event_medium[PTC_MAX_EVENTS * i ...] = those events sorted by t
 * (when there are more than PTC_MAX_EVENTS, the ones the traversal met first); either array may be NULL */
int ptc_occluded_volumetric(ptc_ctx *ctx, const ptc_ray *rays, const float *max_t, uint32_t n, uint8_t *occluded,
                            uint32_t *n_events, float *event_t, uint32_t *event_medium);
/* Scene::testVolumetricIntersect (src/scene.cpp:225-353): closest hit that is not a container-with-medium surface, plus the
 * volume events in front of it */
int ptc_intersect_volumetric(ptc_ctx *ctx, const ptc_ray *rays, uint32_t n, ptc_isect *out, uint32_t *n_events, float *event_t,
                             uint32_t *event_medium);
/* device-resident variants used by the benchmark (rays/hits already in HBM) */
int ptc_intersect_device(ptc_ctx *ctx, const ptc_ray *rays_device, uint32_t n, ptc_hit *hits_device, void *cuda_stream);
int ptc_occluded_device(ptc_ctx *ctx, const ptc_ray *rays_device, const float *max_t_device, uint32_t n,
                        uint8_t *occluded_device, void *cuda_stream);

/* ---- function-level probes (parity of shading / sampling code against the reference) --------- */
/* Camera::generateRay(float row, float col) (src/camera.cpp:32-47) */
int ptc_camera_rays(ptc_ctx *ctx, const float *row_col, uint32_t n, ptc_ray *rays);
/* Material::f(isect, wi, &pdf) */
int ptc_bsdf_eval(ptc_ctx *ctx, uint32_t material, const ptc_isect *isects, const float *wi, uint32_t n,
                  float *f_rgb, float *pdf);
/* Material::sample(isect, random) with the random stream given explicitly: xi[3*i .. 3*i+2] */
int ptc_bsdf_sample(ptc_ctx *ctx, uint32_t material, const ptc_isect *isects, const float *xi, uint32_t n,
                    float *wi, float *pdf, float *throughput_rgb);
/* Scene::sampleDirectLights(point, random): xi[3*i] picks the light, xi[3*i+1..2] the point */
int ptc_light_sample(ptc_ctx *ctx, const float *ref_points, const float *xi, uint32_t n, ptc_light_sample_t *out);
/* Scene::lightsPDF / environmentPDF for the ray origin -> direction: >= 0 light pdf when the ray lands on
 * an emitter, -1 when it contributes nothing, -2 - pdf for an environment miss */
int ptc_light_pdf(ptc_ctx *ctx, const ptc_ray *rays, uint32_t n, float *pdf);
/* Scene::environmentL(direction) */
int ptc_environment_radiance(ptc_ctx *ctx, const float *directions, uint32_t n, float *rgb);
/* body of SampleIntegrator::samplePixel + PathTracer::L (or VolumePathTracer::L, see ptc_set_integrator) for explicit primary rays, the random stream
 * replayed sequentially from xi[i*stride ...] (test hook: same draws in the same order as the reference) */
int ptc_radiance_replay(ptc_ctx *ctx, const ptc_ray *rays, const float *xi, uint32_t stride, uint32_t n,
                        int start_bounce, int last_bounce, float *rgb);

/* ---- introspection ------------------------------------------------------------------------- */
int ptc_num_lights(ptc_ctx *ctx, uint32_t *out); /* Scene::lights().size() */
int ptc_get_stats(ptc_ctx *ctx, ptc_stats *out);
int ptc_reset_stats(ptc_ctx *ctx);
/* queue sizes of the most recent wave: extend_counts[k] = rays that left vertex k (k = 0: camera rays), shadow_counts[k] =
 * NEE shadow rays cast at vertex k; up to `capacity` (<= PTC_MAX_BOUNCES + 2) entries each (of the wave's first lane when it was
 * traced as several, see "lanes") */
int ptc_get_wave_counts(ptc_ctx *ctx, uint32_t *extend_counts, uint32_t *shadow_counts, uint32_t capacity);
int ptc_set_option(ptc_ctx *ctx, const char *name, int64_t value); /* "stage_timing", "count_traversal", "paths_per_wave",
                                                                      "overlap_shadow", "bvh_builder" (before ptc_commit: 1 device,
                                                                      0 host), "volume_megakernel" (1: VolumePathTracer as one
                                                                      thread per path instead of wavefront stages), "lanes" (a
                                                                      wave traced as n part-waves side by side on n streams; 0,
                                                                      the default: chosen per wave; the image does not depend on n),
                                                                      "framebuffer_moments" (1: ptc_framebuffer_render* also add the
                                                                      squared samples into a context buffer that ptc_framebuffer_clear
                                                                      zeroes, read with PTC_GATHER_MOMENTS; set it before the clear;
                                                                      the sums do not change) */
/* scalar reference traversal of the device BVH on the host side of the library: counts inner-node
 * visits and triangle tests per ray (SURVEY.md §8(d): algorithmic bytes per ray) */
int ptc_count_traversal(ptc_ctx *ctx, const ptc_ray *rays, uint32_t n, uint64_t *inner_visits, uint64_t *triangle_tests);

/* host-only self-check of the BVH builder and of the traversal code it shares with the kernels (needs no GPU and no
 * context): builds the compressed wide BVH of a triangle soup, traces `rays` (closest hit, tnear 1e-3, tfar 1e5) with the
 * scalar traversal and by brute force over all triangles with the same triangle test.
 * stats: [0] inner nodes, [1] leaf triangles, [2] occupied child slots, [3] max depth, [4] inner visits, [5] triangle tests */
int ptc_bvh_selfcheck(const float *positions, uint32_t n_vertices, const uint32_t *indices, uint32_t n_triangles,
                      const ptc_ray *rays, uint32_t n_rays, float *t_bvh, uint32_t *prim_bvh, float *t_brute,
                      uint32_t *prim_brute, uint64_t stats[6]);

/* the same check with the builder chosen: 0 = the host binned-SAH builder, 1 = the DEVICE builder's per-element code
 * (Morton order, PLOC clustering, collapse, emission) executed serially on the host -- a test hook for the CPU suite;
 * ptc_commit runs that code only as CUDA kernels.  sah_cost: cost of the wide BVH under the collapse's cost model. */
int ptc_bvh_selfcheck_builder(int builder, const float *positions, uint32_t n_vertices, const uint32_t *indices,
                              uint32_t n_triangles, const ptc_ray *rays, uint32_t n_rays, float *t_bvh, uint32_t *prim_bvh,
                              float *t_brute, uint32_t *prim_brute, uint64_t stats[6], double *sah_cost);

#ifdef __cplusplus
}
#endif
#endif /* PATHED_CUDA_H */
