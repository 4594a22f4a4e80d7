// C entry points over the host layer, for Python (ctypes) tests and bench.py.
// The C++ classes (Job, Image, Scene, CudaPathTracer) are the drop-in surface for C++ callers;
// these wrappers only expose the parsers so scripts can load a scene file into any library that
// exports the ptc_* scene-description calls.
#include "exr_io.hpp"
#include "image_loader.hpp"
#include "pathed.hpp"
#include "scene_description.hpp"
#include "scene_parser.hpp"

#include <cstdio>
#include <cstring>
#include <exception>
#include <fstream>
#include <sstream>

using namespace pathed;

extern "C" {

int pth_scene_load(const char *sceneJson, const char *rootDirectory, int width, int height, void **out, char *err, int errLen)
{
    try {
        *out = new SceneDescription(parseScene(sceneJson, rootDirectory ? rootDirectory : "", width, height));
        return 0;
    } catch (const std::exception &e) {
        if (err && errLen > 0) { snprintf(err, (size_t)errLen, "%s", e.what()); }
        return -1;
    }
}

void pth_scene_free(void *scene) { delete (SceneDescription *)scene; }

int pth_scene_feed(void *scene, const SceneSink *sink) { return feedScene(*(SceneDescription *)scene, *sink); }

void pth_scene_counts(void *scene, uint32_t *geometries, uint32_t *triangles, uint32_t *spheres, uint32_t *materials)
{
    const SceneDescription &s = *(SceneDescription *)scene;
    uint32_t tris = 0, sph = 0;
    for (const GeometryDesc &g : s.geometries) { if (g.isSphere) { sph++; } else { tris += (uint32_t)g.materialOfTri.size(); } }
    *geometries = (uint32_t)s.geometries.size(); *triangles = tris; *spheres = sph; *materials = (uint32_t)s.materials.size();
}

// geometry access for tests (vertex-level fixtures)
int pth_scene_geometry(void *scene, uint32_t geom, const float **positions, uint32_t *nVertices, const uint32_t **indices,
                       const uint32_t **materialOfTri, uint32_t *nTriangles)
{
    const SceneDescription &s = *(SceneDescription *)scene;
    if (geom >= s.geometries.size() || s.geometries[geom].isSphere) { return -1; }
    const GeometryDesc &g = s.geometries[geom];
    *positions = g.positions.data(); *nVertices = (uint32_t)(g.positions.size() / 3);
    *indices = g.indices.data(); *materialOfTri = g.materialOfTri.data(); *nTriangles = (uint32_t)g.materialOfTri.size();
    return 0;
}

int pth_scene_material(void *scene, uint32_t id, ptc_material_desc *out)
{
    const SceneDescription &s = *(SceneDescription *)scene;
    if (id >= s.materials.size()) { return -1; }
    *out = s.materials[id];
    return 0;
}

// Texture::load's decode step: returns 0 and the size; copies the texels when `rgb` has room for them
int pth_image_load_rgb8(const char *path, uint8_t *rgb, size_t capacityBytes, int *width, int *height, char *err, int errLen)
{
    try {
        std::vector<uint8_t> data;
        loadImageRGB8(path, data, *width, *height);
        if (rgb && capacityBytes >= data.size()) { memcpy(rgb, data.data(), data.size()); }
        return 0;
    } catch (const std::exception &e) {
        if (err && errLen > 0) { snprintf(err, (size_t)errLen, "%s", e.what()); }
        return -1;
    }
}

int pth_exr_write_rgb_f32(const char *path, int width, int height, const float *rgb /*interleaved, top row first*/)
{
    try {
        std::vector<float> planes[3];
        for (int c = 0; c < 3; c++) { planes[c].resize((size_t)width * height); }
        for (size_t i = 0; i < (size_t)width * height; i++) { for (int c = 0; c < 3; c++) { planes[c][i] = rgb[3 * i + c]; } }
        saveEXR(path, width, height, {"B", "G", "R"}, {planes[2].data(), planes[1].data(), planes[0].data()}, false);
        return 0;
    } catch (const std::exception &) { return -1; }
}

int pth_exr_read_rgba(const char *path, float *rgba, int capacityPixels, int *width, int *height)
{
    try {
        std::vector<float> data;
        loadEXR(path, data, *width, *height);
        if (rgba && (size_t)capacityPixels >= (size_t)*width * *height) { memcpy(rgba, data.data(), data.size() * sizeof(float)); }
        return 0;
    } catch (const std::exception &) { return -1; }
}

// ---- Job / BounceController / Image: the host API of pathed.hpp, flattened for scripts

// every accessor of Job as one JSON object; "integrator_status" = "ok" | the text Job::integrator() threw
int pth_job_describe(const char *jobPath, char *out, int outLen, char *err, int errLen)
{
    try {
        std::ifstream file(jobPath);
        if (!file) { throw std::runtime_error(std::string("cannot open job file: ") + jobPath); }
        Job job(file);
        std::string status = "ok";
        try { job.integrator(); } catch (const char *message) { status = message; }
        std::ostringstream o;
        o << "{\"width\": " << job.width() << ", \"height\": " << job.height() << ", \"spp\": " << job.spp()
          << ", \"showUI\": " << (job.showUI() ? "true" : "false") << ", \"force\": " << (job.force() ? "true" : "false")
          << ", \"startBounce\": " << job.startBounce() << ", \"lastBounce\": " << job.lastBounce()
          << ", \"gpus\": " << job.gpus() << ", \"seed\": " << job.seed() << ", \"wave_spp\": " << job.waveSpp()
          << ", \"adaptive\": " << (job.adaptive() ? "true" : "false") << ", \"adaptive_threshold\": " << job.adaptiveThreshold()
          << ", \"adaptive_min_spp\": " << job.adaptiveMinSpp() << ", \"adaptive_step_spp\": " << job.adaptiveStepSpp()
          << ", \"denoise\": " << (job.denoise() ? "true" : "false")
          << ", \"denoise_checkpoints\": " << (job.denoiseCheckpoints() ? "true" : "false")
          << ", \"scene\": \"" << job.scene() << "\", \"output_directory\": \"" << job.outputDirectory()
          << "\", \"output_name\": \"" << job.outputName() << "\", \"integrator_status\": \"" << status << "\"}";
        snprintf(out, (size_t)outLen, "%s", o.str().c_str());
        return 0;
    } catch (const std::exception &e) {
        if (err && errLen > 0) { snprintf(err, (size_t)errLen, "%s", e.what()); }
        return -1;
    }
}

// bit 0 = checkCounts(bounce), bit 1 = checkDone(bounce); copyAfterBounce() window in *startAfter / *lastAfter
int pth_bounce_controller(int start, int last, int bounce, int *startAfter, int *lastAfter)
{
    const BounceController c(start, last), next = c.copyAfterBounce();
    if (startAfter) { *startAfter = next.startBounce(); }
    if (lastAfter) { *lastAfter = next.lastBounce(); }
    return (c.checkCounts(bounce) ? 1 : 0) | (c.checkDone(bounce) ? 2 : 0);
}

// Image::set for every pixel of rgb (row 0 = bottom scanline, like radianceLookup), then setSpp + saveCheckpoint(stem) into
// outputDirectory and write(bmpName); returns the 8-bit preview in preview (3*W*H)
int pth_image_save(const char *outputDirectory, const char *stem, const char *bmpName, int width, int height, int spp, const float *rgb, unsigned char *preview)
{
    try {
        std::istringstream jobText(std::string("{\"startBounce\": 0, \"lastBounce\": 0, \"output_directory\": \"") + outputDirectory + "\"}");
        Job job(jobText);
        Job *previous = g_job;
        g_job = &job;
        Image image(width, height);
        for (int row = 0; row < height; row++) {
            for (int col = 0; col < width; col++) {
                const float *px = rgb + 3 * ((size_t)row * width + col);
                image.set(row, col, px[0], px[1], px[2]);
            }
        }
        image.setSpp(spp);
        image.saveCheckpoint(stem);
        if (bmpName && bmpName[0]) { image.write(bmpName); }
        if (preview) { memcpy(preview, image.data().data(), image.data().size()); }
        g_job = previous;
        return 0;
    } catch (const std::exception &) { return -1; }
}

// Scene::testIntersect / Scene::testOcclusion for one ray (GPU): out = hit, t, point[3], normal[3], shadingNormal[3], uv[2], material
int pth_scene_query(void *sceneDescription, const float origin[3], const float direction[3], float maxT, float *out14, int *occluded, char *err, int errLen)
{
    try {
        Scene scene(*(SceneDescription *)sceneDescription, 1);
        Ray ray;
        for (int a = 0; a < 3; a++) { ray.origin[a] = origin[a]; ray.direction[a] = direction[a]; }
        const Intersection is = scene.testIntersect(ray);
        out14[0] = is.hit ? 1.f : 0.f; out14[1] = is.t;
        for (int a = 0; a < 3; a++) { out14[2 + a] = is.point[a]; out14[5 + a] = is.normal[a]; out14[8 + a] = is.shadingNormal[a]; }
        out14[11] = is.uv[0]; out14[12] = is.uv[1]; out14[13] = (float)is.material;
        *occluded = scene.testOcclusion(ray, maxT) ? 1 : 0;
        return 0;
    } catch (const std::exception &e) {
        if (err && errLen > 0) { snprintf(err, (size_t)errLen, "%s", e.what()); }
        return -1;
    }
}

} // extern "C"
