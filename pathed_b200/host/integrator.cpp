// Scene (ray queries over the GPU BVH), Integrator::run and CudaPathTracer: the rendering side of the host API.
// The reference's loop is /root/reference/src/integrator.cpp:19-106 -> src/sample_integrator.cpp:80-113 -> src/path_tracer.cpp:19-216;
// here one call into the C ABI covers a whole batch of samples per pixel and the framebuffer stays in HBM between checkpoints.
#include "pathed.hpp"

#include "exr_io.hpp"
#include "scene_parser.hpp"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <future>
#include <cstdio>
#include <iomanip>
#include <sstream>
#include <stdexcept>
#include <thread>

namespace pathed {

namespace {

void check(ptc_ctx *ctx, int status, const char *what)
{
    if (status != PTC_OK) { throw std::runtime_error(std::string(what) + ": " + ptc_last_error(ctx)); }
}

// adapters from the C ABI to the parser's sink table
int sinkMaterial(void *c, const ptc_material_desc *d, uint32_t *id) { return ptc_add_material((ptc_ctx *)c, d, id); }
int sinkMesh(void *c, const float *p, const float *n, const float *uv, uint32_t nv, const uint32_t *i, const uint32_t *m, uint32_t nt, uint32_t *g)
{
    return ptc_add_triangle_mesh((ptc_ctx *)c, p, n, uv, nv, i, m, nt, g);
}
int sinkSphere(void *c, const float *cr, uint32_t m, uint32_t *g) { return ptc_add_sphere((ptc_ctx *)c, cr, m, g); }
int sinkEnvironment(void *c, const float *rgba, int w, int h, float s, const float *m2w, const float *w2m)
{
    return ptc_set_environment((ptc_ctx *)c, rgba, w, h, s, m2w, w2m);
}
int sinkCamera(void *c, const float *o, const float *t, const float *u, float f, int w, int h, int flip)
{
    return ptc_set_camera((ptc_ctx *)c, o, t, u, f, w, h, flip);
}
int sinkCommit(void *c) { return ptc_commit((ptc_ctx *)c); }
int sinkTexture(void *c, const uint8_t *rgb, int w, int h, uint32_t *id) { return ptc_add_texture((ptc_ctx *)c, rgb, w, h, id); }
int sinkMedium(void *c, const float *st, const float *ss, uint32_t *id) { return ptc_add_medium((ptc_ctx *)c, st, ss, id); }
int sinkInternalMedium(void *c, uint32_t geom, uint32_t medium) { return ptc_set_internal_medium((ptc_ctx *)c, geom, medium); }
int sinkBeginInstance(void *c, uint32_t *scene) { return ptc_begin_instance((ptc_ctx *)c, scene); }
int sinkEndInstance(void *c) { return ptc_end_instance((ptc_ctx *)c); }
int sinkAddInstance(void *c, uint32_t scene, const float *m, uint32_t *g) { return ptc_add_instance((ptc_ctx *)c, scene, m, g); }

double now()
{
    return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// The guide buffers need far fewer samples than the colour (a pixel's first hits differ only across its footprint): at most this many
const uint32_t kGuideSpp = 16;
uint32_t guideSpp() { return std::min<uint32_t>((uint32_t)g_job->spp(), kGuideSpp); }

// The guides of the first guideSpp() samples on device 0 for ptc_framebuffer_denoise_begin, enqueued without waiting for them
void enqueueGuides(ptc_ctx *ctx, uint64_t seed)
{
    check(ctx, ptc_framebuffer_guides(ctx, seed, 0, guideSpp(), nullptr, nullptr, nullptr, nullptr), "guide buffers");
}

} // namespace

// ------------------------------------------------------------------------------------------------ Scene
Scene::Scene(const SceneDescription &description, int gpus, ptc_ctx *first, uint64_t reservePaths) : m_width(description.camera.width), m_height(description.camera.height)
{
    // device 0 is fed and builds the BVH; the other devices of the spp split receive copies of the finished device data (SURVEY 8(e))
    ptc_ctx *ctx = first;
    if (!ctx && (ptc_create(0, &ctx) != PTC_OK || !ctx)) { throw std::runtime_error("Failed to create device 0 (no CUDA device? there is no CPU path)"); }
    m_contexts.push_back(ctx);
    const SceneSink sink = {ctx, sinkMaterial, sinkMesh, sinkSphere, sinkEnvironment, sinkCamera, sinkCommit, sinkTexture, sinkMedium, sinkInternalMedium, sinkBeginInstance, sinkEndInstance, sinkAddInstance};
    const int status = feedScene(description, sink);
    if (status != PTC_OK) {
        const std::string message = ptc_last_error(ctx);
        ptc_destroy(ctx); m_contexts.clear();
        throw std::runtime_error("scene upload failed: " + message);
    }
    // one thread per further device: creating a CUDA context takes a few hundred milliseconds, the copies run over NVLink side by side
    const int devices = std::max(1, gpus);
    std::vector<ptc_ctx *> copies((size_t)devices, nullptr);
    std::vector<int> outcome((size_t)devices, PTC_OK);
    std::vector<std::thread> workers;
    for (int device = 1; device < devices; device++) {
        workers.emplace_back([&, device]() {
            outcome[(size_t)device] = ptc_replicate(ctx, device, &copies[(size_t)device]);
            if (outcome[(size_t)device] == PTC_OK && copies[(size_t)device] && reservePaths) { ptc_reserve_paths(copies[(size_t)device], reservePaths); }
        });
    }
    for (std::thread &worker : workers) { worker.join(); }
    for (int device = 1; device < devices; device++) {
        if (outcome[(size_t)device] != PTC_OK || !copies[(size_t)device]) {
            const std::string message = ptc_last_error(ctx);
            for (ptc_ctx *c : copies) { if (c) { ptc_destroy(c); } }
            ptc_destroy(ctx); m_contexts.clear();
            throw std::runtime_error("Failed to replicate the scene to device " + std::to_string(device) + ": " + message);
        }
        m_contexts.push_back(copies[(size_t)device]);
    }
}

Scene::~Scene()
{
    for (ptc_ctx *ctx : m_contexts) { ptc_destroy(ctx); }
}

Intersection Scene::testIntersect(const Ray &ray) const
{
    std::lock_guard<std::mutex> guard(m_queryLock);
    ptc_ray r;
    for (int a = 0; a < 3; a++) { r.origin[a] = ray.origin[a]; r.direction[a] = ray.direction[a]; }
    ptc_isect is;
    check(m_contexts[0], ptc_intersect_full(m_contexts[0], &r, 1, &is), "testIntersect");
    Intersection out;
    out.hit = is.hit != 0;
    out.t = is.t; // miss: std::numeric_limits<float>::max(), like IntersectionHelper::miss (include/intersection.h:60-72)
    for (int a = 0; a < 3; a++) {
        out.point[a] = is.point[a]; out.woWorld[a] = is.wo[a]; out.normal[a] = is.normal[a]; out.shadingNormal[a] = is.shading_normal[a];
    }
    out.uv[0] = is.uv[0]; out.uv[1] = is.uv[1];
    out.material = is.material;
    return out;
}

bool Scene::testOcclusion(const Ray &ray, float maxT) const
{
    std::lock_guard<std::mutex> guard(m_queryLock);
    ptc_ray r;
    for (int a = 0; a < 3; a++) { r.origin[a] = ray.origin[a]; r.direction[a] = ray.direction[a]; }
    uint8_t occluded = 0;
    check(m_contexts[0], ptc_occluded(m_contexts[0], &r, &maxT, 1, &occluded), "testOcclusion");
    return occluded != 0;
}

uint32_t Scene::lightCount() const
{
    uint32_t n = 0;
    check(m_contexts[0], ptc_num_lights(m_contexts[0], &n), "lightCount");
    return n;
}

std::unique_ptr<Scene> parseSceneForJob(const Job &job, const std::string &rootDirectory)
{
    // the CUDA runtime comes up (driver initialisation, module load: seconds on a multi-GPU box) while the host parses the scene files
    // ... and so does the path state of the first wave: resolution and sample count are the job's, not the scene's
    const uint64_t wavePaths = (uint64_t)std::max(1, job.width()) * (uint64_t)std::max(1, job.height()) *
                               (uint64_t)std::max(1, std::min(job.waveSpp(), (job.spp() + std::max(1, job.gpus()) - 1) / std::max(1, job.gpus())));
    std::future<ptc_ctx *> device = std::async(std::launch::async, [wavePaths]() {
        ptc_ctx *ctx = nullptr;
        if (ptc_create(0, &ctx) == PTC_OK && ctx) { ptc_reserve_paths(ctx, wavePaths); } // best effort: the first render allocates what is missing
        return ctx;
    });
    const double begin = now();
    SceneDescription description;
    try { description = parseScene(job.scene(), rootDirectory, job.width(), job.height()); }
    catch (...) { if (ptc_ctx *ctx = device.get()) { ptc_destroy(ctx); } throw; }
    const double parsed = now();
    ptc_ctx *first = device.get();
    if (!first) { throw std::runtime_error("Failed to create device 0 (no CUDA device? there is no CPU path)"); }
    const double ready = now();
    std::unique_ptr<Scene> scene(new Scene(description, job.gpus(), first, wavePaths));
    printf("Scene: %0.2fs parsing, %0.2fs more until the device was up, %0.2fs upload + BVH build + copies to %d more GPU(s)\n",
           parsed - begin, ready - parsed, now() - ready, job.gpus() - 1);
    return scene;
}

// ------------------------------------------------------------------------------------------------ Integrator
// The reference's loop, kept for integrators that only provide sampleImage: one spp per wave through a HOST radianceLookup.
void Integrator::run(Image &image, Scene &scene, std::function<void(RenderStatus)> callback, bool *quit)
{
    const int width = g_job->width(), height = g_job->height(), primarySamples = g_job->spp();
    printf("Beginning pre-process...\n");
    const double preBegin = now();
    preprocess(scene);
    printf("Pre-process complete (%0.1fs elapsed)\n", now() - preBegin);

    std::vector<float> radianceLookup((size_t)3 * width * height, 0.f);
    for (int i = 0; i < primarySamples; i++) {
        const double begin = now();
        sampleImage(radianceLookup, scene);
        const double end = now();
        postwave(scene, i + 1);
        RenderStatus status;
        status.setSample(i + 1);
        callback(status);
        {
            std::lock_guard<std::mutex> guard(image.getLock());
            image.setSpp(i + 1);
            for (int row = 0; row < height; row++) {
                for (int col = 0; col < width; col++) {
                    const size_t index = 3 * ((size_t)row * width + col);
                    image.set(row, col, radianceLookup[index] / (i + 1), radianceLookup[index + 1] / (i + 1), radianceLookup[index + 2] / (i + 1));
                }
            }
            const int maxJ = (int)log2f((float)primarySamples);
            for (int j = 0; j <= maxJ; j++) { if (1 << j == i + 1) { image.saveCheckpoint("auto"); } }
        }
        std::ostringstream line;
        line << "sample: " << i + 1 << "/" << primarySamples << std::fixed << std::setprecision(1) << " (" << (end - begin) << "s elapsed)";
        Logger::line(line.str());
        if (*quit) { return; }
    }
}

// ------------------------------------------------------------------------------------------------ CudaPathTracer
CudaPathTracer::CudaPathTracer(BounceController bounceController, uint64_t seed, int waveSpp, int integrator)
    : m_bounceController(bounceController), m_seed(seed), m_waveSpp(std::max(1, waveSpp)), m_integrator(integrator)
{}

CudaVolumePathTracer::CudaVolumePathTracer(BounceController bounceController, uint64_t seed, int waveSpp)
    : CudaPathTracer(bounceController, seed, waveSpp, PTC_INTEGRATOR_VOLUME_PATH_TRACER)
{}

void CudaPathTracer::sampleImage(std::vector<float> &radianceLookup, Scene &scene)
{
    ptc_ctx *ctx = scene.context(0);
    check(ctx, ptc_set_integrator(ctx, m_integrator), "integrator");
    check(ctx, ptc_render(ctx, m_seed, m_nextSample, 1, m_bounceController.startBounce(), m_bounceController.lastBounce(), radianceLookup.data()),
          "sampleImage");
    m_nextSample++;
    m_samples += (uint64_t)scene.width() * scene.height();
}

// A wave covers up to wave_spp samples per GPU, split over the GPUs in contiguous blocks of global sample indices, each GPU
// accumulating into its own device framebuffer.  The images the reference checkpoints (after 1, 2, 4, ... samples,
// src/integrator.cpp:87-92) that fall inside a wave are snapshots the resolve kernel keeps on the way (ptc_framebuffer_render_
// checkpoints): waves do not end there.  After a wave ONE kernel on GPU 0 per image sums the framebuffers (or snapshots) through peer
// (NVLink) loads and divides by the sample count (K7 resolve); the copies to the host are asynchronous, and the next wave is
// enqueued before the host converts, reports and saves this one -- GPU and host work overlap.  With "denoise_checkpoints" every
// checkpoint of at least 2 samples is also denoised on GPU 0 from the same snapshots (ptc_framebuffer_denoise_begin), its image
// fetched through the same ticket queue, and saved as denoised-auto; the guides are rendered once, after the first wave's renders.
void CudaPathTracer::run(Image &image, Scene &scene, std::function<void(RenderStatus)> callback, bool *quit)
{
    const int width = g_job->width(), height = g_job->height(), primarySamples = g_job->spp();
    if (width != scene.width() || height != scene.height()) { throw std::runtime_error("job resolution differs from the scene's camera"); }
    printf("Beginning pre-process...\n");
    const double preBegin = now();
    preprocess(scene);
    printf("Pre-process complete (%0.1fs elapsed)\n", now() - preBegin);
    if (g_job->adaptive()) { runAdaptive(image, scene, callback, quit); return; }

    const int gpus = scene.gpus();
    const int start = m_bounceController.startBounce(), last = m_bounceController.lastBounce();
    for (int g = 0; g < gpus; g++) {
        check(scene.context(g), ptc_set_integrator(scene.context(g), m_integrator), "integrator");
        if (g_job->denoise()) { check(scene.context(g), ptc_set_option(scene.context(g), "framebuffer_moments", 1), "framebuffer moments"); }
        check(scene.context(g), ptc_framebuffer_clear(scene.context(g)), "framebuffer clear");
    }
    std::vector<ptc_ctx *> peers;
    for (int g = 1; g < gpus; g++) { peers.push_back(scene.context(g)); }
    ptc_ctx *root = scene.context(0);
    std::vector<float> resolved((size_t)3 * width * height);
    const bool denoiseCheckpoints = g_job->denoiseCheckpoints();
    const ptc_denoise_desc desc = PTC_DENOISE_DEFAULTS;
    std::unique_ptr<Image> denoised(denoiseCheckpoints ? new Image(width, height) : nullptr); // the destructor waits for its files

    struct Pending { int spp; uint32_t ticket; bool checkpoint; bool denoised = false; };
    struct Wave { int first = 0, end = 0; std::vector<Pending> images; double enqueued = 0.0; };
    // enqueue the wave that starts at sample `first`: renders on every GPU, then one gather per image wanted from it
    auto enqueue = [&](int first) {
        Wave wave;
        wave.first = first; wave.end = std::min(first + m_waveSpp * gpus, primarySamples);
        wave.enqueued = now();
        std::vector<uint32_t> counts; // power-of-two sample counts inside the wave, the wave's end excluded (that is the live framebuffer)
        for (int c = 1; c < wave.end; c <<= 1) { if (c > first) { counts.push_back((uint32_t)c); } }
        if (counts.size() > PTC_MAX_CHECKPOINTS) { counts.resize(PTC_MAX_CHECKPOINTS); }
        // contiguous blocks: GPU g takes samples [first + g*per, ...); any split gives the same sums up to fp32 order
        const int per = (wave.end - first + gpus - 1) / gpus;
        for (int g = 0; g < gpus; g++) {
            const int from = std::min(first + g * per, wave.end), count = std::min(per, wave.end - from);
            // a GPU without samples in this wave still snapshots its sums: a checkpoint is the sum over all GPUs
            check(scene.context(g), ptc_framebuffer_render_checkpoints(scene.context(g), m_seed, (uint32_t)from, (uint32_t)count, start, last,
                                                                       counts.data(), (uint32_t)counts.size()), "render");
        }
        if (denoiseCheckpoints && first == 0) { enqueueGuides(root, m_seed); }
        // the denoised image of snapshot `snapshot` (-1: the framebuffers), a checkpoint of `spp` samples
        auto denoise = [&](int snapshot, int spp) {
            if (!denoiseCheckpoints || spp < 2) { return; }
            Pending d; d.spp = spp; d.checkpoint = true; d.denoised = true;
            check(root, ptc_framebuffer_denoise_begin(root, peers.data(), (uint32_t)peers.size(), snapshot, (uint32_t)spp, &desc, &d.ticket), "checkpoint denoise");
            wave.images.push_back(d);
        };
        for (size_t i = 0; i < counts.size(); i++) {
            Pending p; p.spp = (int)counts[i]; p.checkpoint = true;
            check(root, ptc_framebuffer_gather_begin(root, peers.data(), (uint32_t)peers.size(), (int)i, counts[i], &p.ticket), "checkpoint gather");
            wave.images.push_back(p);
            denoise((int)i, p.spp);
        }
        Pending p; p.spp = wave.end; p.checkpoint = (wave.end & (wave.end - 1)) == 0;
        check(root, ptc_framebuffer_gather_begin(root, peers.data(), (uint32_t)peers.size(), -1, (uint32_t)wave.end, &p.ticket), "framebuffer gather");
        wave.images.push_back(p);
        if (p.checkpoint) { denoise(-1, p.spp); }
        return wave;
    };

    const double loopBegin = now();
    Wave current = enqueue(0);
    while (current.first < primarySamples) {
        Wave next;
        const bool more = current.end < primarySamples && !*quit;
        if (more) { next = enqueue(current.end); } // the GPUs go on while the host handles the images of `current`
        for (const Pending &p : current.images) {
            check(root, ptc_framebuffer_gather_end(root, p.ticket, resolved.data()), "framebuffer gather");
            if (p.denoised) {
                denoised->setSpp(p.spp);
                denoised->setAll(resolved.data());
                denoised->saveCheckpoint("denoised-auto");
                continue;
            }
            std::lock_guard<std::mutex> guard(image.getLock());
            image.setSpp(p.spp);
            image.setAll(resolved.data());
            if (p.checkpoint) { image.saveCheckpoint("auto"); }
        }
        const double end = now();
        m_samples += (uint64_t)(current.end - current.first) * width * height;
        m_nextSample = (uint32_t)current.end;
        m_renderSeconds = end - loopBegin;
        postwave(scene, current.end);
        RenderStatus status;
        status.setSample(current.end);
        callback(status);
        std::ostringstream line;
        line << "sample: " << current.end << "/" << primarySamples << std::fixed << std::setprecision(1) << " (" << (end - current.enqueued) << "s elapsed)";
        Logger::line(line.str());
        if (!more) { break; }
        current = next;
    }
}

// Adaptive sampling (ptc_adaptive_pass): every pass gives the pixels still active the same number of further samples and ends with
// the stopping test on the device.  After each pass the host fetches the sums and the per-pixel counts and shows the per-pixel means
// S_p / n_p (divided as the K7 resolve divides); a pass that ends at a power-of-two count is saved as that checkpoint.  At the end
// adaptive-spp.exr holds the sample count of every pixel (one fp32 channel Y).
void CudaPathTracer::runAdaptive(Image &image, Scene &scene, std::function<void(RenderStatus)> callback, bool *quit)
{
    const int width = g_job->width(), height = g_job->height(), maxSpp = g_job->spp();
    const size_t pixels = (size_t)width * height;
    ptc_ctx *ctx = scene.context(0);
    check(ctx, ptc_set_integrator(ctx, m_integrator), "integrator");
    ptc_adaptive_desc desc;
    desc.threshold = g_job->adaptiveThreshold();
    desc.min_spp = (uint32_t)g_job->adaptiveMinSpp(); desc.step_spp = (uint32_t)g_job->adaptiveStepSpp(); desc.max_spp = (uint32_t)maxSpp;
    check(ctx, ptc_adaptive_begin(ctx, &desc), "adaptive begin");
    std::vector<float> sums(3 * pixels), resolved(3 * pixels);
    std::vector<uint32_t> counts(pixels);
    const ptc_denoise_desc denoiseDesc = PTC_DENOISE_DEFAULTS;
    std::unique_ptr<Image> denoised(g_job->denoiseCheckpoints() ? new Image(width, height) : nullptr);
    const double loopBegin = now();
    for (int pass = 1;; pass++) {
        const double begin = now();
        uint32_t active = 0, n = 0;
        check(ctx, ptc_adaptive_pass(ctx, m_seed, m_bounceController.startBounce(), m_bounceController.lastBounce(), &active, &n), "adaptive pass");
        check(ctx, ptc_framebuffer_gather(ctx, nullptr, 0, 1, sums.data()), "framebuffer gather");
        check(ctx, ptc_adaptive_state(ctx, counts.data(), nullptr), "adaptive state");
        uint64_t samples = 0;
        for (size_t p = 0; p < pixels; p++) {
            samples += counts[p];
            for (int c = 0; c < 3; c++) { resolved[3 * p + c] = sums[3 * p + c] / (float)counts[p]; }
        }
        const double end = now();
        m_samples = samples;
        m_nextSample = n;
        m_renderSeconds = end - loopBegin;
        {
            std::lock_guard<std::mutex> guard(image.getLock());
            image.setSpp((int)n);
            image.setAll(resolved.data());
            if ((n & (n - 1)) == 0) { image.saveCheckpoint("auto"); }
        }
        if (denoised) {
            if (pass == 1) { enqueueGuides(ctx, m_seed); }
            if ((n & (n - 1)) == 0 && n >= 2) { // n is ignored: the per-pixel counts of the adaptive render are used
                uint32_t ticket = 0;
                check(ctx, ptc_framebuffer_denoise_begin(ctx, nullptr, 0, -1, n, &denoiseDesc, &ticket), "checkpoint denoise");
                check(ctx, ptc_framebuffer_gather_end(ctx, ticket, resolved.data()), "checkpoint denoise");
                denoised->setSpp((int)n);
                denoised->setAll(resolved.data());
                denoised->saveCheckpoint("denoised-auto");
            }
        }
        postwave(scene, (int)n);
        RenderStatus status;
        status.setSample((int)n);
        callback(status);
        std::ostringstream line;
        line << "adaptive pass " << pass << ": " << n << "/" << maxSpp << " spp, " << active << " pixels active" << std::fixed << std::setprecision(1)
             << " (" << (end - begin) << "s elapsed)";
        Logger::line(line.str());
        if (active == 0 || *quit) { break; }
    }
    std::vector<float> plane(pixels); // top scanline first, like every image the job writes
    for (int row = 0; row < height; row++) {
        for (int col = 0; col < width; col++) { plane[(size_t)(height - 1 - row) * width + col] = (float)counts[(size_t)row * width + col]; }
    }
    saveEXR(g_job->outputDirectory() + "adaptive-spp.exr", width, height, {"Y"}, {plane.data()}, false);
}

// "denoise": true -- after run(), from what the contexts still hold: ptc_framebuffer_denoise_begin with the default parameters over
// the sums and second moments of every GPU (an adaptive job: the sums, per-pixel counts and moments of its adaptive render on device
// 0) and the guides of the first min(spp, kGuideSpp) samples on device 0, rendered here again when the checkpoints were denoised (the
// same bytes: this call also fetches their sums, which the checkpoints' asynchronous guide pass did not wait for).
// denoised.exr is written like final.exr (Image: HALF, B,G,R, top scanline first); albedo.exr and normal.exr hold the guide
// buffers' means in fp32, what an external denoiser takes besides the colour.
void CudaPathTracer::writeDenoised(Scene &scene)
{
    const int width = g_job->width(), height = g_job->height();
    const size_t pixels = (size_t)width * height;
    ptc_ctx *ctx = scene.context(0);
    std::vector<ptc_ctx *> peers;
    for (int g = 1; g < scene.gpus(); g++) { peers.push_back(scene.context(g)); }
    const uint32_t aovSpp = guideSpp();
    std::vector<float> albedo(3 * pixels, 0.f), normal(3 * pixels, 0.f);
    check(ctx, ptc_framebuffer_guides(ctx, m_seed, 0, aovSpp, albedo.data(), normal.data(), nullptr, nullptr), "guide buffers");
    const ptc_denoise_desc desc = PTC_DENOISE_DEFAULTS;
    std::vector<float> out(3 * pixels);
    uint32_t ticket = 0;
    // uniform jobs: m_nextSample = the samples every pixel holds
    check(ctx, ptc_framebuffer_denoise_begin(ctx, peers.data(), (uint32_t)peers.size(), -1, m_nextSample, &desc, &ticket), "denoise");
    check(ctx, ptc_framebuffer_gather_end(ctx, ticket, out.data()), "denoise");
    {
        Image denoised(width, height);
        denoised.setAll(out.data());
        denoised.save("denoised"); // the destructor waits for the file
    }
    for (const char *name : {"albedo", "normal"}) {
        const std::vector<float> &sum = name[0] == 'a' ? albedo : normal;
        std::vector<float> planes[3];
        for (int c = 0; c < 3; c++) { planes[c].resize(pixels); }
        for (int row = 0; row < height; row++) {
            for (int col = 0; col < width; col++) {
                const size_t from = (size_t)row * width + col, to = (size_t)(height - 1 - row) * width + col;
                for (int c = 0; c < 3; c++) { planes[c][to] = sum[3 * from + c] / (float)aovSpp; }
            }
        }
        saveEXR(g_job->outputDirectory() + name + ".exr", width, height, {"B", "G", "R"}, {planes[2].data(), planes[1].data(), planes[0].data()}, false);
        printf("Saved exr file. [ %s%s.exr ] \n", g_job->outputDirectory().c_str(), name);
    }
}

} // namespace pathed
