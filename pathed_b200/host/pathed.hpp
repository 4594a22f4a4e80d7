// Host API of the drop-in: the classes a Pathed caller (app/main.cpp) touches, with the reference's
// names, argument meaning and error behaviour, re-based on the C ABI of include/pathed_cuda.h.
//
//   reference                                         here
//   Job            include/job.h:13-75, src/job.cpp   pathed::Job         (same keys; + optional "gpus", "seed", "wave_spp")
//   BounceController  src/bounce_controller.cpp       pathed::BounceController
//   Image          include/image.h, src/image.cpp     pathed::Image       (raw fp32 flipped, 8-bit preview, EXR HALF B,G,R)
//   Scene          include/scene.h:83-130             pathed::Scene       (testIntersect / testOcclusion over the GPU BVH)
//   Integrator     include/integrator.h:16-55         pathed::Integrator  (run / preprocess / sampleImage)
//   PathTracer     include/path_tracer.h              pathed::CudaPathTracer (what Job::integrator() returns for "PathTracer")
//   RenderStatus   include/render_status.h            pathed::RenderStatus (sample count only: no per-pixel debug paths on the GPU)
//   Logger         src/logger.cpp                     pathed::Logger
//
// There is no CPU rendering path behind these classes: every query and every sample goes to libpathed_cuda.so.
#pragma once

#include "scene_description.hpp"

#include <functional>
#include <future>
#include <istream>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

namespace pathed {

class Json;
class Integrator;

// src/bounce_controller.cpp:6-25
class BounceController {
public:
    BounceController(int startBounce, int lastBounce);
    bool checkCounts(int bounce) const;
    bool checkDone(int bounce) const;
    int startBounce() const { return m_startBounce; }
    int lastBounce() const { return m_lastBounce; }
    BounceController copyAfterBounce() const;

private:
    int m_startBounce, m_lastBounce;
};

// include/job.h:13-75.  Accessors throw std::runtime_error where nlohmann's get<T>() would throw.
class Job {
public:
    explicit Job(std::istream &jobFile);
    ~Job();
    Job(const Job &) = delete;
    Job &operator=(const Job &) = delete;

    void init(); // mkdir output + visualization directories, write report.json; exit(1) unless "force" (src/job.cpp:33-63)

    bool showUI() const;
    bool force() const;
    int width() const;
    int height() const;
    int spp() const; // <= 0 -> 9999999
    std::string outputDirectory() const; // with trailing '/'
    std::string outputName() const;
    std::string scene() const;
    std::string visualizationDirectory() const { return outputDirectory() + "visualization/"; }
    int startBounce() const { return m_bounceController.startBounce(); }
    int lastBounce() const { return m_bounceController.lastBounce(); }
    BounceController bounceController() const { return m_bounceController; }

    // additions (optional keys, defaults keep the reference's behaviour)
    int gpus() const;          // "gpus": number of devices the spp are split over (default 1)
    uint64_t seed() const;     // "seed": Philox key (default 0x5EED; the reference seeds from random_device)
    int waveSpp() const;       // "wave_spp": max samples per pixel per device call between callbacks (default 64)
    // adaptive sampling (ptc_adaptive_*): present "adaptive_threshold" (tau > 0) makes the job adaptive, "spp" is then the most
    // samples a pixel gets; "adaptive_min_spp" (>= 2, <= spp, default 16) samples every pixel gets, "adaptive_step_spp" (>= 1,
    // default 16) samples per later pass.  Checked by the constructor, like "gpus" == 1 (adaptive sampling runs on one GPU)
    bool adaptive() const;
    float adaptiveThreshold() const;
    int adaptiveMinSpp() const;
    int adaptiveStepSpp() const;
    // "denoise": true (default false) also writes denoised.exr (ptc_denoise of the final sums), albedo.exr and normal.exr (the
    // guide buffers it used); any value but a bool is refused by the constructor, and so is true with spp < 2 (the filter needs
    // each pixel's variance)
    bool denoise() const;
    // "denoise_checkpoints": true (default false; needs "denoise": true, any value but a bool is refused) also denoises every
    // checkpoint of at least 2 samples on the devices: denoised-auto.exr and denoised-auto-%05dspp.exr, like auto-*.exr
    bool denoiseCheckpoints() const;

    // string -> integrator (src/job.cpp:65-97); anything but "PathTracer" throws const char* "Unimplemented"
    std::shared_ptr<Integrator> integrator() const;

private:
    std::unique_ptr<Json> m_json;
    BounceController m_bounceController;
};

extern Job *g_job; // include/globals.h:7

// src/logger.cpp:8-16
struct Logger {
    static void line(const std::string &line);
};

// include/render_status.h:9-34 without the UI-only debug payloads
class RenderStatus {
public:
    void setSample(int sample) { m_sample = sample; }
    int sample() const { return m_sample; }

private:
    int m_sample = 0;
};

// include/image.h, src/image.cpp
class Image {
public:
    Image(int width, int height);
    ~Image();
    void flush();                                          // waits until every file handed to the writer thread is on disk
    void set(int row, int col, float r, float g, float b); // row 0 = bottom scanline (Q14)
    void setAll(const float *rgb);                         // set(row, col, ...) for every pixel of a row-major 3*W*H buffer, on all host threads
    void save(const std::string &filestem);           // <outdir>/<stem>.exr
    void saveCheckpoint(const std::string &filestem); // + <outdir>/<stem>-%05dspp.exr
    void write(const std::string &filename);          // 24-bit BMP of the 8-bit preview
    const std::vector<unsigned char> &data() { return m_data; }
    const std::vector<float> &raw() const { return m_raw; } // top scanline first
    std::mutex &getLock() { return m_lock; }
    void setSpp(int spp) { m_spp = spp; }
    int width() const { return m_width; }
    int height() const { return m_height; }

private:
    void save(const std::string &filestem, bool checkpoint);
    int m_height, m_width, m_spp;
    std::vector<unsigned char> m_data;
    std::vector<float> m_raw;
    std::mutex m_lock;
    std::shared_future<void> m_lastWrite; // files are written in call order by a background task chain
};

struct Ray {
    float origin[3];
    float direction[3];
};

// include/intersection.h:13-24 (material is the id the scene description assigned)
struct Intersection {
    bool hit = false;
    float t = 0.f;
    float point[3] = {0, 0, 0}, woWorld[3] = {0, 0, 0}, normal[3] = {0, 0, 0}, shadingNormal[3] = {0, 0, 0}, uv[2] = {0, 0};
    uint32_t material = PTC_INVALID_ID;
};

// The committed scene on one or more GPUs (one ptc_ctx per device, scene replicated).
class Scene {
public:
    // `first`: an already created context for device 0 (ownership passes to the Scene); null = create one
    // reservePaths: path state the further devices allocate while they are set up (ptc_reserve_paths; the first one did it while the scene was parsed)
    Scene(const SceneDescription &description, int gpus = 1, ptc_ctx *first = nullptr, uint64_t reservePaths = 0);
    ~Scene();
    Scene(const Scene &) = delete;
    Scene &operator=(const Scene &) = delete;

    Intersection testIntersect(const Ray &ray) const;      // include/scene.h:94
    bool testOcclusion(const Ray &ray, float maxT) const;   // include/scene.h:97
    int gpus() const { return (int)m_contexts.size(); }
    ptc_ctx *context(int device = 0) const { return m_contexts[(size_t)device]; }
    int width() const { return m_width; }
    int height() const { return m_height; }
    uint32_t lightCount() const;

private:
    std::vector<ptc_ctx *> m_contexts;
    int m_width, m_height;
    mutable std::mutex m_queryLock; // a context is not thread-safe; the reference's queries are re-entrant
};

// Scene parseScene(std::ifstream&) of the reference (src/scene_parser.cpp:140): resolution from g_job
std::unique_ptr<Scene> parseSceneForJob(const Job &job, const std::string &rootDirectory);

// include/integrator.h:16-55
class Integrator {
public:
    virtual ~Integrator() {}
    virtual void run(Image &image, Scene &scene, std::function<void(RenderStatus)> callback, bool *quit);
    virtual void preprocess(const Scene &) {}
    virtual void postwave(const Scene &, int /*sample*/) {}
    // one spp per call, accumulated into radianceLookup (src/sample_integrator.cpp:80-113)
    virtual void sampleImage(std::vector<float> &radianceLookup, Scene &scene) = 0;
};

// "PathTracer": the surface path tracer (src/path_tracer.cpp) on the GPU
class CudaPathTracer : public Integrator {
public:
    explicit CudaPathTracer(BounceController bounceController, uint64_t seed = 0x5EED, int waveSpp = 64,
                            int integrator = 0 /* PTC_INTEGRATOR_PATH_TRACER */);
    // device-resident spp loop: framebuffers stay in HBM between checkpoints, spp split over scene.gpus() devices,
    // one peer-memory reduce + resolve per callback (replaces the per-wave host loop of src/integrator.cpp:42-105)
    void run(Image &image, Scene &scene, std::function<void(RenderStatus)> callback, bool *quit) override;
    void sampleImage(std::vector<float> &radianceLookup, Scene &scene) override;

    double renderSeconds() const { return m_renderSeconds; } // wall time inside run() spent rendering + reducing
    uint64_t samplesRendered() const { return m_samples; }
    // job.json "denoise": denoised.exr, albedo.exr and normal.exr from the render run() left on the devices.  Called after the job's
    // image is saved, so that a failure here cannot cost the job final.exr
    void writeDenoised(Scene &scene);

private:
    BounceController m_bounceController;
    uint64_t m_seed;
    int m_waveSpp;
    int m_integrator; // which L() the device runs (ptc_set_integrator)
    uint32_t m_nextSample = 0;
    double m_renderSeconds = 0.0;
    uint64_t m_samples = 0;
    // the job's adaptive render: passes on device 0 until every pixel has stopped
    void runAdaptive(Image &image, Scene &scene, std::function<void(RenderStatus)> callback, bool *quit);
};

// "VolumePathTracer" (src/volume_path_tracer.cpp): the same device-resident loop with the participating-media L()
class CudaVolumePathTracer : public CudaPathTracer {
public:
    explicit CudaVolumePathTracer(BounceController bounceController, uint64_t seed = 0x5EED, int waveSpp = 64);
};

} // namespace pathed
