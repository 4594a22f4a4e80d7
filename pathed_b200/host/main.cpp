// pathed — command-line renderer, the drop-in for the reference's `./pathed [job.json]` (/root/reference/app/main.cpp:43-126)
// without the nanogui window: job.json -> parseScene -> Job::integrator() -> Integrator::run -> EXR checkpoints.
//
//   pathed [job.json] [--root DIR]
// --root plays the part of the reference's chdir("..") (app/main.cpp:60): scene and asset paths are relative to it.
#include "pathed.hpp"

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <iostream>
#include <unistd.h>

using namespace pathed;

int main(int argc, char *argv[])
{
    printf("Hello, world!\n");
    std::string jobPath = "job.json", root;
    for (int i = 1; i < argc; i++) {
        if (!strcmp(argv[i], "--root") && i + 1 < argc) { root = argv[++i]; }
        else { jobPath = argv[i]; }
    }
    std::ifstream jobFile(jobPath);
    if (!jobFile) { std::cout << "Failed to open job file: " << jobPath << std::endl; return 1; }
    try {
        Job job(jobFile);
        g_job = &job;
        if (!root.empty() && chdir(root.c_str()) != 0) { std::cout << "Failed to enter: " << root << std::endl; return 1; }
        job.init();
        printf("Job: {spp: %d}\n", job.spp());
        Image image(job.width(), job.height());
        const auto buildBegin = std::chrono::steady_clock::now();
        std::unique_ptr<Scene> scene = parseSceneForJob(job, "");
        const double buildSeconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - buildBegin).count();
        printf("Scene ready on %d GPU(s): %u lights (%0.2fs parse + BVH build + upload)\n", scene->gpus(), scene->lightCount(), buildSeconds);
        std::shared_ptr<Integrator> integrator = job.integrator();
        bool quit = false;
        integrator->run(image, *scene, [](RenderStatus) {}, &quit);
        image.save(job.outputName());
        if (CudaPathTracer *tracer = dynamic_cast<CudaPathTracer *>(integrator.get())) {
            printf("PATHED_RESULT {\"samples\": %llu, \"render_wall_s\": %.6f, \"msamples_per_s\": %.3f, \"gpus\": %d}\n",
                   (unsigned long long)tracer->samplesRendered(), tracer->renderSeconds(),
                   tracer->samplesRendered() / std::max(tracer->renderSeconds(), 1e-9) * 1e-6, scene->gpus());
            if (job.denoise()) { tracer->writeDenoised(*scene); } // after final.exr was handed to the writer
        }
    } catch (const std::exception &e) {
        std::cout << "error: " << e.what() << std::endl;
        return 1;
    } catch (const char *message) { // Job::integrator(): throw "Unimplemented" (src/job.cpp:96)
        std::cout << "error: " << message << std::endl;
        return 1;
    }
    return 0;
}
