// Job, BounceController, Logger: the configuration side of the host API (pathed.hpp).
// Behaviour follows /root/reference/include/job.h:13-75, src/job.cpp:25-97, src/bounce_controller.cpp, src/logger.cpp.
#include "pathed.hpp"

#include "json.hpp"

#include <algorithm>
#include <cerrno>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <iostream>
#include <iterator>
#include <sstream>
#include <sys/stat.h>

namespace pathed {

Job *g_job = nullptr;

BounceController::BounceController(int startBounce, int lastBounce) : m_startBounce(startBounce), m_lastBounce(lastBounce)
{
    // the reference asserts (compiled out, SURVEY F8); the C ABI rejects the same windows with PTC_ERR_INVALID
}

bool BounceController::checkCounts(int bounce) const
{
    if (m_startBounce > bounce) { return false; }
    return !checkDone(bounce);
}

bool BounceController::checkDone(int bounce) const
{
    if (m_lastBounce == -1) { return false; }
    return bounce > m_lastBounce;
}

BounceController BounceController::copyAfterBounce() const
{
    const int start = std::max(0, m_startBounce - 1);
    const int last = m_lastBounce == -1 ? -1 : std::max(0, m_lastBounce - 1);
    return BounceController(start, last);
}

static Json parseJobFile(std::istream &jobFile)
{
    const std::string text((std::istreambuf_iterator<char>(jobFile)), std::istreambuf_iterator<char>());
    return Json::parse(text);
}

Job::Job(std::istream &jobFile)
    : m_json(new Json(parseJobFile(jobFile))),
      m_bounceController((*m_json)["startBounce"].asInt(), (*m_json)["lastBounce"].asInt())
{
    const Json &denoiseKey = (*m_json)["denoise"];
    if (!denoiseKey.isNull() && !denoiseKey.isBool()) { throw std::runtime_error("denoise must be true or false"); }
    if (denoise() && spp() < 2) { throw std::runtime_error("denoise needs spp >= 2: the filter estimates each pixel's variance"); }
    const Json &checkpointsKey = (*m_json)["denoise_checkpoints"];
    if (!checkpointsKey.isNull() && !checkpointsKey.isBool()) { throw std::runtime_error("denoise_checkpoints must be true or false"); }
    if (denoiseCheckpoints() && !denoise()) { throw std::runtime_error("denoise_checkpoints needs \"denoise\": true"); }
    if (!adaptive()) { return; }
    const double threshold = (*m_json)["adaptive_threshold"].asNumber();
    if (!(threshold > 0.0) || !std::isfinite(threshold)) { throw std::runtime_error("adaptive_threshold must be a number > 0"); }
    for (const char *key : {"adaptive_min_spp", "adaptive_step_spp"}) {
        const Json &value = (*m_json)[key];
        if (!value.isNull() && (!value.isNumber() || value.asNumber() != std::floor(value.asNumber()))) { throw std::runtime_error(std::string(key) + " must be an integer"); }
    }
    if (adaptiveMinSpp() < 2) { throw std::runtime_error("adaptive_min_spp must be >= 2"); }
    if (adaptiveStepSpp() < 1) { throw std::runtime_error("adaptive_step_spp must be >= 1"); }
    if (spp() < adaptiveMinSpp()) { throw std::runtime_error("spp (the most samples a pixel gets) must be >= adaptive_min_spp"); }
    if (gpus() != 1) { throw std::runtime_error("adaptive sampling runs on one GPU: set \"gpus\": 1 or drop adaptive_threshold"); }
}

Job::~Job() {}

bool Job::showUI() const { return (*m_json)["showUI"].asBool(); }
bool Job::force() const { return (*m_json)["force"].isBool() && (*m_json)["force"].asBool(); }
int Job::width() const { return (*m_json)["width"].asInt(); }
int Job::height() const { return (*m_json)["height"].asInt(); }

int Job::spp() const
{
    const int spp = (*m_json)["spp"].asInt();
    return spp > 0 ? spp : 9999999;
}

std::string Job::outputDirectory() const { return (*m_json)["output_directory"].asString() + "/"; }
std::string Job::outputName() const { return (*m_json)["output_name"].asString(); }
std::string Job::scene() const { return (*m_json)["scene"].asString(); }

int Job::gpus() const { return (*m_json)["gpus"].isNumber() ? std::max(1, (*m_json)["gpus"].asInt()) : 1; }
uint64_t Job::seed() const { return (*m_json)["seed"].isNumber() ? (uint64_t)(*m_json)["seed"].asNumber() : 0x5EEDull; }
int Job::waveSpp() const { return (*m_json)["wave_spp"].isNumber() ? std::max(1, (*m_json)["wave_spp"].asInt()) : 64; }
bool Job::denoise() const { return (*m_json)["denoise"].isBool() && (*m_json)["denoise"].asBool(); }
bool Job::denoiseCheckpoints() const { return (*m_json)["denoise_checkpoints"].isBool() && (*m_json)["denoise_checkpoints"].asBool(); }
bool Job::adaptive() const { return !(*m_json)["adaptive_threshold"].isNull(); }
float Job::adaptiveThreshold() const { return adaptive() ? (float)(*m_json)["adaptive_threshold"].asNumber() : 0.f; }
int Job::adaptiveMinSpp() const { return (*m_json)["adaptive_min_spp"].isNumber() ? (*m_json)["adaptive_min_spp"].asInt() : 16; }
int Job::adaptiveStepSpp() const { return (*m_json)["adaptive_step_spp"].isNumber() ? (*m_json)["adaptive_step_spp"].asInt() : 16; }

void Job::init()
{
    const std::string directory = outputDirectory();
    int result = mkdir(directory.c_str(), S_IRWXU | S_IRWXG | S_IROTH | S_IXOTH);
    if (result == -1) {
        if (errno == EEXIST) { std::cout << "Output directory already exists: " << directory << std::endl; }
        else { std::cout << "Failed to create: " << directory << std::endl; }
        if (!force()) { exit(1); }
    }
    result = mkdir(visualizationDirectory().c_str(), S_IRWXU | S_IRWXG | S_IROTH | S_IXOTH);
    if (result == -1) {
        std::cout << "Failed to create: " << visualizationDirectory() << std::endl;
        if (!force()) { exit(1); }
    }
    std::ofstream report(directory + "/report.json");
    report << m_json->dump(4) << std::endl;
}

std::shared_ptr<Integrator> Job::integrator() const
{
    const std::string name = (*m_json)["integrator"].asString();
    if (name == "PathTracer") { return std::make_shared<CudaPathTracer>(m_bounceController, seed(), waveSpp()); }
    if (name == "VolumePathTracer") { return std::make_shared<CudaVolumePathTracer>(m_bounceController, seed(), waveSpp()); }
    // the other eleven integrators of src/job.cpp:65-95 are research code outside the accelerated path
    throw "Unimplemented";
}

void Logger::line(const std::string &line)
{
    const std::string directory = g_job ? g_job->outputDirectory() : std::string();
    std::cout << "[" << directory << "] " << line << std::endl;
}

} // namespace pathed
