// Denoising (ptc_render_aovs, ptc_denoise, ptc_framebuffer_guides, ptc_framebuffer_denoise_begin; DESIGN §10).  Included by
// pathed_cuda.cu after the probe kernels: it traces with the same camera, traversal and Intersection code as the path tracer and
// ptc_intersect_full.  The host-input filter (ptc_denoise) and the device-resident one build their records with the same functions
// (colourRecord, writeGuideRecord), so the two give the same bytes for the same sums.
//
// Guide buffers.  aovKernel re-traces the first hit of the camera ray the path tracer traces for (seed, pixel, sample): draws 0 and
// 1 of vertex 0 jitter the ray exactly as generateKernel / volumePathKernel do, and the closest hit is intersectFullKernel's.  One
// thread per pixel adds its samples in sample order into the (uploaded) buffers, so a call over samples 0 .. 7 followed by one over
// 8 .. 15 gives the bytes of one call over 0 .. 15.
//
// The filter is the spatial part of SVGF (Schied et al., HPG 2017) with an albedo term, in fp32 (--fmad=false: every product and
// sum is rounded on its own, in the order written here and in DESIGN §10):
//   inputs per pixel   n = counts[p] (or spp); c = S / n; var_k = (M_k - n (c_k c_k)) / (n - 1), negative -> 0;
//                      v = ((var_r + var_g) + var_b) / (3 n)  (variance of the mean); a = albedo / aov_spp;
//                      N = normal / sqrt(normal . normal), 0 when that is 0; z = depth / max(hits, 1)
//   luminance          l(c) = (0.2126 c_r + 0.7152 c_g) + 0.0722 c_b, of the iteration's input colour
//   iteration i        h = 2^i; ~v_p = sum k3 v_q / sum k3 over the 3x3 neighbours q of p (step 1) that are in the image and
//                      finite, k3 = (1/4, 1/2, 1/4) per axis; taps q = p + h (dx, dy), dx, dy in -2 .. 2 (dy outer), in the image
//                      and finite, with k5 = (1/16, 1/4, 3/8, 1/4, 1/16) per axis:
//                      w = ((k5_dx k5_dy) exp(((-|l_p - l_q| / (sigma_l sqrt(~v_p) + eps)) - |a_p - a_q|_1 / sigma_a)
//                                             - |z_p - z_q| / ((sigma_z h) max(z_p, z_q, eps)))) g(N_p, N_q)
//                      g = max(0, N_p . N_q)^sigma_n; 1 when both normals are 0, 0 when exactly one is
//                      c' = sum w c_q / sum w, v' = sum (w w) v_q / (sum w)^2
//   non-finite pixels  a pixel whose c or v is not finite has weight 0 as a neighbour and passes through unchanged.
// No atomics: every output is one thread's fixed-order sum, so two calls give the same bytes.
#pragma once

// ------------------------------------------------------------------------------------------------ guide buffers
__global__ void __launch_bounds__(128) aovKernel(DScene scene, uint64_t seed, uint32_t firstSample, uint32_t nSpp, float *albedo, float *normal,
                                                 float *depth, uint32_t *hits)
{
    const uint32_t width = (uint32_t)scene.width, nPixels = width * (uint32_t)scene.height;
    for (uint32_t pixel = blockIdx.x * blockDim.x + threadIdx.x; pixel < nPixels; pixel += gridDim.x * blockDim.x) {
        const int row = (int)(pixel / width), col = (int)(pixel % width);
        V3 a = mk(albedo[3 * (size_t)pixel], albedo[3 * (size_t)pixel + 1], albedo[3 * (size_t)pixel + 2]);
        V3 n = mk(normal[3 * (size_t)pixel], normal[3 * (size_t)pixel + 1], normal[3 * (size_t)pixel + 2]);
        float z = depth[pixel];
        uint32_t count = hits[pixel];
        for (uint32_t s = 0; s < nSpp; s++) {
            Rng rng;
            rng.initPhilox(seed, pixel, firstSample + s);
            rng.beginVertex(0);
            const float jitterX = rng.next() - 0.5f; // generateKernel's draws
            const float jitterY = rng.next() - 0.5f;
            V3 o, d;
            cameraRay(scene, row + jitterY, col + jitterX, o, d);
            RayHit h;
            if (!traverseBVH<false, false>(scene.bvh, o.x, o.y, o.z, d.x, d.y, d.z, PTC_TNEAR, PTC_TFAR, h, nullptr)) { continue; }
            Isect is;
            makeIsect(scene, o, d, h, is);
            const DMaterial &m = scene.materials[is.material];
            const bool diffuse = m.type == PTC_LAMBERTIAN || m.type == PTC_OREN_NAYAR || m.type == PTC_PLASTIC;
            a = a + (diffuse ? lambertAlbedo(m, is) : mk(1.f, 1.f, 1.f));
            n = n + is.ns;
            z += h.t;
            count++;
        }
        albedo[3 * (size_t)pixel] = a.x; albedo[3 * (size_t)pixel + 1] = a.y; albedo[3 * (size_t)pixel + 2] = a.z;
        normal[3 * (size_t)pixel] = n.x; normal[3 * (size_t)pixel + 1] = n.y; normal[3 * (size_t)pixel + 2] = n.z;
        depth[pixel] = z;
        hits[pixel] = count;
    }
}

// ------------------------------------------------------------------------------------------------ filter
// Records: colour = float4 (c rgb, v), 16 B, ping-pong; guide = two float4 (a rgb, z | N xyz, 0), 32 B aligned = one sector.
struct DenoiseInputs {
    const float *sums, *moments, *albedo, *normal, *depth;
    const uint32_t *counts, *hits; // counts null: every pixel has `spp`
    uint32_t spp, aovSpp, nPixels;
};

// The colour record of one pixel from its sums S, second moments M and sample count n
__device__ __forceinline__ float4 colourRecord(const float S[3], const float M[3], float n)
{
    float c[3], var[3];
    for (int k = 0; k < 3; k++) {
        c[k] = S[k] / n;
        var[k] = (M[k] - n * (c[k] * c[k])) / (n - 1.f);
        if (var[k] < 0.f) { var[k] = 0.f; } // keeps a NaN
    }
    return make_float4(c[0], c[1], c[2], ((var[0] + var[1]) + var[2]) / (3.f * n));
}

// The guide record of pixel p from the guide sums over aovSpp samples
__device__ __forceinline__ void writeGuideRecord(const float *albedo, const float *normal, const float *depth, const uint32_t *hits, uint32_t aovSppCount,
                                                 uint32_t p, float4 *guide)
{
    const float aovSpp = (float)aovSppCount;
    const float nx = normal[3 * (size_t)p], ny = normal[3 * (size_t)p + 1], nz = normal[3 * (size_t)p + 2];
    const float len2 = (nx * nx + ny * ny) + nz * nz;
    const float len = len2 > 0.f ? sqrtf(len2) : 0.f;
    guide[2 * (size_t)p] = make_float4(albedo[3 * (size_t)p] / aovSpp, albedo[3 * (size_t)p + 1] / aovSpp, albedo[3 * (size_t)p + 2] / aovSpp,
                                       depth[p] / (float)max(hits[p], 1u));
    guide[2 * (size_t)p + 1] = len > 0.f ? make_float4(nx / len, ny / len, nz / len, 0.f) : make_float4(0.f, 0.f, 0.f, 0.f);
}

__global__ void __launch_bounds__(256) denoisePrepareKernel(DenoiseInputs in, float4 *colour, float4 *guide)
{
    for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < in.nPixels; p += gridDim.x * blockDim.x) {
        colour[p] = colourRecord(in.sums + 3 * (size_t)p, in.moments + 3 * (size_t)p, (float)(in.counts ? in.counts[p] : in.spp));
        writeGuideRecord(in.albedo, in.normal, in.depth, in.hits, in.aovSpp, p, guide);
    }
}

// ptc_framebuffer_guides: the guide records from the device guide sums of aovKernel
__global__ void __launch_bounds__(256) denoiseGuideKernel(const float *albedo, const float *normal, const float *depth, const uint32_t *hits, uint32_t aovSpp,
                                                          uint32_t nPixels, float4 *guide)
{
    for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < nPixels; p += gridDim.x * blockDim.x) { writeGuideRecord(albedo, normal, depth, hits, aovSpp, p, guide); }
}

// ptc_framebuffer_denoise_begin: the colour records of the sums and second moments of root + peers, each summed in
// gatherResolveKernel's order (set.fb[0] first, then the peers in turn); n = counts[p] (an adaptive root) or spp
__global__ void __launch_bounds__(256) denoiseGatherKernel(FramebufferSet sums, FramebufferSet moments, const uint32_t *counts, uint32_t spp, uint32_t nPixels,
                                                           float4 *colour)
{
    for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < nPixels; p += gridDim.x * blockDim.x) {
        float S[3], M[3];
        for (int k = 0; k < 3; k++) {
            const size_t i = 3 * (size_t)p + k;
            S[k] = sums.fb[0][i]; M[k] = moments.fb[0][i];
            for (int g = 1; g < sums.count; g++) { S[k] += sums.fb[g][i]; M[k] += moments.fb[g][i]; }
        }
        colour[p] = colourRecord(S, M, (float)(counts ? counts[p] : spp));
    }
}

// rgb of the last a-trous output, as ptc_denoise hands it out
__global__ void __launch_bounds__(256) denoisePackKernel(const float4 *colour, float *out, uint32_t nPixels)
{
    for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < nPixels; p += gridDim.x * blockDim.x) {
        const float4 c = colour[p];
        out[3 * (size_t)p] = c.x; out[3 * (size_t)p + 1] = c.y; out[3 * (size_t)p + 2] = c.z;
    }
}

__device__ __forceinline__ bool finiteRecord(float4 r) { return isfinite(r.x) && isfinite(r.y) && isfinite(r.z) && isfinite(r.w); }
__device__ __forceinline__ float luminance(float4 c) { return (0.2126f * c.x + 0.7152f * c.y) + 0.0722f * c.z; }

struct DenoiseParams { float sigmaL, sigmaN, sigmaZ, sigmaA, eps; };

// One a-trous level at step h; the variance prefilter ~v_p is taken from the same input (3x3, step 1: L1 hits of the 5x5 taps' rows)
__global__ void __launch_bounds__(256) denoiseAtrousKernel(const float4 *__restrict__ in, float4 *__restrict__ out, const float4 *__restrict__ guide,
                                                           int width, int height, int h, DenoiseParams dp)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= width || y >= height) { return; }
    const size_t p = (size_t)y * width + x;
    const float4 cp = __ldg(in + p);
    if (!finiteRecord(cp)) { out[p] = cp; return; }
    const float k3[3] = {0.25f, 0.5f, 0.25f};
    float vs = 0.f, ks = 0.f;
    for (int dy = -1; dy <= 1; dy++) {
        const int qy = y + dy;
        if (qy < 0 || qy >= height) { continue; }
        for (int dx = -1; dx <= 1; dx++) {
            const int qx = x + dx;
            if (qx < 0 || qx >= width) { continue; }
            const float4 cq = __ldg(in + (size_t)qy * width + qx);
            if (!finiteRecord(cq)) { continue; }
            const float k = k3[dx + 1] * k3[dy + 1];
            vs += k * cq.w; ks += k;
        }
    }
    const float vt = vs / ks;
    const float4 ga = __ldg(guide + 2 * p), gn = __ldg(guide + 2 * p + 1);
    const bool pZero = gn.x == 0.f && gn.y == 0.f && gn.z == 0.f;
    const float lp = luminance(cp);
    const float denomL = dp.sigmaL * sqrtf(vt) + dp.eps;
    const float stepZ = dp.sigmaZ * (float)h;
    const float k5[5] = {1.f / 16.f, 0.25f, 0.375f, 0.25f, 1.f / 16.f};
    float sw = 0.f, sr = 0.f, sg = 0.f, sb = 0.f, sv = 0.f;
    for (int dy = -2; dy <= 2; dy++) {
        const int qy = y + h * dy;
        if (qy < 0 || qy >= height) { continue; }
        for (int dx = -2; dx <= 2; dx++) {
            const int qx = x + h * dx;
            if (qx < 0 || qx >= width) { continue; }
            const size_t q = (size_t)qy * width + qx;
            const float4 cq = __ldg(in + q);
            if (!finiteRecord(cq)) { continue; }
            const float4 qa = __ldg(guide + 2 * q), qn = __ldg(guide + 2 * q + 1);
            const bool qZero = qn.x == 0.f && qn.y == 0.f && qn.z == 0.f;
            float g;
            if (pZero || qZero) { g = pZero && qZero ? 1.f : 0.f; }
            else { g = powf(fmaxf(0.f, (gn.x * qn.x + gn.y * qn.y) + gn.z * qn.z), dp.sigmaN); }
            const float dl = fabsf(lp - luminance(cq)) / denomL;
            const float da = ((fabsf(ga.x - qa.x) + fabsf(ga.y - qa.y)) + fabsf(ga.z - qa.z)) / dp.sigmaA;
            const float dz = fabsf(ga.w - qa.w) / (stepZ * fmaxf(fmaxf(ga.w, qa.w), dp.eps));
            const float w = ((k5[dx + 2] * k5[dy + 2]) * expf(((-dl) - da) - dz)) * g;
            sw += w;
            sr += w * cq.x; sg += w * cq.y; sb += w * cq.z;
            sv += (w * w) * cq.w;
        }
    }
    out[p] = make_float4(sr / sw, sg / sw, sb / sw, sv / (sw * sw));
}
