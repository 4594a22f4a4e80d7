// libpathed_cuda.so — sm_100a wavefront path tracer behind the C ABI of include/pathed_cuda.h.
//
// Wavefront stages per wave of P = pixels x spp_per_wave paths (SURVEY §2.5 K1..K7):
//   generate  K1  camera rays (Camera::generateRay, src/camera.cpp:32-55) + path-state initialisation
//   extend    K2  closest hit over the compressed 8-wide BVH (rtcIntersect1 via Scene::testIntersect)
//   shadow    K3  any hit for the NEE shadow rays (rtcOccluded1 via Scene::testOcclusion)
//   logic     K5/K6  finalise the previous vertex's direct lighting (NEE + MIS'd BSDF hit / environment miss), update the
//             throughput, terminate; survivors are binned by the material class of the surface they hit
//   material  K4  one kernel per material class present in the scene (compile-time specialised BSDF code, coherent
//             warps): build the Intersection, sample the BSDF, set up NEE, append to the next extend / shadow queues
//             (all queue appends are warp-aggregated: ballot + popc + one atomic per warp)
//   resolve   K7  sum the wave's per-sample radiance into the fp32 framebuffer in sample order
// The MIS probe ray (src/path_tracer.cpp:175) and the continuation ray (:44) are the same ray: traced once.
// All queue sizes live on the device; a wave is a fixed launch sequence with no host synchronisation.
#include "bvh.h"
#include "shading.cuh"
#include "volume.cuh"

#include <cuda_runtime.h>
#include <cub/device/device_select.cuh>

#include <algorithm>
#include <cstdio>
#include <cstring>
#include <functional>
#include <optional>
#include <string>
#include <chrono>
#include <vector>

using namespace ptc;

// ================================================================================================ device state
#define PTC_MATERIAL_CLASSES 7 /* PTC_LAMBERTIAN .. PTC_PASSTHROUGH */
// Path state.  A path does not keep its slot: the material stage of vertex k writes the state of every path that goes on to the
// slot it gets in the NEXT bounce's ray list (one warp-aggregated append), so the paths alive at bounce k always occupy slots
// 0 .. n_k - 1 of the state arrays and every stage reads and writes dense, coalesced records however few paths survive (replaces
// the implicit `break`s of PathTracer::L, src/path_tracer.cpp:45,56-58; the slot a path started in -- pixel and sample, the Philox
// key and the place its radiance is written -- travels with it in the spare word of the ray record).
// Layout rule: what one stage reads or writes TOGETHER is one 32-byte record moved by ONE 256-bit instruction (sm_100:
// ld/st.global.v8.f32), what stages touch separately is a 16-byte array of its own -- so that every store covers whole 32-byte
// sectors (a 16-byte store into half of a sector that is not in L2 costs a DRAM read to fill the other half plus a full-sector
// write; measured on the earlier paired layout: +32 B read per hit record, per throughput record, ...).  Fields that a later kernel
// still reads at the old slots are double-buffered (current / next); the rest are written at the new slot only after their last
// reader of the old slot finished.
// Path state is streamed: every record is read once and written once per stage, 15 GB per wave, while the scene data the same
// kernels gather from (BVH, per-triangle shading records, environment map and its CDFs: ~160 MB for the dragon workload) is re-used
// and should own the 126 MB L2.  PTC_STREAM_STATE = 1 issues the path-state accesses with the evict-first policy (ld.global.cs /
// st.global.cs), so they pass through L2 without displacing the scene.
#ifndef PTC_STREAM_STATE
#define PTC_STREAM_STATE 1
#endif
template <typename T> __device__ __forceinline__ T streamLoad(const T *p) { return PTC_STREAM_STATE ? __ldcs(p) : *p; }
template <typename T> __device__ __forceinline__ void streamStore(T *p, T v) { if (PTC_STREAM_STATE) { __stcs(p, v); } else { *p = v; } }
struct Rec32 { float4 a, b; };
__device__ __forceinline__ Rec32 loadRec(const float4 *base, uint32_t slot) // 32-byte record `slot`: one LDG.256
{
    const float4 *p = base + 2 * (size_t)slot;
    Rec32 r;
#if PTC_STREAM_STATE
    asm volatile("ld.global.cs.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
#else
    asm volatile("ld.global.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
#endif
                 : "=f"(r.a.x), "=f"(r.a.y), "=f"(r.a.z), "=f"(r.a.w), "=f"(r.b.x), "=f"(r.b.y), "=f"(r.b.z), "=f"(r.b.w) : "l"(p));
    return r;
}
__device__ __forceinline__ void storeRec(float4 *base, uint32_t slot, const float4 a, const float4 b) // one STG.256: a whole sector
{
    float4 *p = base + 2 * (size_t)slot;
#if PTC_STREAM_STATE
    asm volatile("st.global.cs.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
#else
    asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
#endif
                 :: "l"(p), "f"(a.x), "f"(a.y), "f"(a.z), "f"(a.w), "f"(b.x), "f"(b.y), "f"(b.z), "f"(b.w) : "memory");
}
struct PathBuffers {
    // 32-byte records, current / next
    float4 *ray, *nRay;          // a = ray origin (= current vertex) xyz, w = origin slot bits | b = ray direction xyz
    float4 *modThr, *nModThr;    // a = modulation rgb up to the previous vertex, w = pdf of the BSDF sample that produced the ray |
                                 // b = that sample's throughput rgb, w = |n_s . wi|.  The modulation up to THIS vertex is a product of
                                 // the two halves (advanceModulation): the logic stage tests it, the material stage recomputes it
    // 32-byte record, single-buffered (written by the material stage at the new slot, read by the next shadow and logic stages)
    float4 *nee;                 // a = pending light-sampling contribution rgb | b = shadow ray direction, w = distance to the light sample
    // 16-byte arrays
    float4 *hit;                 // t, u, v, prim bits: written by the traversal, read by logic and material at the same slot
    float4 *result, *nResult;    // L() accumulator rgb, w = flags (current / next)
    uint8_t *occluded;           // outcome of the NEE shadow ray of the path in this slot (written for every traced shadow ray)
    float4 *out;                 // per-sample radiance by origin slot, written once when the path ends (FLAG_BASE: added to the
                                 // camera-hit emission the logic stage of bounce 0 stored there)
    uint32_t *shadowQueue;       // slots (next-bounce numbering) whose NEE shadow ray has to be traced
    uint32_t *classQueue[PTC_MATERIAL_CLASSES]; // survivors of the logic stage, binned by material class (null: class absent from the scene)
};

#define FLAG_BOUNCE_MASK 0xFFu
#define FLAG_DELTA 0x100u
#define FLAG_DIRECT 0x200u
#define FLAG_NEE 0x400u
#define FLAG_BASE 0x800u /* out[origin] already holds the camera-hit emission of this path */

struct WaveParams {
    uint64_t seed;
    uint32_t firstSample;  // global index of the first sample of this wave
    uint32_t sppWave;      // samples per pixel in this wave
    uint32_t nPixels;
    int32_t startBounce, lastBounce;
    uint32_t groupShift;   // log2 of the sample group (slotToPixelSample)
    const uint32_t *pixels; // the wave's pixel list (adaptive passes: nPixels pixels still active); null = every pixel of the image
};

// Device-side bookkeeping of one wave: queue sizes and work cursors per bounce (no host synchronisation inside a wave)
struct BounceCounters {
    uint32_t extendCount, shadowCount;           // rays leaving vertex k / NEE shadow rays cast at vertex k
    uint32_t classCount[PTC_MATERIAL_CLASSES];   // survivors of logic(k) per material class
    uint32_t extendCursor, shadowCursor;         // work cursors of the two traversal launches (lane refill)
    // VolumePathTracer wavefront (volume_wavefront.cuh): paths in the slot list of bounce k (there extendCount is the length of the
    // merged-ray queue, a subset of the slots), scatter-point shadow rays and their cursor
    uint32_t slotCount, scatterCount, scatterCursor;
    uint32_t pad[18];
};
static_assert(sizeof(BounceCounters) == 128, "one cache line per bounce");
#define CNT_STRIDE (PTC_MAX_BOUNCES + 2)
#define PTC_MAX_LANES 8

// Path slot q of a wave -> pixel.  Slots are laid out in 8x4 pixel tiles so that the 32 camera rays of a warp (and the
// secondary rays they spawn) stay spatially coherent; falls back to row-major when the image is not tileable.
__device__ __forceinline__ uint32_t slotToPixel(uint32_t q, uint32_t width, uint32_t height)
{
    if ((width & 7u) || (height & 3u)) { return q; }
    const uint32_t tile = q >> 5, within = q & 31u, tilesX = width >> 3;
    const uint32_t col = (tile % tilesX) * 8u + (within & 7u), row = (tile / tilesX) * 4u + (within >> 3);
    return row * width + col;
}
// Pixel slot q of a wave -> pixel, the one mapping every stage uses: an adaptive pass lists the pixels still active (a stable
// selection from slotToPixel's order, so a warp's camera rays stay in neighbouring tiles); a wave without a list covers the image.
// LISTED = false: compiled for waves without a list (the material kernels, whose register budget the test of the pointer would
// strain: +8..40 B of spills per class measured with -Xptxas -v)
template <bool LISTED = true>
__device__ __forceinline__ uint32_t wavePixel(uint32_t q, const WaveParams &wp, uint32_t width, uint32_t height)
{
    return LISTED && wp.pixels ? __ldg(wp.pixels + q) : slotToPixel(q, width, height);
}

// Origin slot p of a wave -> (pixel slot q, sample s of the wave).  G = 2^groupShift consecutive slots hold consecutive samples of
// one pixel, so a warp covers 32 / G neighbouring pixels x G samples: the rays of a warp start from (nearly) the same point of the
// scene at every bounce, and the node fetches of the traversal and the per-triangle gathers of the shading kernels hit the same
// sectors (measured on the dragon workload, 64-spp waves: G = 1 705.6, 8 712.5, 16 714.6, 32 716.2, 64 716.3 Msamples/s).  G is the
// largest power of two <= PTC_SAMPLE_GROUP that divides the wave's sample count (launch parameter); G = 1 is sample-major order (a warp =
// one 8x4 pixel tile of one sample).  The mapping only moves paths between slots: every path keeps its Philox key (pixel, sample) and
// the resolve adds a pixel's samples in sample order, so the image does not depend on G.
#ifndef PTC_SAMPLE_GROUP
#define PTC_SAMPLE_GROUP 32
#endif
__device__ __forceinline__ void slotToPixelSample(uint32_t p, const WaveParams &wp, uint32_t &q, uint32_t &s)
{
    const uint32_t shift = wp.groupShift;
    const uint32_t block = p >> shift; // block = sBlock * nPixels + q
    q = block % wp.nPixels; s = ((block / wp.nPixels) << shift) + (p & ((1u << shift) - 1u));
}
__device__ __forceinline__ size_t pixelSampleToSlot(uint32_t q, uint32_t s, const WaveParams &wp)
{
    const uint32_t shift = wp.groupShift;
    return ((((size_t)(s >> shift) * wp.nPixels + q) << shift) + (s & ((1u << shift) - 1u)));
}
static uint32_t groupShiftFor(uint32_t sppWave)
{
    uint32_t shift = 0;
    while ((2u << shift) <= PTC_SAMPLE_GROUP && sppWave % (2u << shift) == 0) { shift++; }
    return shift;
}

__device__ __forceinline__ uint32_t warpAppend(uint32_t *counter, bool pred)
{
    const uint32_t mask = __ballot_sync(0xFFFFFFFFu, pred); // called by all 32 lanes of the (warp-uniform) work loop
    if (!pred) { return 0xFFFFFFFFu; }
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t leader = __ffs(mask) - 1;
    uint32_t base = 0;
    if (lane == leader) { base = atomicAdd(counter, __popc(mask)); }
    base = __shfl_sync(mask, base, leader);
    return base + __popc(mask & ((1u << lane) - 1u));
}

// ------------------------------------------------------------------------------------------------ K1 generate
__global__ void __launch_bounds__(256) generateKernel(DScene scene, PathBuffers pb, WaveParams wp, BounceCounters *counters)
{
    const uint32_t nPaths = wp.nPixels * wp.sppWave;
    for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < nPaths; p += gridDim.x * blockDim.x) {
        uint32_t q, s;
        slotToPixelSample(p, wp, q, s);
        const uint32_t pixel = wavePixel(q, wp, (uint32_t)scene.width, (uint32_t)scene.height);
        Rng rng;
        rng.initPhilox(wp.seed, pixel, wp.firstSample + s);
        rng.beginVertex(0);
        const float jitterX = rng.next() - 0.5f; // box filter, src/camera.cpp:49-55
        const float jitterY = rng.next() - 0.5f;
        const int row = (int)(pixel / (uint32_t)scene.width), col = (int)(pixel % (uint32_t)scene.width);
        V3 o, d;
        cameraRay(scene, row + jitterY, col + jitterX, o, d);
        storeRec(pb.ray, p, make_float4(o.x, o.y, o.z, __uint_as_float(p)), make_float4(d.x, d.y, d.z, 0.f));
        streamStore(pb.result + p, make_float4(0.f, 0.f, 0.f, __uint_as_float(0u)));
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) { counters[0].extendCount = nPaths; }
}

// ------------------------------------------------------------------------------------------------ K2 extend / K3 shadow
__device__ __forceinline__ void flushCounters(const TraverseCounters &c, unsigned long long *work)
{
    uint32_t inner = c.inner, tris = c.tris;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { inner += __shfl_xor_sync(0xFFFFFFFFu, inner, o); tris += __shfl_xor_sync(0xFFFFFFFFu, tris, o); }
    if ((threadIdx.x & 31u) == 0) { atomicAdd(work, (unsigned long long)inner); atomicAdd(work + 1, (unsigned long long)tris); }
}

// Persistent warps with lane refill: every lane owns one ray; when a ray finishes its lane goes idle, and once at most
// PTC_REFILL_BELOW lanes are still busy the warp pulls new rays for all idle lanes from the queue cursor with a single
// atomic.  Keeps SIMT lanes busy although rays take very different numbers of steps (sky rays: 2-3, mesh rays: 20+).
// Inside an iteration the warp runs the node phase for every busy ray, then triangle rounds (one triangle per ray and
// round) while at least 1/PTC_POSTPONE_DIV of the busy rays have a triangle pending; the rays left over put their
// triangle group back on their stack and test it in a later, fuller round.
#ifndef PTC_REFILL_BELOW
#define PTC_REFILL_BELOW 24
#endif
#ifndef PTC_POSTPONE_DIV
#define PTC_POSTPONE_DIV 1000 /* off: measured slower on B200 (profiles/r01_sweep_postpone.txt) */
#endif

// 64 registers -> 8 resident CTAs per SM (48 / 10 before the phase split); forcing 12 or 16 CTAs (40 / 32 registers) spills and was measured slower
// (profiles/r01_sweep_occupancy.txt)
#ifdef PTC_TRAVERSE_MIN_BLOCKS
#define PTC_TRAVERSE_BOUNDS __launch_bounds__(128, PTC_TRAVERSE_MIN_BLOCKS)
#else
#define PTC_TRAVERSE_BOUNDS __launch_bounds__(128)
#endif
// Cooperative triangle phase.  After a node phase only a few lanes of a warp hold pending triangles (measured: 3.3 of 32
// lanes per sequential round, 4.4 rounds per node phase), so the (ray, triangle) pairs of all lanes are compacted with a
// warp prefix sum and spread over the 32 lanes: lane w tests pair w with the owner's ray fetched by shuffles, and owners
// collect accepted candidates in the order a sequential scan would have met them (highest group bit first), re-applying the
// upper end of the depth interval with their current hit distance -- the result is bit-identical to one-triangle-per-round.
#ifndef PTC_COOP_TRI
#define PTC_COOP_TRI 0
#endif
// Triangle rounds per node phase in the one-triangle-per-lane scheme.  Running a ray's whole triangle group before the
// warp's next node phase (the classic while-while loop) leaves 3 of 32 lanes active for 4.4 rounds per node phase on the
// dragon workload; with a bound, rays with triangles left skip node phases until their group is finished, so triangle
// rounds fill up with the leftovers of several node phases.  Per-ray order of operations, hence every result, is unchanged.
#ifndef PTC_TRI_ROUNDS
#define PTC_TRI_ROUNDS 2 /* sweep on the dragon workload: 1000 (while-while) 560, 1: 602, 2: 607, 3: 590 Msamples/s */
#endif
#ifndef PTC_TRI_ROUNDS_ANY
#define PTC_TRI_ROUNDS_ANY 1 /* shadow rays stop at the first hit: one round per node phase measured 47.6 against 49.2 ms per 4 steps */
#endif
template <bool ANY>
__device__ __forceinline__ bool coopTriangles(const BvhView &bvh, TraversalState &st, bool eligible, uint8_t *ownerOf)
{
    const uint32_t FULL = 0xFFFFFFFFu;
    const uint32_t lane = threadIdx.x & 31u;
    bool done = false;
    for (;;) {
        const uint32_t y = (eligible && !done) ? st.tgroup.y : 0u;
        const uint32_t want = __ballot_sync(FULL, y != 0u);
        if (want == 0u) { break; }
        const uint32_t c = __popc(y);
        uint32_t incl = c;
#pragma unroll
        for (uint32_t o = 1; o < 32u; o <<= 1) {
            const uint32_t v = __shfl_up_sync(FULL, incl, o);
            if (lane >= o) { incl += v; }
        }
        const uint32_t S = incl - c;                       // first pair index of this owner
        const uint32_t total = __shfl_sync(FULL, incl, 31);
        if (c) { ownerOf[__popc(want & ((1u << lane) - 1u))] = (uint8_t)lane; }
        const uint32_t starts = __reduce_or_sync(FULL, (c && S < 32u) ? 1u << S : 0u);
        __syncwarp();
        const bool work = lane < total;
        const uint32_t owner = work ? ownerOf[__popc(starts & (FULL >> (31u - lane))) - 1u] : lane;
        __syncwarp();
        const uint32_t So = __shfl_sync(FULL, S, owner);
        uint32_t yo = __brev(__shfl_sync(FULL, y, owner)); // highest group bit first
        const uint32_t base = __shfl_sync(FULL, st.tgroup.x, owner);
        const float ox = __shfl_sync(FULL, st.ox, owner), oy = __shfl_sync(FULL, st.oy, owner), oz = __shfl_sync(FULL, st.oz, owner);
        const float dx = __shfl_sync(FULL, st.dx, owner), dy = __shfl_sync(FULL, st.dy, owner), dz = __shfl_sync(FULL, st.dz, owner);
        const float tfar = __shfl_sync(FULL, st.hit.t, owner);
        bool accepted = false;
        float T = 0.f, U = 0.f, V = 0.f, absDen = 1.f;
        uint32_t prim = 0;
        if (work) {
            for (uint32_t k = lane - So; k; k--) { yo &= yo - 1u; }
            const uint32_t bit = 32u - (uint32_t)__ffs((int)yo);
            const float4 *tri = bvh.triangles + (size_t)(base + bit) * 3;
            const float4 a = loadNodeWord(tri), b = loadNodeWord(tri + 1), cc = loadNodeWord(tri + 2);
            accepted = triangleTestRaw(a, b, cc, ox, oy, oz, dx, dy, dz, PTC_TNEAR, tfar, T, U, V, absDen);
            prim = f2u(a.w);
        }
        const uint32_t acc = __ballot_sync(FULL, accepted);
        // owners retire the triangles that were tested this round (all of them unless the warp had more than 32 pairs)
        uint32_t n = 0;
        if (c && S < 32u) {
            n = min(c, 32u - S);
            if (n == c) { st.tgroup.y = 0u; }
            else {
                uint32_t yr = __brev(y);
                for (uint32_t k = n; k; k--) { yr &= yr - 1u; }
                st.tgroup.y = __brev(yr);
            }
        }
        uint32_t seg = n ? (acc >> S) & (FULL >> (32u - n)) : 0u;
        if (ANY) {
            if (seg) { done = true; st.found = true; }
        } else if (acc) {
            const float t = divIeee(T, absDen);
            while (__any_sync(FULL, seg != 0u)) {
                const uint32_t src = seg ? S + (uint32_t)__ffs((int)seg) - 1u : lane;
                const float ct = __shfl_sync(FULL, t, src), cu = __shfl_sync(FULL, U, src), cv = __shfl_sync(FULL, V, src);
                const float cT = __shfl_sync(FULL, T, src), cA = __shfl_sync(FULL, absDen, src);
                const uint32_t cp = __shfl_sync(FULL, prim, src);
                if (seg) {
                    seg &= seg - 1u;
                    if (cT <= cA * st.hit.t) { // the candidate passed (tnear, round-start tfar]; tfar may have shrunk since
                        if (!(st.found && ct == st.hit.t && cp < st.hit.prim)) { st.hit.t = ct; st.hit.u = cu; st.hit.v = cv; st.hitDen = cA; st.hit.prim = cp; }
                        st.found = true;
                    }
                }
            }
        }
    }
    return done;
}

// FILTER (shadow rays of a scene with container surfaces): Scene::testOcclusion's filter, src/scene.cpp:42-84, :369-370
// INSTANCES: the scene holds flattened instance placements, whose triangles are tested in the instance's space (traverse.cuh: rayToPlacement)
template <bool ANY, bool COUNT, bool FILTER = false, bool INSTANCES = false>
__global__ void PTC_TRAVERSE_BOUNDS traverseKernel(DScene scene, PathBuffers pb, const uint32_t *queue, const uint32_t *count, uint32_t *cursor,
                                                      unsigned long long *work)
{
    __shared__ uint2 fastStack[(PTC_FAST_STACK > 0 ? PTC_FAST_STACK : 1) * PTC_FAST_STRIDE]; // [entry][thread]: conflict-free 64-bit accesses
    uint2 *const fast = fastStack + threadIdx.x;
    __shared__ uint8_t ownerSlots[128];
    uint8_t *const ownerOf = ownerSlots + (threadIdx.x & ~31u); // this warp's 32 entries
    const uint32_t n = *count;
    const uint32_t lane = threadIdx.x & 31u;
    TraverseCounters tc = {0, 0};
    TraversalState st;
    bool busy = false, more = n > 0;
    uint32_t p = 0;
    const bool hasNodes = scene.bvh.nNodes != 0;
    for (;;) {
        const uint32_t idle = __ballot_sync(0xFFFFFFFFu, !busy);
        if (idle && more) {
            const uint32_t k = __popc(idle);
            uint32_t base = 0;
            if (lane == 0) { base = atomicAdd(cursor, k); }
            base = __shfl_sync(0xFFFFFFFFu, base, 0);
            if (!busy) {
                const uint32_t item = base + __popc(idle & ((1u << lane) - 1u));
                if (item < n) {
                    p = queue ? streamLoad(queue + item) : item; // extend: the paths of a bounce occupy slots 0 .. n - 1
                    if (ANY) { // Scene::testOcclusion, src/scene.cpp:355-381: any hit in (1e-3, maxT - 1e-3]
                        const float4 o = streamLoad(pb.ray + 2 * (size_t)p), d = streamLoad(pb.nee + 2 * (size_t)p + 1);
                        traversalInit(st, o.x, o.y, o.z, d.x, d.y, d.z, PTC_TNEAR, d.w - 1e-3f);
                    } else {   // Scene::testIntersect, src/scene.cpp:91-120
                        const Rec32 r = loadRec(pb.ray, p);
                        traversalInit(st, r.a.x, r.a.y, r.a.z, r.b.x, r.b.y, r.b.z, PTC_TNEAR, PTC_TFAR);
                    }
                    if (!hasNodes) { st.ngroup.y = 0u; }
                    busy = true;
                }
            }
            more = base + k < n;
        }
        uint32_t active = __ballot_sync(0xFFFFFFFFu, busy);
        if (active == 0u) { break; }
        for (;;) {
            // a ray whose triangle group is not finished yet (more triangles than PTC_TRI_ROUNDS) sits out this node phase
            if (busy && hasNodes && st.tgroup.y == 0u) { traversalNode<COUNT>(scene.bvh, st, &tc, fast); }
            bool done = false; // this ray needs no further BVH work
            if (PTC_COOP_TRI && !COUNT && !FILTER && !INSTANCES) { done = coopTriangles<ANY>(scene.bvh, st, busy, ownerOf); }
            else {
                for (int round = 0; round < (ANY ? PTC_TRI_ROUNDS_ANY : PTC_TRI_ROUNDS); round++) { // triangle rounds, warp-uniform control flow
                    bool pending = busy && !done && st.tgroup.y != 0u;
                    const uint32_t want = __ballot_sync(0xFFFFFFFFu, pending);
                    if (want == 0u) { break; }
                    if (__popc(want) * PTC_POSTPONE_DIV < __popc(active)) {
                        if (pending && traversalPostpone(st, fast)) { pending = false; }
                        if (!__any_sync(0xFFFFFFFFu, pending)) { break; }
                    }
                    if (pending && traversalTriangle<COUNT, FILTER, INSTANCES>(scene.bvh, st, &tc) && ANY) { done = true; }
                }
            }
            if (busy && (done || (st.tgroup.y == 0u && traversalPop(st, fast)))) {
                const bool found = traversalSpheres<ANY, FILTER>(scene.bvh, st);
                if (ANY) { pb.occluded[p] = found ? 1 : 0; }
                else { streamStore(pb.hit + p, make_float4(st.hit.t, st.hit.u, st.hit.v, __uint_as_float(st.hit.prim))); }
                busy = false;
            }
            active = __ballot_sync(0xFFFFFFFFu, busy);
            if (active == 0u || (more && __popc(active) <= PTC_REFILL_BELOW)) { break; }
        }
    }
    if (COUNT) { flushCounters(tc, work); }
}

// ------------------------------------------------------------------------------------------------ K5-K6 logic
// Handles the result of the ray that left vertex k (k = 0: the camera ray): everything in PathTracer::L between two
// BSDF samples.  Cheap per path (the Intersection is only built for emitter hits); survivors go to the class queues.
// Registers / occupancy (profiles/r02_sweep_shade_occupancy.txt, dragon workload, shade ms per 4 steps): the material kernels at 64
// registers -> 8 CTAs of 128 per SM, with ~170 bytes of spills: 117.2; 80 registers / 6 CTAs 120.7; 96-100 / 5 CTAs 123.4; 10, 12, 16 CTAs
// 125.8, 135.4, 136.0 -- they wait on dependent loads and fixed-latency arithmetic, so more resident warps pay until the spills take
// over.  The logic kernel stays at the compiler's 76 registers (3 CTAs of 256): 64 / 48 registers measured 124.5 / 125.3 against 123.4.
// SampleIntegrator::samplePixel's container branch (src/sample_integrator.cpp:35-51): the camera ray hit a Passthrough surface;
// adds what lies behind it, attenuated by the medium.
__device__ __forceinline__ void cameraContainerTerm(const DScene &scene, float ox, float oy, float oz, float dx, float dy, float dz, float *rgb)
{
    const V3 O = mk(ox, oy, oz), D = mk(dx, dy, dz);
    VolumeEvents ev; RayHit vh;
    const bool vHit = traverseFiltered<false>(scene, O, D, PTC_TNEAR, PTC_TFAR, vh, ev);
    const V3 tr = rayTransmission(scene, O, D, ev, -1);
    V3 add;
    if (vHit) {
        Isect vi; makeIsect(scene, O, D, vh, vi);
        const DMaterial &vm = scene.materials[vi.material];
        add = mk(vm.emit[0], vm.emit[1], vm.emit[2]) * tr;
    } else { add = envRadiance(scene, D) * tr; }
    rgb[0] = add.x; rgb[1] = add.y; rgb[2] = add.z;
}

// Runs between logic(0) and the material kernels of vertex 1, only for scenes with container surfaces: the camera ray and its
// hit are still in the path state, and out[p] holds the camera-hit emission (0 for a Passthrough surface).
__global__ void __launch_bounds__(128) containerKernel(const __grid_constant__ DScene scene, PathBuffers pb, WaveParams wp, const BounceCounters *bc)
{
    const uint32_t n = bc->extendCount;
    if (!checkCounts(wp.startBounce, wp.lastBounce, 0)) { return; }
    for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < n; p += gridDim.x * blockDim.x) { // bounce 0: slot = origin
        const float4 h4 = streamLoad(pb.hit + p);
        const uint32_t prim = __float_as_uint(h4.w);
        if (prim == PTC_MISS) { continue; }
        const uint32_t material = (prim & PTC_SPHERE_FLAG) ? __ldg(scene.sphereIds + (prim & ~PTC_SPHERE_FLAG)).y : __ldg(&scene.prims[prim].w);
        if (__ldg(&scene.materials[material].type) != PTC_PASSTHROUGH) { continue; }
        const Rec32 r = loadRec(pb.ray, p);
        float add[3];
        cameraContainerTerm(scene, r.a.x, r.a.y, r.a.z, r.b.x, r.b.y, r.b.z, add);
        // a Passthrough surface is no emitter, so logic(0) stored no base colour: this term becomes the base (FLAG_BASE)
        streamStore(pb.out + p, make_float4(add[0], add[1], add[2], 0.f));
        const float4 res4 = streamLoad(pb.result + p);
        streamStore(pb.result + p, make_float4(res4.x, res4.y, res4.z, __uint_as_float(__float_as_uint(res4.w) | FLAG_BASE)));
    }
}

#ifndef PTC_LAZY_DIRECTION
#define PTC_LAZY_DIRECTION 1
#endif
// modulation up to the vertex a ray arrives at, from the (modulation up to the previous vertex, pdf | throughput, cosine) record of
// the ray: PathTracer::L, src/path_tracer.cpp:51-53.  One function for the logic stage (tests it) and the material stage (carries it on)
__device__ __forceinline__ V3 advanceModulation(const float4 mp, const float4 tc)
{
    const float invPDF = 1.f / mp.w;
    return mk(mp.x, mp.y, mp.z) * ((mk(tc.x, tc.y, tc.z) * tc.w) * invPDF);
}

// color += L(...), src/sample_integrator.cpp:53: the path ends, its radiance goes to the entry of its origin slot
__device__ __forceinline__ void finishPath(const PathBuffers &pb, uint32_t origin, uint32_t flags, const V3 result)
{
    float4 c = make_float4(0.f, 0.f, 0.f, 0.f);
    if (flags & FLAG_BASE) { c = streamLoad(pb.out + origin); }
    streamStore(pb.out + origin, make_float4(c.x + result.x, c.y + result.y, c.z + result.z, 0.f));
}

// `bounce` = k of every path of the launch (ray k leaves vertex k), so which records a path needs is known before any of them
// arrives: hit, result, (modulation | throughput) and the occlusion byte are requested together, the pending NEE term as soon as the
// flags are there.  The class of the surface (material type, emitter bit) comes from one byte per primitive (DScene::primClass)
// instead of the index record and the material table one after the other.
#ifndef PTC_LOGIC_MIN_BLOCKS
#define PTC_LOGIC_MIN_BLOCKS 3
#endif
__global__ void __launch_bounds__(256, PTC_LOGIC_MIN_BLOCKS) logicKernel(DScene scene, PathBuffers pb, WaveParams wp, BounceCounters *bc, uint32_t classMask, int bounce)
{
    const uint32_t n = bc->extendCount;
    const int k = bounce;
    const uint32_t lane = threadIdx.x & 31u;
    // uniform cost per path: static warp-strided assignment (whole warps stay in the loop together for the ballots below);
    // slot p of the current buffers = item p of this bounce's ray list, so every load below is a dense, coalesced one
    for (uint32_t base = (blockIdx.x * blockDim.x + threadIdx.x) & ~31u; base < n; base += gridDim.x * blockDim.x) {
        const uint32_t p = base + lane;
        int cls = -1;
        if (p < n) {
            const float4 h4 = streamLoad(pb.hit + p);
            const float4 res4 = streamLoad(pb.result + p);
            Rec32 mt; mt.a = mt.b = make_float4(0.f, 0.f, 0.f, 0.f);
            uint8_t occluded = 0;
            if (k > 0) { mt = loadRec(pb.modThr, p); occluded = pb.occluded[p]; }
            const uint32_t flags = __float_as_uint(res4.w);
            float4 ne = make_float4(0.f, 0.f, 0.f, 0.f);
            if (k > 0 && (flags & FLAG_NEE)) { ne = streamLoad(pb.nee + 2 * (size_t)p); }
            const uint32_t prim = __float_as_uint(h4.w);
            const bool isHit = prim != PTC_MISS;
            uint32_t surface = 0; // material type | emitter << 3
            if (isHit) { surface = (prim & PTC_SPHERE_FLAG) ? __ldg(scene.sphereClass + (prim & ~PTC_SPHERE_FLAG)) : __ldg(scene.primClass + prim); }
            const bool emitter = (surface & 8u) != 0;
            V3 result = mk(res4.x, res4.y, res4.z);
            bool alive = true;
            // the ray (origin, direction) is only needed for environment misses and emitter hits: a surviving ordinary hit never reads it
            const bool needRay = PTC_LAZY_DIRECTION ? (!isHit || emitter) : true;
            Rec32 ray;
            if (needRay) { ray = loadRec(pb.ray, p); }
            uint32_t material = 0;
            if (isHit && emitter) { material = (prim & PTC_SPHERE_FLAG) ? __ldg(scene.sphereIds + (prim & ~PTC_SPHERE_FLAG)).y : __ldg(&scene.prims[prim].w); }
            if (k == 0) {
                // SampleIntegrator::samplePixel, src/sample_integrator.cpp:18-59; bounce 0: slot = origin slot
                if (!isHit) {
                    const V3 color = envRadiance(scene, mk(ray.b.x, ray.b.y, ray.b.z));
                    streamStore(pb.out + p, make_float4(color.x + result.x, color.y + result.y, color.z + result.z, 0.f));
                    alive = false;
                } else if (emitter && checkCounts(wp.startBounce, wp.lastBounce, 0)) {
                    RayHit hit; hit.t = h4.x; hit.u = h4.y; hit.v = h4.z; hit.prim = prim;
                    Isect bi;
                    makeIsect(scene, mk(ray.a.x, ray.a.y, ray.a.z), mk(ray.b.x, ray.b.y, ray.b.z), hit, bi);
                    const DMaterial &m = scene.materials[material];
                    if (!(dot(bi.n, bi.wo) < 0.f)) { // what samplePixel adds itself waits in `out` for the end of the path
                        streamStore(pb.out + p, make_float4(__ldg(&m.emit[0]), __ldg(&m.emit[1]), __ldg(&m.emit[2]), 0.f));
                        streamStore(pb.result + p, make_float4(res4.x, res4.y, res4.z, __uint_as_float(flags | FLAG_BASE)));
                    }
                }
            } else {
                if (flags & FLAG_DIRECT) { // direct() of vertex k, src/path_tracer.cpp:79-111
                    V3 Ld = mk(0.f, 0.f, 0.f);
                    if ((flags & FLAG_NEE) && !occluded) { Ld = Ld + mk(ne.x, ne.y, ne.z); }
                    if (!isHit || emitter) { // directSampleBSDF contributes only for emitter hits and environment misses
                        const V3 O = mk(ray.a.x, ray.a.y, ray.a.z), D = mk(ray.b.x, ray.b.y, ray.b.z);
                        Isect bi;
                        if (isHit) { RayHit hit; hit.t = h4.x; hit.u = h4.y; hit.v = h4.z; hit.prim = prim; makeIsect(scene, O, D, hit, bi); }
                        Ld = Ld + directBsdf(scene, O, mt.b.w, D, mt.a.w, mk(mt.b.x, mt.b.y, mt.b.z), (flags & FLAG_DELTA) != 0, isHit, &bi);
                    }
                    result = result + Ld * mk(mt.a.x, mt.a.y, mt.a.z);
                }
                // loop header and body of PathTracer::L, src/path_tracer.cpp:41-58
                if (checkDone(wp.lastBounce, k + 1) || !isHit || isBlack(advanceModulation(mt.a, mt.b))) { alive = false; }
                if (alive && (flags & FLAG_DIRECT)) { streamStore(pb.result + p, make_float4(result.x, result.y, result.z, res4.w)); }
                if (!alive) {
                    const uint32_t origin = needRay ? __float_as_uint(ray.a.w) : __float_as_uint(streamLoad(&pb.ray[2 * (size_t)p].w));
                    finishPath(pb, origin, flags, result);
                }
            }
            if (alive) { cls = (int)(surface & 7u); }
        }
        // survivors join the queue of their material class: the warp's counts of all classes are added with atomics issued back to
        // back by one lane (one round trip for all of them), then every survivor takes its place behind the lanes before it
        uint32_t masks[PTC_MATERIAL_CLASSES], starts[PTC_MATERIAL_CLASSES];
#pragma unroll
        for (int t = 0; t < PTC_MATERIAL_CLASSES; t++) {
            masks[t] = 0u; starts[t] = 0u;
            if (!(classMask & (1u << t))) { continue; }
            masks[t] = __ballot_sync(0xFFFFFFFFu, cls == t);
            if (lane == 0 && masks[t]) { starts[t] = atomicAdd(&bc->classCount[t], __popc(masks[t])); }
        }
        uint32_t mine = 0, myBase = 0;
#pragma unroll
        for (int t = 0; t < PTC_MATERIAL_CLASSES; t++) {
            if (!(classMask & (1u << t))) { continue; }
            const uint32_t start = __shfl_sync(0xFFFFFFFFu, starts[t], 0);
            if (cls == t) { mine = masks[t]; myBase = start; }
        }
        if (cls >= 0) { streamStore(pb.classQueue[cls] + myBase + __popc(mine & ((1u << lane) - 1u)), p); }
    }
}

// ------------------------------------------------------------------------------------------------ K4 material
// Vertex k + 1 of every surviving path whose hit surface has material class TYPE: Intersection, BSDF sample, NEE set-up.
// LISTED: the wave has a pixel list (wavePixel)
template <int TYPE, bool LISTED>
#ifndef PTC_MATERIAL_MIN_BLOCKS
#define PTC_MATERIAL_MIN_BLOCKS 8
#endif
__global__ void __launch_bounds__(128, PTC_MATERIAL_MIN_BLOCKS) materialKernel(DScene scene, PathBuffers pb, WaveParams wp, BounceCounters *bc, BounceCounters *next)
{
    const uint32_t n = bc->classCount[TYPE];
    const uint32_t *queue = pb.classQueue[TYPE];
    for (uint32_t base = (blockIdx.x * blockDim.x + threadIdx.x) & ~31u; base < n; base += gridDim.x * blockDim.x) {
        const uint32_t item = base + (threadIdx.x & 31u);
        bool pushExtend = false, pushShadow = false;
        // what the path carries to its slot of the next bounce
        float4 nO = make_float4(0.f, 0.f, 0.f, 0.f), nD = nO, nMod = nO, nThr = nO, nRes = nO, nNee = nO, nSh = nO;
        if (item < n) {
            const uint32_t p = streamLoad(queue + item);
            const Rec32 ray = loadRec(pb.ray, p);
            const float4 h4 = streamLoad(pb.hit + p), res4 = streamLoad(pb.result + p);
            const uint32_t origin = __float_as_uint(ray.a.w);
            const uint32_t flags = __float_as_uint(res4.w);
            const int k = (int)(flags & FLAG_BOUNCE_MASK);
            RayHit hit; hit.t = h4.x; hit.u = h4.y; hit.v = h4.z; hit.prim = __float_as_uint(h4.w);
            Isect bi;
            makeIsect(scene, mk(ray.a.x, ray.a.y, ray.a.z), mk(ray.b.x, ray.b.y, ray.b.z), hit, bi);
            const DMaterial &m = scene.materials[bi.material];
            Rng rng;
            uint32_t oq, os;
            slotToPixelSample(origin, wp, oq, os);
            rng.initPhilox(wp.seed, wavePixel<LISTED>(oq, wp, (uint32_t)scene.width, (uint32_t)scene.height), wp.firstSample + os);
            rng.beginVertex((uint32_t)(k + 1));
            BsdfSample bs;
            bsdfSample<TYPE>(m, bi, rng, bs);
            const bool wantDirect = checkCounts(wp.startBounce, wp.lastBounce, k + 1) && !__ldg(&m.emitter);
            if (wantDirect) {
                V3 contribution, sd; float maxT;
                // a contribution that is exactly black adds nothing whether or not the light is visible (src/path_tracer.cpp:
                // 138-164: occluded -> 0, else the contribution), e.g. a light sampled below the surface: no shadow ray for it
                if (directLightsSetup<TYPE>(scene, m, bi, bs, rng, contribution, sd, maxT) && !isBlack(contribution)) {
                    nNee = make_float4(contribution.x, contribution.y, contribution.z, 0.f);
                    nSh = make_float4(sd.x, sd.y, sd.z, maxT);
                    pushShadow = true;
                }
            }
            const bool wantNext = !checkDone(wp.lastBounce, k + 2);
            if (wantDirect || wantNext) {
                nO = make_float4(bi.point.x, bi.point.y, bi.point.z, ray.a.w);
                nD = make_float4(bs.wi.x, bs.wi.y, bs.wi.z, 0.f);
                if (k == 0) { nMod = make_float4(1.f, 1.f, 1.f, bs.pdf); } // the modulation starts at 1
                else { const Rec32 mt = loadRec(pb.modThr, p); const V3 mod = advanceModulation(mt.a, mt.b); nMod = make_float4(mod.x, mod.y, mod.z, bs.pdf); }
                nThr = make_float4(bs.thr.x, bs.thr.y, bs.thr.z, fabsf(dot(bi.ns, bs.wi)));
                const uint32_t nf = (uint32_t)(k + 1) | (bs.delta ? FLAG_DELTA : 0u) | (wantDirect ? FLAG_DIRECT : 0u) | (pushShadow ? FLAG_NEE : 0u) | (flags & FLAG_BASE);
                nRes = make_float4(res4.x, res4.y, res4.z, __uint_as_float(nf));
                pushExtend = true;
            } else { // the path ends here: color += L(...)
                pushShadow = false;
                finishPath(pb, origin, flags, mk(res4.x, res4.y, res4.z));
            }
        }
        // compaction: the path moves to slot e of the next bounce; consecutive lanes get consecutive slots (coalesced stores)
        const uint32_t e = warpAppend(&next->extendCount, pushExtend);
        if (pushExtend) {
            storeRec(pb.nRay, e, nO, nD);
            storeRec(pb.nModThr, e, nMod, nThr);
            streamStore(pb.nResult + e, nRes);
            if (pushShadow) { storeRec(pb.nee, e, nNee, nSh); }
        }
        const uint32_t sh = warpAppend(&next->shadowCount, pushShadow);
        if (pushShadow) { streamStore(pb.shadowQueue + sh, e); }
    }
}

// ------------------------------------------------------------------------------------------------ K7 resolve
// Checkpoints that fall inside a wave (src/integrator.cpp:87-92 saves the image after 1, 2, 4, ... samples): the resolve keeps a copy
// of the running sums after `at[i]` samples of the wave in dst[i], so a wave does not have to end at every power of two
struct CheckpointPlan { uint32_t n; uint32_t at[PTC_MAX_CHECKPOINTS]; float *dst[PTC_MAX_CHECKPOINTS]; };
// MOMENTS (adaptive passes, option framebuffer_moments): moments[3 * pixel + c] += x_c^2 for every sample x, in sample order like the
// sums.  A checkpoint copy then holds both: dst[i] is a buffer of 6 x W x H floats, the sums followed by the second moments (the
// moments' destination is not a field of the plan, so the plain instance keeps its parameters and code)
template <bool MOMENTS>
__global__ void __launch_bounds__(256) accumulateKernel(PathBuffers pb, WaveParams wp, float *accum, float *moments, uint32_t width, uint32_t height, const __grid_constant__ CheckpointPlan plan)
{
    const size_t momentsAt = 3 * (size_t)width * height; // MOMENTS: offset of a checkpoint's moments in its buffer
    for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < wp.nPixels; q += gridDim.x * blockDim.x) {
        const size_t pixel = wavePixel(q, wp, width, height);
        float r = accum[3 * pixel], g = accum[3 * pixel + 1], b = accum[3 * pixel + 2];
        float mr = 0.f, mg = 0.f, mb = 0.f;
        if (MOMENTS) { mr = moments[3 * pixel]; mg = moments[3 * pixel + 1]; mb = moments[3 * pixel + 2]; }
        uint32_t next = 0;
        for (uint32_t s = 0; s < wp.sppWave; s++) { // radianceLookup += color, one sample after the other (src/sample_integrator.cpp:61-63)
            while (next < plan.n && plan.at[next] == s) {
                float *d = plan.dst[next++]; d[3 * pixel] = r; d[3 * pixel + 1] = g; d[3 * pixel + 2] = b;
                if (MOMENTS) { d += momentsAt; d[3 * pixel] = mr; d[3 * pixel + 1] = mg; d[3 * pixel + 2] = mb; }
            }
            const float4 c = streamLoad(pb.out + pixelSampleToSlot(q, s, wp));
            r += c.x; g += c.y; b += c.z;
            if (MOMENTS) { mr += c.x * c.x; mg += c.y * c.y; mb += c.z * c.z; }
        }
        while (next < plan.n) {
            float *d = plan.dst[next++]; d[3 * pixel] = r; d[3 * pixel + 1] = g; d[3 * pixel + 2] = b;
            if (MOMENTS) { d += momentsAt; d[3 * pixel] = mr; d[3 * pixel + 1] = mg; d[3 * pixel + 2] = mb; }
        }
        accum[3 * pixel] = r; accum[3 * pixel + 1] = g; accum[3 * pixel + 2] = b;
        if (MOMENTS) { moments[3 * pixel] = mr; moments[3 * pixel + 1] = mg; moments[3 * pixel + 2] = mb; }
    }
}

// Adaptive sampling: the stopping test after a pass that ended at n samples per listed pixel.  Pixel p stops when for every channel
// var_c / n <= tau^2 (mean_c^2 + 1e-2) (mean = S / n, var = max(0, (M - n mean^2) / (n - 1)), in fp64): the expected per-pixel
// term of the relMSE metric (x - r)^2 / (r^2 + 1e-2) is below the target tau^2.  A non-finite estimate never stops a pixel, and
// every pixel stops at n = maxSpp.  counts[pixel] = n for every listed pixel; next[q] = the pixel if it goes on, else ~0u (dropped by
// the stable selection that follows).  --fmad=false: no contraction, the test is the plain fp64 expression.
__global__ void __launch_bounds__(256) adaptiveTestKernel(WaveParams wp, const float *sums, const float *moments, uint32_t *counts, uint32_t *next,
                                                          uint32_t width, uint32_t height, double tau2, uint32_t n, uint32_t maxSpp)
{
    for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < wp.nPixels; q += gridDim.x * blockDim.x) {
        const uint32_t pixel = wavePixel(q, wp, width, height);
        bool stop = n >= maxSpp;
        if (!stop) {
            stop = true;
            const double dn = (double)n;
            for (int c = 0; c < 3; c++) {
                const double mean = (double)sums[3 * (size_t)pixel + c] / dn;
                const double sq = mean * mean;
                double var = ((double)moments[3 * (size_t)pixel + c] - dn * sq) / (dn - 1.0);
                if (var < 0.0) { var = 0.0; }
                stop = stop && isfinite(mean) && isfinite(var) && var / dn <= tau2 * (sq + 1e-2);
            }
        }
        counts[pixel] = n;
        next[q] = stop ? ~0u : pixel;
    }
}
struct StillActive { __device__ __forceinline__ bool operator()(uint32_t v) const { return v != ~0u; } };

// ------------------------------------------------------------------------------------------------ VolumePathTracer
// One thread follows one path from the camera to its end (volume.cuh: volumeRadiance); warps pull 32 paths at a time from a
// global cursor, so a warp whose paths ended early does not wait for the rest of the wave.  First correct form of the
// participating-media integrator (SURVEY 8(f) N3); its rays are data-dependent in number (container probes, scatter shadow
// rays), which is what the wavefront stages above would have to be widened for.
// 16 resident CTAs per SM (32 registers, the rest spills to L1): measured 2.1x faster than the compiler's own allocation
// (186 registers, 2 CTAs) -- the kernel waits on dependent loads, not on issue slots (profiles/r01_sweep_volume_occupancy.txt)
#ifndef PTC_VOLUME_MIN_BLOCKS
#define PTC_VOLUME_MIN_BLOCKS 16
#endif
template <bool COUNT>
__global__ void __launch_bounds__(128, PTC_VOLUME_MIN_BLOCKS) volumePathKernel(const __grid_constant__ DScene scene, float4 *out, WaveParams wp, uint32_t *cursor, unsigned long long *totals)
{
    const uint32_t nPaths = wp.nPixels * wp.sppWave;
    const uint32_t lane = threadIdx.x & 31u;
    VolumeWork work = {0, 0, {0, 0}, {0, 0}};
    for (;;) {
        uint32_t base = 0;
        if (lane == 0) { base = atomicAdd(cursor, 32u); }
        base = __shfl_sync(0xFFFFFFFFu, base, 0);
        if (base >= nPaths) { break; }
        const uint32_t p = base + lane;
        if (p < nPaths) {
            uint32_t q, s;
            slotToPixelSample(p, wp, q, s);
            const uint32_t pixel = wavePixel(q, wp, (uint32_t)scene.width, (uint32_t)scene.height);
            Rng rng;
            rng.initPhilox(wp.seed, pixel, wp.firstSample + s);
            rng.beginVertex(0);
            const float jitterX = rng.next() - 0.5f;
            const float jitterY = rng.next() - 0.5f;
            const int row = (int)(pixel / (uint32_t)scene.width), col = (int)(pixel % (uint32_t)scene.width);
            V3 o, d;
            cameraRay(scene, row + jitterY, col + jitterX, o, d);
            const V3 L = volumeRadiance<COUNT>(scene, o, d, rng, wp.startBounce, wp.lastBounce, &work);
            out[p] = make_float4(L.x, L.y, L.z, 0.f);
        }
    }
    // totals: [0] closest rays, [1] shadow rays, [2..3] inner visits / triangle tests of the closest-hit rays, [4..5] of the shadow rays
    uint32_t v[6] = {work.closestRays, work.shadowRays, work.closest.inner, work.closest.tris, work.shadow.inner, work.shadow.tris};
#pragma unroll
    for (int k = 0; k < 6; k++) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { v[k] += __shfl_xor_sync(0xFFFFFFFFu, v[k], o); }
        if (lane == 0 && (k < 2 || COUNT)) { atomicAdd(totals + k, (unsigned long long)v[k]); }
    }
}

#include "volume_wavefront.cuh"
// K7 resolve fused with the spp-split reduce (gatherResolveKernel) and the device-resident denoise read these: every framebuffer but the
// first lives on another GPU and is read through its NVLink peer mapping (or a staged local copy when peer access is unavailable)
struct FramebufferSet { const float *fb[PTC_MAX_PEERS + 1]; int count; };
#include "denoise.cuh"

__global__ void resolveKernel(const float *accum, float *out, uint32_t n, uint32_t spp) // src/integrator.cpp:74-85
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) { out[i] = accum[i] / (int)spp; }
}

// K7 resolve fused with the spp-split reduce, summed in a fixed order
__global__ void __launch_bounds__(256) gatherResolveKernel(FramebufferSet set, float *out, uint32_t n, uint32_t divisor)
{
    const uint32_t n4 = n >> 2;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += gridDim.x * blockDim.x) {
        float4 sum = reinterpret_cast<const float4 *>(set.fb[0])[i];
        for (int g = 1; g < set.count; g++) {
            const float4 v = reinterpret_cast<const float4 *>(set.fb[g])[i];
            sum.x += v.x; sum.y += v.y; sum.z += v.z; sum.w += v.w;
        }
        reinterpret_cast<float4 *>(out)[i] = make_float4(sum.x / (int)divisor, sum.y / (int)divisor, sum.z / (int)divisor, sum.w / (int)divisor);
    }
    for (uint32_t i = (n4 << 2) + blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        float sum = set.fb[0][i];
        for (int g = 1; g < set.count; g++) { sum += set.fb[g][i]; }
        out[i] = sum / (int)divisor;
    }
}

// SURVEY 8(f) N4, after the BVH build over the flattened (world-space) placements: the leaf triangles of a placement get the
// instance's LOCAL-space corners back and the tag of their placement, so that the traversal tests them where Embree does
__global__ void localizeLeavesKernel(LeafTriangle *triangles, uint32_t n, const float4 *positions, const uint4 *prims, const uint32_t *tags)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        LeafTriangle t = triangles[i];
        const uint32_t tag = tags[t.prim];
        if (!tag) { continue; }
        const uint4 ix = prims[t.prim];
        const float4 v0 = positions[ix.x], v1 = positions[ix.y], v2 = positions[ix.z];
        t.v0[0] = v0.x; t.v0[1] = v0.y; t.v0[2] = v0.z;
        t.e1[0] = v0.x - v1.x; t.e1[1] = v0.y - v1.y; t.e1[2] = v0.z - v1.z; t.pad0 = tag;
        t.e2[0] = v2.x - v0.x; t.e2[1] = v2.y - v0.y; t.e2[2] = v2.z - v0.z;
        triangles[i] = t;
    }
}

__global__ void tallyKernel(const BounceCounters *counters, unsigned long long *totals)
{
    if (threadIdx.x == 0) {
        unsigned long long closest = 0, shadow = 0;
        for (int b = 0; b < CNT_STRIDE; b++) { closest += counters[b].extendCount; shadow += counters[b].shadowCount + counters[b].scatterCount; }
        totals[0] += closest; totals[1] += shadow;
    }
}

// ================================================================================================ probe kernels
__global__ void intersectKernel(DScene scene, const ptc_ray *rays, uint32_t n, ptc_hit *hits, uint2 *inst)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const ptc_ray r = rays[i];
        RayHit h;
        ptc_hit out;
        uint2 instance = make_uint2(PTC_INVALID_ID, PTC_INVALID_ID);
        if (traverseBVH<false, false>(scene.bvh, r.origin[0], r.origin[1], r.origin[2], r.direction[0], r.direction[1], r.direction[2], PTC_TNEAR, PTC_TFAR, h, nullptr)) {
            Isect is; V3 ng;
            makeIsect(scene, mk(r.origin[0], r.origin[1], r.origin[2]), mk(r.direction[0], r.direction[1], r.direction[2]), h, is, &ng);
            out.t = h.t; out.u = h.u; out.v = h.v; out.ng[0] = ng.x; out.ng[1] = ng.y; out.ng[2] = ng.z;
            if (h.prim & PTC_SPHERE_FLAG) { out.geom_id = scene.sphereIds[h.prim & ~PTC_SPHERE_FLAG].x; out.prim_id = 0; }
            else {
                const uint2 id = scene.primIds[h.prim]; out.geom_id = id.x; out.prim_id = id.y;
                if (scene.instIds) { instance = scene.instIds[h.prim]; }
            }
        } else {
            out.t = PTC_TFAR; out.u = 0.f; out.v = 0.f; out.geom_id = PTC_INVALID_ID; out.prim_id = PTC_INVALID_ID; out.ng[0] = out.ng[1] = out.ng[2] = 0.f;
        }
        hits[i] = out;
        if (inst) { inst[i] = instance; }
    }
}

__device__ __forceinline__ void exportIsect(const Isect &s, float t, ptc_isect &o)
{
    o.hit = 1; o.t = t;
    o.point[0] = s.point.x; o.point[1] = s.point.y; o.point[2] = s.point.z;
    o.wo[0] = s.wo.x; o.wo[1] = s.wo.y; o.wo[2] = s.wo.z;
    o.normal[0] = s.n.x; o.normal[1] = s.n.y; o.normal[2] = s.n.z;
    o.shading_normal[0] = s.ns.x; o.shading_normal[1] = s.ns.y; o.shading_normal[2] = s.ns.z;
    o.uv[0] = s.u; o.uv[1] = s.v; o.material = s.material;
}
__device__ __forceinline__ void importIsect(const ptc_isect &p, Isect &s)
{
    s.point = mk(p.point[0], p.point[1], p.point[2]); s.wo = mk(p.wo[0], p.wo[1], p.wo[2]);
    s.n = mk(p.normal[0], p.normal[1], p.normal[2]); s.ns = mk(p.shading_normal[0], p.shading_normal[1], p.shading_normal[2]);
    s.u = p.uv[0]; s.v = p.uv[1]; s.material = p.material; s.prim = 0;
    makeFrame(s.ns, s.wo, s.tx, s.tz);
}

__global__ void intersectFullKernel(DScene scene, const ptc_ray *rays, uint32_t n, ptc_isect *out)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const ptc_ray r = rays[i];
        RayHit h;
        ptc_isect o;
        memset(&o, 0, sizeof(o));
        if (traverseBVH<false, false>(scene.bvh, r.origin[0], r.origin[1], r.origin[2], r.direction[0], r.direction[1], r.direction[2], PTC_TNEAR, PTC_TFAR, h, nullptr)) {
            Isect is;
            makeIsect(scene, mk(r.origin[0], r.origin[1], r.origin[2]), mk(r.direction[0], r.direction[1], r.direction[2]), h, is);
            exportIsect(is, h.t, o);
        } else { o.t = 3.402823466e+38f; o.material = PTC_INVALID_ID; }
        out[i] = o;
    }
}

__device__ __forceinline__ void exportEvents(const VolumeEvents &ev, uint32_t i, uint32_t *nEvents, float *eventT, uint32_t *eventMedium)
{
    if (nEvents) { nEvents[i] = ev.count; }
    for (uint32_t e = 0; e < PTC_MAX_EVENTS; e++) {
        const bool have = e < ev.count;
        if (eventT) { eventT[(size_t)i * PTC_MAX_EVENTS + e] = have ? ev.t[e] : 0.f; }
        if (eventMedium) { eventMedium[(size_t)i * PTC_MAX_EVENTS + e] = have ? (uint32_t)ev.medium[e] : PTC_NO_MEDIUM; }
    }
}

// Scene::testVolumetricIntersect, src/scene.cpp:225-353
__global__ void intersectVolumetricKernel(const __grid_constant__ DScene scene, const ptc_ray *rays, uint32_t n, ptc_isect *out, uint32_t *nEvents, float *eventT, uint32_t *eventMedium)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const ptc_ray r = rays[i];
        const V3 O = mk(r.origin[0], r.origin[1], r.origin[2]), D = mk(r.direction[0], r.direction[1], r.direction[2]);
        RayHit h; VolumeEvents ev;
        ptc_isect o;
        memset(&o, 0, sizeof(o));
        if (traverseFiltered<false>(scene, O, D, PTC_TNEAR, PTC_TFAR, h, ev)) {
            Isect is;
            makeIsect(scene, O, D, h, is);
            exportIsect(is, h.t, o);
        } else { o.t = 3.402823466e+38f; o.material = PTC_INVALID_ID; }
        out[i] = o;
        exportEvents(ev, i, nEvents, eventT, eventMedium);
    }
}

__global__ void occludedKernel(const __grid_constant__ DScene scene, const ptc_ray *rays, const float *maxT, uint32_t n, uint8_t *occluded)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const ptc_ray r = rays[i];
        occluded[i] = sceneOccluded(scene, mk(r.origin[0], r.origin[1], r.origin[2]), mk(r.direction[0], r.direction[1], r.direction[2]), maxT[i]) ? 1 : 0;
    }
}

// Scene::testVolumetricOcclusion, src/scene.cpp:383-424 (events are reported for unoccluded rays only)
__global__ void occludedVolumetricKernel(const __grid_constant__ DScene scene, const ptc_ray *rays, const float *maxT, uint32_t n, uint8_t *occluded, uint32_t *nEvents,
                                         float *eventT, uint32_t *eventMedium)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const ptc_ray r = rays[i];
        RayHit h; VolumeEvents ev;
        const bool occ = traverseFiltered<true>(scene, mk(r.origin[0], r.origin[1], r.origin[2]), mk(r.direction[0], r.direction[1], r.direction[2]), PTC_TNEAR, maxT[i] - 1e-3f, h, ev);
        if (occ) { ev.count = 0; }
        occluded[i] = occ ? 1 : 0;
        exportEvents(ev, i, nEvents, eventT, eventMedium);
    }
}


__global__ void cameraRaysKernel(DScene scene, const float *rowCol, uint32_t n, ptc_ray *rays)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        V3 o, d;
        cameraRay(scene, rowCol[2 * i], rowCol[2 * i + 1], o, d);
        ptc_ray r; r.origin[0] = o.x; r.origin[1] = o.y; r.origin[2] = o.z; r.direction[0] = d.x; r.direction[1] = d.y; r.direction[2] = d.z;
        rays[i] = r;
    }
}

__global__ void bsdfEvalKernel(DScene scene, uint32_t material, const ptc_isect *isects, const float *wi, uint32_t n, float *f, float *pdf)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        Isect s; importIsect(isects[i], s);
        float p;
        const V3 v = bsdfEval(scene.materials[material], s, mk(wi[3 * i], wi[3 * i + 1], wi[3 * i + 2]), p);
        f[3 * i] = v.x; f[3 * i + 1] = v.y; f[3 * i + 2] = v.z; pdf[i] = p;
    }
}

__global__ void bsdfSampleKernel(DScene scene, uint32_t material, const ptc_isect *isects, const float *xi, uint32_t n, float *wi, float *pdf, float *thr)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        Isect s; importIsect(isects[i], s);
        Rng rng; rng.initReplay(xi + 3 * i, 3);
        BsdfSample b;
        bsdfSample(scene.materials[material], s, rng, b);
        wi[3 * i] = b.wi.x; wi[3 * i + 1] = b.wi.y; wi[3 * i + 2] = b.wi.z; pdf[i] = b.pdf;
        thr[3 * i] = b.thr.x; thr[3 * i + 1] = b.thr.y; thr[3 * i + 2] = b.thr.z;
    }
}

__global__ void lightSampleKernel(DScene scene, const float *ref, const float *xi, uint32_t n, ptc_light_sample_t *out)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const V3 p = mk(ref[3 * i], ref[3 * i + 1], ref[3 * i + 2]);
        Rng rng; rng.initReplay(xi + 3 * i, 3);
        SurfSample ls;
        const DLight *l = sampleDirectLights(scene, p, rng, ls);
        ptc_light_sample_t o;
        o.point[0] = ls.point.x; o.point[1] = ls.point.y; o.point[2] = ls.point.z;
        o.normal[0] = ls.normal.x; o.normal[1] = ls.normal.y; o.normal[2] = ls.normal.z;
        o.inv_pdf = ls.invPDF; o.measure = ls.measure; o.solid_angle_pdf = solidAnglePdf(ls, p);
        const V3 lwo = -normalize(ls.point - p);
        const V3 e = l->kind == 2 ? envRadiance(scene, -lwo) : mk(l->emit[0], l->emit[1], l->emit[2]);
        o.emit[0] = e.x; o.emit[1] = e.y; o.emit[2] = e.z;
        out[i] = o;
    }
}

__global__ void lightPdfKernel(DScene scene, const ptc_ray *rays, uint32_t n, float *pdf)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const ptc_ray r = rays[i];
        const V3 O = mk(r.origin[0], r.origin[1], r.origin[2]), D = mk(r.direction[0], r.direction[1], r.direction[2]);
        RayHit h;
        if (traverseBVH<false, false>(scene.bvh, O.x, O.y, O.z, D.x, D.y, D.z, PTC_TNEAR, PTC_TFAR, h, nullptr)) {
            Isect s; makeIsect(scene, O, D, h, s);
            pdf[i] = scene.materials[s.material].emitter ? lightsPdf(scene, O, s) : -1.f;
        } else if (scene.hasEnv && !isBlack(envRadiance(scene, D))) {
            pdf[i] = -2.f - envPdf(scene, D) / (float)scene.nLights;
        } else { pdf[i] = -1.f; }
    }
}

__global__ void envRadianceKernel(DScene scene, const float *dirs, uint32_t n, float *rgb)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const V3 e = envRadiance(scene, mk(dirs[3 * i], dirs[3 * i + 1], dirs[3 * i + 2]));
        rgb[3 * i] = e.x; rgb[3 * i + 1] = e.y; rgb[3 * i + 2] = e.z;
    }
}

// samplePixel body + PathTracer::L as one sequential loop per path (test hook for the replayed random stream);
// uses the same device functions as the wavefront stages
__global__ void radianceReplayKernel(const __grid_constant__ DScene scene, const ptc_ray *rays, const float *xi, uint32_t stride, uint32_t n, int start, int last, float *rgb)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const ptc_ray r = rays[i];
        V3 O = mk(r.origin[0], r.origin[1], r.origin[2]), D = mk(r.direction[0], r.direction[1], r.direction[2]);
        Rng rng; rng.initReplay(xi + (size_t)i * stride, stride);
        V3 color = mk(0.f, 0.f, 0.f), result = mk(0.f, 0.f, 0.f), modulation = mk(1.f, 1.f, 1.f);
        RayHit h;
        Isect isect;
        if (!traverseBVH<false, false>(scene.bvh, O.x, O.y, O.z, D.x, D.y, D.z, PTC_TNEAR, PTC_TFAR, h, nullptr)) {
            color = envRadiance(scene, D);
        } else {
            makeIsect(scene, O, D, h, isect);
            if (checkCounts(start, last, 0)) {
                const DMaterial &m = scene.materials[isect.material];
                if (m.emitter && !(dot(isect.n, isect.wo) < 0.f)) { color = mk(m.emit[0], m.emit[1], m.emit[2]); }
                if (scene.hasFilter && m.type == PTC_PASSTHROUGH) {
                    float add[3];
                    cameraContainerTerm(scene, O.x, O.y, O.z, D.x, D.y, D.z, add);
                    color = color + mk(add[0], add[1], add[2]);
                }
            }
            BsdfSample bs;
            bsdfSample(scene.materials[isect.material], isect, rng, bs);
            for (int bounce = 1;;) {
                const DMaterial &m = scene.materials[isect.material];
                const bool wantDirect = checkCounts(start, last, bounce) && !m.emitter;
                V3 Ld = mk(0.f, 0.f, 0.f);
                if (wantDirect) {
                    V3 contribution, sd; float maxT;
                    if (directLightsSetup(scene, m, isect, bs, rng, contribution, sd, maxT)) {
                        if (!sceneOccluded(scene, isect.point, sd, maxT)) { Ld = Ld + contribution; }
                    }
                }
                const bool wantNext = !checkDone(last, bounce + 1);
                if (!wantDirect && !wantNext) { break; }
                Isect bi;
                const bool isHit = traverseBVH<false, false>(scene.bvh, isect.point.x, isect.point.y, isect.point.z, bs.wi.x, bs.wi.y, bs.wi.z, PTC_TNEAR, PTC_TFAR, h, nullptr);
                if (isHit) { makeIsect(scene, isect.point, bs.wi, h, bi); }
                const float cosT = fabsf(dot(isect.ns, bs.wi));
                if (wantDirect) {
                    Ld = Ld + directBsdf(scene, isect.point, cosT, bs.wi, bs.pdf, bs.thr, bs.delta, isHit, &bi);
                    result = result + Ld * modulation;
                }
                if (!wantNext) { break; }
                bounce++;
                if (!isHit) { break; }
                const float invPDF = 1.f / bs.pdf;
                modulation = modulation * ((bs.thr * cosT) * invPDF);
                if (isBlack(modulation)) { break; }
                bsdfSample(scene.materials[bi.material], bi, rng, bs);
                isect = bi;
            }
        }
        rgb[3 * i] = color.x + result.x; rgb[3 * i + 1] = color.y + result.y; rgb[3 * i + 2] = color.z + result.z;
    }
}

__global__ void volumeReplayKernel(const __grid_constant__ DScene scene, const ptc_ray *rays, const float *xi, uint32_t stride, uint32_t n, int start, int last, float *rgb)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const ptc_ray r = rays[i];
        Rng rng; rng.initReplay(xi + (size_t)i * stride, stride);
        VolumeWork work = {0, 0, {0, 0}, {0, 0}};
        const V3 L = volumeRadiance<false>(scene, mk(r.origin[0], r.origin[1], r.origin[2]), mk(r.direction[0], r.direction[1], r.direction[2]), rng, start, last, &work);
        rgb[3 * i] = L.x; rgb[3 * i + 1] = L.y; rgb[3 * i + 2] = L.z;
    }
}

// the counter-based generator on its own (known-answer tests: Random123's philox4x32-10 vectors, the draw order of a path vertex)
__global__ void philoxKernel(const uint32_t *counters, const uint32_t *keys, uint32_t n, uint32_t *out)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        uint32_t block[4];
        philox4x32_10(counters[4 * i], counters[4 * i + 1], counters[4 * i + 2], counters[4 * i + 3], keys[2 * i], keys[2 * i + 1], block);
        for (int c = 0; c < 4; c++) { out[4 * i + c] = block[c]; }
    }
}
__global__ void uniformsKernel(uint64_t seed, const uint32_t *streams, uint32_t nStreams, uint32_t draws, float *out)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < nStreams; i += gridDim.x * blockDim.x) {
        Rng rng;
        rng.initPhilox(seed, streams[3 * i], streams[3 * i + 1]);
        rng.beginVertex(streams[3 * i + 2]);
        for (uint32_t d = 0; d < draws; d++) { out[(size_t)i * draws + d] = rng.next(); }
    }
}

// ================================================================================================ host context
struct HostGeometry {
    int32_t medium = -1; // Surface::m_internalMedium of every surface of the geometry
    bool isSphere = false;
    uint32_t firstVertex = 0, nVertices = 0, firstPrim = 0, nPrims = 0;
    float centerRadius[4] = {0, 0, 0, 0};
    uint32_t sphereMaterial = 0;
    // SURVEY 8(f) N4: the scene the geometry is attached to (0 = root) and its geometry id there; a placement of an instance scene
    // (RTC_GEOMETRY_TYPE_INSTANCE) is a geometry too: it takes an id, and carries the instanced scene and its local-to-world map
    uint32_t scene = 0, localId = 0;
    bool isInstance = false;
    uint32_t instanceScene = 0;
    float l2w[12] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0}; // rows of the 3x4 affine map
    float w2l[12] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0}; // its inverse as Embree keeps it (Instance::setTransform: world2local = rcp(local2world))
};
struct HostScene { uint32_t nGeoms = 0; std::vector<uint32_t> members; }; // members: indices into ptc_ctx::geometries, attach order

// Owners of the CUDA resources a context (or a query's scope) holds: each is released with its owner, so no release is listed anywhere.
// Buffer: `size()` elements of device memory, or of page-locked host memory when PINNED.  resize(n) reallocates when n differs from
// the size, reserve(n) only when n is larger; the contents after a reallocation are undefined.
template <typename T, bool PINNED = false>
class Buffer {
public:
    Buffer() = default;
    Buffer(T *p, size_t n) : p_(p), n_(n) {} // takes ownership of an allocation made elsewhere
    Buffer(Buffer &&o) noexcept : p_(o.p_), n_(o.n_) { o.p_ = nullptr; o.n_ = 0; }
    Buffer &operator=(Buffer &&o) noexcept { std::swap(p_, o.p_); std::swap(n_, o.n_); return *this; }
    ~Buffer() { release(); }
    cudaError_t resize(size_t n)
    {
        if (n == n_) { return cudaSuccess; }
        release();
        const cudaError_t e = PINNED ? cudaMallocHost((void **)&p_, n * sizeof(T)) : cudaMalloc((void **)&p_, n * sizeof(T));
        if (e == cudaSuccess) { n_ = n; } else { p_ = nullptr; }
        return e;
    }
    cudaError_t reserve(size_t n) { return n > n_ ? resize(n) : cudaSuccess; }
    T *get() const { return p_; }
    size_t size() const { return n_; }
private:
    void release() { if (p_) { if (PINNED) { cudaFreeHost(p_); } else { cudaFree(p_); } } p_ = nullptr; n_ = 0; }
    T *p_ = nullptr; size_t n_ = 0;
};
template <typename T> using PinnedBuffer = Buffer<T, true>;
// A non-blocking stream and an event; create() makes the handle on its first call (events without timing unless asked)
class Stream {
public:
    Stream() = default;
    Stream(Stream &&o) noexcept : s_(o.s_) { o.s_ = nullptr; }
    Stream &operator=(Stream &&o) noexcept { std::swap(s_, o.s_); return *this; }
    ~Stream() { if (s_) { cudaStreamDestroy(s_); } }
    cudaError_t create() { return s_ ? cudaSuccess : cudaStreamCreateWithFlags(&s_, cudaStreamNonBlocking); }
    operator cudaStream_t() const { return s_; }
private:
    cudaStream_t s_ = nullptr;
};
class Event {
public:
    Event() = default;
    Event(Event &&o) noexcept : e_(o.e_) { o.e_ = nullptr; }
    Event &operator=(Event &&o) noexcept { std::swap(e_, o.e_); return *this; }
    ~Event() { if (e_) { cudaEventDestroy(e_); } }
    cudaError_t create(unsigned flags = cudaEventDisableTiming) { return e_ ? cudaSuccess : cudaEventCreateWithFlags(&e_, flags); }
    operator cudaEvent_t() const { return e_; }
private:
    cudaEvent_t e_ = nullptr;
};

// What ptc_add_* / ptc_set_environment / ptc_begin|end_instance accumulate for ptc_commit, which releases it
struct Staging {
    std::vector<ptc_material_desc> materials;
    struct HostTexture { std::vector<uint32_t> texels; int width, height; };
    std::vector<HostTexture> textures;
    std::vector<float> positions4, normals4, uvs2;
    std::vector<uint32_t> prims4, primIds2;
    std::vector<HostGeometry> geometries;
    std::vector<HostScene> scenes = std::vector<HostScene>(1); // [0] = the root scene
    std::vector<uint32_t> sceneStack;                          // instance scenes being described (parseInstance recurses)
    std::vector<uint32_t> rootGeometry;                        // root geometry id -> index into geometries
    struct HostMedium { float sigmaT[3], sigmaS[3]; };
    std::vector<HostMedium> media;
    bool hasEnv = false; std::vector<float> envRgba; int envW = 0, envH = 0; float envScale = 1.f; float envM2W[16], envW2M[16];
};

// One device allocation of a committed scene and what points at it: the DScene field at byte offset `field` (NO_FIELD: none), and
// for texels the material-table entries whose `texels` it holds.  ptc_replicate points them at its copy.
static constexpr size_t NO_FIELD = ~(size_t)0; struct SceneAllocation { Buffer<uint8_t> data; size_t field; std::vector<uint32_t> materials; };

// The committed scene as the renders and queries read it.  ptc_commit assembles a Committed and moves it into the context once every
// step succeeded; ptc_replicate assigns this part to the replica.
struct SceneState {
    DScene view = {};                 // the kernels' parameter; before ptc_commit only its camera is set
    std::vector<DMaterial> materials; // the material table as uploaded (texel pointers included)
    uint32_t classMask = 0;           // material classes present in the scene
    uint32_t bvhTriangles = 0, bvhDepth = 0, bvhPlocIterations = 0; float bvhBuildMs = 0.f; // ptc_get_stats (nodes: view.bvh.nNodes)
    std::vector<float> placements;    // host copy of view.bvh.placements (ptc_count_traversal)
};
struct Committed : SceneState {
    std::vector<SceneAllocation> allocations; // the device memory `view` and `materials` point into
    Buffer<uint8_t> buildWorkspace;           // the device builder's working set, released with the context (bvh.h: buildWideBVHDevice)
};

// ptc_set_option's settings and the integrator: what a replica inherits
struct Options {
    int integrator = PTC_INTEGRATOR_PATH_TRACER;
    int64_t pathsPerWave = 1 << 27; // up to 134 M paths x 237 B = 31.8 GB of path state per wave (of 180 GB; allocated for the paths a render call needs):
                                    // the queues of the late bounces (1 % of the paths) stay long enough to keep 148 SMs busy.  Dragon workload: 613 / 648 / 653
                                    // Msamples/s with 2^24 / 2^26 / 2^27; teapot 1920x1080, 64-spp steps: 2306 (two waves of 32 spp at 2^26) vs 2374 (one wave)
    bool stageTiming = false, countTraversal = false;
    // the shadow rays of a bounce are traced on a second stream, concurrently with the bounce's extend rays: both grids fill the GPU, so
    // the shadow CTAs become resident as the extend kernel drains -- the tail of one launch is filled with the head of the other
    bool overlapShadow = true;
    // A wave is traced as `lanes` interleaved part-waves (consecutive blocks of the wave's samples, each with its own share of the path
    // state, its own counters and streams): while one lane's paths are in a shading stage (waiting on dependent loads, half of the issue
    // slots idle) another lane's rays are in a traversal stage (issue-bound, hardly any DRAM traffic), and the SMs hold CTAs of both.
    // Lane 0 runs on the caller's stream; the samples are still added to the image in sample order (launchWave), so the result does
    // not depend on the number of lanes.
    int lanes = 0; // 0 = chosen per wave (renderInternal)
    // VolumePathTracer as wavefront stages (volume_wavefront.cuh); volumeMegakernel = 1 keeps the one-thread-per-path kernel
    bool volumeMegakernel = false;
    int bvhBuilder = 1; // 1: device builder (bvh_build_gpu.cu), 0: host binned-SAH builder (bvh_build.cu)
    bool framebufferMoments = false; // see ptc_ctx::moments
};

struct ptc_ctx {
    int device = 0;
    std::string error;
    bool committed = false, hasCamera = false;
    Staging staged; Committed scene; Options options;
    std::optional<WideBVH> hostBvh; // host copy of the device BVH, fetched when ptc_count_traversal first walks it
    Buffer<float4> volumeOut; Buffer<uint32_t> volumeCursor;
    int gridVolume = 0;
    VolumeBuffers volumeBuffers = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr}; Buffer<uint8_t> volumeArrays[6];
    int gridVolumeTraverse = 0, gridVolumeLogic = 0, gridVolumeShade = 0;
    PathBuffers paths; uint32_t pathCapacity = 0; Buffer<uint8_t> pathSlab;
    Buffer<uint32_t> classQueues[PTC_MATERIAL_CLASSES];
    Buffer<BounceCounters> counters;
    Buffer<unsigned long long> totals;
    Buffer<float> accumScratch;
    Buffer<float> framebuffer, gatherStage;
    Event framebufferReady;
    std::vector<Buffer<float>> snapshots;                // checkpoint copies of the framebuffer (ptc_framebuffer_render_checkpoints)
    // snapshots allocated with option framebuffer_moments on hold the sums and then the second moments (accumulateKernel<true>); a
    // snapshot's moments are complete when they cover every sample its sums hold (momentsComplete when it was written)
    bool snapshotsHoldMoments = false;
    size_t snapshotSize = 0; // floats of sums per snapshot: the framebuffer size they were allocated for
    std::vector<bool> snapshotMomentsComplete;
    struct Gather { Buffer<float> device; PinnedBuffer<float> pinned; Event done; bool busy = false; };
    std::vector<Gather> gathers;                         // results of ptc_framebuffer_gather_begin in flight
    Event gatherRead;                                    // the last gather kernel of this (root) context finished reading the framebuffers
    PinnedBuffer<float> pinned;
    // ptc_render: the caller's radianceLookup is uploaded on its own stream while the first wave's kernels run (uploadSums)
    Stream copyStream; Event uploadDone;
    Stream stream;
    Event evStart, evStop;
    int numSMs = 148;
    int gridTraverse = 0, gridShade = 0, gridLogic = 0, gridSimple = 0;
    int gridTraverseShared = 0, gridVolumeTraverseShared = 0; // traversal grids of a wave traced as several lanes: two CTAs per SM fewer
    Stream shadowStream; Event shadeDone, shadowDone;
    struct Lane { Stream stream, shadowStream; Event shadeDone, shadowDone, done; Buffer<BounceCounters> counters; };
    std::vector<Lane> extraLanes; // lanes 1 ..
    Event laneFork;
    // adaptive sampling (ptc_adaptive_*): between begin and the next ptc_framebuffer_clear the framebuffer belongs to the passes.
    // Per pixel: second moments (`moments` below), sample count, and two list entries (active pixels, the stopping test's output)
    // = 24 B, plus cub's selection scratch
    struct Adaptive {
        bool on = false;
        ptc_adaptive_desc desc = {0.f, 0, 0, 0};
        uint32_t n = 0, active = 0; // the samples every active pixel holds; pixels still active
        size_t pixels = 0;          // what the buffers are sized for
        Buffer<uint32_t> counts, list, next, selected;
        PinnedBuffer<uint32_t> selectedHost;
        Buffer<uint8_t> scratch;
    } adaptive;
    // The second moments (3 x fp32 per pixel, next to the framebuffer's sums): the squared samples that the adaptive passes add, and,
    // with option "framebuffer_moments" (options.framebufferMoments), the framebuffer renders; zeroed by ptc_adaptive_begin and, with the option
    // on, by ptc_framebuffer_clear.  The input of ptc_denoise that PTC_GATHER_MOMENTS gathers.  momentsComplete: they cover every
    // sample the framebuffer holds (an adaptive render, or the option on at the last clear and at every render since); the gather
    // refuses them otherwise
    bool momentsOption = false, momentsComplete = false;
    Buffer<float> moments;
    // ptc_denoise's device buffers: the staged inputs (15 x 4 B per pixel) and guide records (32 B); two colour records (16 B each),
    // which ptc_framebuffer_denoise_begin uses as well
    struct Denoise { Buffer<float> inputs; Buffer<float4> guide, colour[2]; } denoise;
    // the device guide sums of ptc_framebuffer_guides (8 x 4 B per pixel)
    Buffer<float> aovs;
    // ptc_framebuffer_guides: the guide records (32 B per pixel) ptc_framebuffer_denoise_begin filters with; aovSpp = 0: none
    struct Guides { int width = 0, height = 0; Buffer<float4> records; uint32_t aovSpp = 0; } guides;
    uint64_t samples = 0, launches = 0;
    float lastRenderMs = 0.f;
    // stage timing: CUDA events on the launching stream around every launch, summed per kernel class
    struct Timed { Event a, b; int kind; };
    std::vector<Timed> pending;
    std::vector<Event> eventPool;
    double stageMs[4] = {0, 0, 0, 0};
    uint64_t stageLaunches[4] = {0, 0, 0, 0};
};

enum { STAGE_EXTEND = 0, STAGE_SHADOW = 1, STAGE_SHADE = 2, STAGE_OTHER = 3 };

static Event takeEvent(ptc_ctx *ctx)
{
    Event e;
    if (!ctx->eventPool.empty()) { e = std::move(ctx->eventPool.back()); ctx->eventPool.pop_back(); }
    else { e.create(cudaEventDefault); }
    return e;
}
static void collectTimings(ptc_ctx *ctx)
{
    for (ptc_ctx::Timed &t : ctx->pending) {
        float ms = 0.f;
        cudaEventSynchronize(t.b);
        cudaEventElapsedTime(&ms, t.a, t.b);
        ctx->stageMs[t.kind] += ms; ctx->stageLaunches[t.kind]++;
        ctx->eventPool.push_back(std::move(t.a)); ctx->eventPool.push_back(std::move(t.b));
    }
    ctx->pending.clear();
}
struct StageTimer { // brackets one launch when stage timing is on
    ptc_ctx *ctx; cudaStream_t stream; Event a; int kind;
    StageTimer(ptc_ctx *c, cudaStream_t s, int k) : ctx(c), stream(s), kind(k)
    {
        if (ctx->options.stageTiming) { a = takeEvent(ctx); cudaEventRecord(a, stream); }
    }
    ~StageTimer()
    {
        if (a) { Event b = takeEvent(ctx); cudaEventRecord(b, stream); ctx->pending.push_back({std::move(a), std::move(b), kind}); }
    }
};

#define CTX_FAIL(ctx, code, ...) do { char _b[512]; snprintf(_b, sizeof(_b), __VA_ARGS__); (ctx)->error = _b; return (code); } while (0)
#define CUDA_TRY(ctx, call) do { cudaError_t _e = (call); if (_e != cudaSuccess) { CTX_FAIL(ctx, PTC_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(_e)); } } while (0)
#define TRY(call) do { const int _rc = (call); if (_rc) { return _rc; } } while (0)

// grid of a grid-stride launch over n >= 1 items
static inline uint32_t gridFor(ptc_ctx *ctx, uint32_t n, uint32_t block = 128) { return std::max(1u, std::min<uint32_t>((n + block - 1) / block, (uint32_t)ctx->gridSimple * 4)); }

// byte offset of `field` inside `s` (SceneAllocation::field)
static size_t fieldOf(const DScene &s, const void *field) { return (size_t)((const char *)field - (const char *)&s); }
// A new device allocation holding `count` elements of `src` (at least one element is allocated), appended to `to`
template <typename T>
static int upload(ptc_ctx *ctx, std::vector<SceneAllocation> &to, const T *src, size_t count, const T **dst, size_t field = NO_FIELD)
{
    Buffer<uint8_t> b;
    CUDA_TRY(ctx, b.resize(std::max<size_t>(count, 1) * sizeof(T)));
    *dst = (const T *)b.get();
    to.push_back({std::move(b), field, {}});
    if (count) { CUDA_TRY(ctx, cudaMemcpy((void *)*dst, src, count * sizeof(T), cudaMemcpyHostToDevice)); }
    return PTC_OK;
}
// ... into the scene `c`, recorded as what its DScene's `field` points at
template <typename T>
static int upload(ptc_ctx *ctx, Committed &c, const T *src, size_t count, const T *&field)
{
    return upload(ctx, c.allocations, src, count, &field, fieldOf(c.view, &field));
}

// Texture::lookup's powf(c / 255.f, 2.2f) (src/texture.cpp:44-48), one table for all textures on the current device
static cudaError_t uploadGammaTable()
{
    float gamma[256]; for (int c = 0; c < 256; c++) { gamma[c] = powf(c / 255.f, 2.2f); }
    return cudaMemcpyToSymbol(c_gammaTable, gamma, sizeof(gamma));
}

extern "C" {

int ptc_create(int device, ptc_ctx **out)
{
    if (!out) { return PTC_ERR_INVALID; }
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) {
        fprintf(stderr, "pathed_cuda: no CUDA device available; this library has no CPU fallback\n");
        return PTC_ERR_CUDA;
    }
    if (device < 0 || device >= count) { return PTC_ERR_INVALID; }
    if (cudaSetDevice(device) != cudaSuccess) { return PTC_ERR_CUDA; }
    ptc_ctx *ctx = new ptc_ctx();
    ctx->device = device;
    memset(&ctx->paths, 0, sizeof(ctx->paths));
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) { ctx->numSMs = prop.multiProcessorCount; }
    if (ctx->stream.create() != cudaSuccess || ctx->shadowStream.create() != cudaSuccess || ctx->copyStream.create() != cudaSuccess ||
        ctx->uploadDone.create() != cudaSuccess || ctx->shadeDone.create() != cudaSuccess || ctx->shadowDone.create() != cudaSuccess ||
        ctx->evStart.create(cudaEventDefault) != cudaSuccess || ctx->evStop.create(cudaEventDefault) != cudaSuccess ||
        ctx->counters.resize(CNT_STRIDE) != cudaSuccess || ctx->totals.resize(6) != cudaSuccess) {
        delete ctx;
        return PTC_ERR_CUDA;
    }
    cudaMemset(ctx->totals.get(), 0, 6 * sizeof(unsigned long long));
    int perSM = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, (traverseKernel<false, false>), 128, 0);
    ctx->gridTraverse = ctx->numSMs * std::max(perSM, 1);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, logicKernel, 256, 0);
    ctx->gridLogic = ctx->numSMs * std::max(perSM, 1);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, (materialKernel<PTC_PLASTIC, false>), 128, 0);
    ctx->gridShade = ctx->numSMs * std::max(perSM, 1);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, volumePathKernel<false>, 128, 0);
    ctx->gridVolume = ctx->numSMs * std::max(perSM, 1);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, (volumeTraverseKernel<VOL_EXTEND, false>), 128, 0);
    ctx->gridVolumeTraverse = ctx->numSMs * std::max(perSM, 1);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, volumeLogicKernel, 256, 0);
    ctx->gridVolumeLogic = ctx->numSMs * std::max(perSM, 1);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, volumeMaterialKernel<PTC_PLASTIC>, 128, 0);
    ctx->gridVolumeShade = ctx->numSMs * std::max(perSM, 1);
    ctx->gridSimple = ctx->numSMs * 8;
    ctx->gridTraverseShared = std::max(ctx->numSMs, ctx->gridTraverse - 2 * ctx->numSMs);
    ctx->gridVolumeTraverseShared = std::max(ctx->numSMs, ctx->gridVolumeTraverse - 2 * ctx->numSMs);
    // tuning hooks (tools/sweep_lanes.sh): number of interleaved lanes and CTAs per SM of the persistent grids
    if (const char *e = getenv("PTC_LANES")) { ctx->options.lanes = std::min(PTC_MAX_LANES, std::max(0, atoi(e))); }
    if (const char *e = getenv("PTC_TRAVERSE_PER_SM")) { ctx->gridTraverse = ctx->gridTraverseShared = ctx->numSMs * std::max(1, atoi(e)); }
    if (const char *e = getenv("PTC_VOLUME_TRAVERSE_PER_SM")) { ctx->gridVolumeTraverse = ctx->gridVolumeTraverseShared = ctx->numSMs * std::max(1, atoi(e)); }
    if (const char *e = getenv("PTC_LOGIC_PER_SM")) { ctx->gridLogic = ctx->numSMs * std::max(1, atoi(e)); }
    if (const char *e = getenv("PTC_SHADE_PER_SM")) { ctx->gridShade = ctx->numSMs * std::max(1, atoi(e)); }
    *out = ctx;
    return PTC_OK;
}

void ptc_destroy(ptc_ctx *ctx)
{
    if (!ctx) { return; }
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    collectTimings(ctx);
    delete ctx; // the members release the context's buffers, streams and events
}

const char *ptc_last_error(ptc_ctx *ctx) { return ctx ? ctx->error.c_str() : "null context"; }

int ptc_add_texture(ptc_ctx *ctx, const uint8_t *rgb, int width, int height, uint32_t *id)
{
    if (!ctx || !rgb) { return PTC_ERR_INVALID; }
    if (ctx->committed) { CTX_FAIL(ctx, PTC_ERR_STATE, "scene already committed"); }
    if (width <= 0 || height <= 0) { CTX_FAIL(ctx, PTC_ERR_INVALID, "Error loading texture: %d x %d", width, height); }
    Staging::HostTexture t;
    t.width = width; t.height = height;
    t.texels.resize((size_t)width * height);
    for (size_t i = 0; i < t.texels.size(); i++) { t.texels[i] = (uint32_t)rgb[3 * i] | ((uint32_t)rgb[3 * i + 1] << 8) | ((uint32_t)rgb[3 * i + 2] << 16); }
    ctx->staged.textures.push_back(std::move(t));
    if (id) { *id = (uint32_t)ctx->staged.textures.size() - 1; }
    return PTC_OK;
}

int ptc_add_material(ptc_ctx *ctx, const ptc_material_desc *desc, uint32_t *id)
{
    if (!ctx || !desc) { return PTC_ERR_INVALID; }
    if (ctx->committed) { CTX_FAIL(ctx, PTC_ERR_STATE, "scene already committed"); }
    if (desc->type < PTC_LAMBERTIAN || desc->type > PTC_PASSTHROUGH) { CTX_FAIL(ctx, PTC_ERR_INVALID, "Unimplemented material type %d", desc->type); }
    if (desc->albedo_kind == PTC_ALBEDO_TEXTURE) {
        if (desc->type != PTC_LAMBERTIAN && desc->type != PTC_PLASTIC) { CTX_FAIL(ctx, PTC_ERR_INVALID, "only Lambertian and Plastic take a texture (src/scene_parser.cpp:625-647)"); }
        if (desc->texture >= ctx->staged.textures.size()) { CTX_FAIL(ctx, PTC_ERR_INVALID, "texture id %u out of range", desc->texture); }
    } else if (desc->albedo_kind != PTC_ALBEDO_CONSTANT && desc->albedo_kind != PTC_ALBEDO_CHECKERBOARD) {
        CTX_FAIL(ctx, PTC_ERR_INVALID, "Unimplemented albedo kind %d", desc->albedo_kind);
    }
    if ((desc->type == PTC_MICROFACET || desc->type == PTC_PLASTIC) && desc->distribution != PTC_BECKMANN && desc->distribution != PTC_GGX) {
        CTX_FAIL(ctx, PTC_ERR_INVALID, "Unimplemented distribution %d", desc->distribution);
    }
    ctx->staged.materials.push_back(*desc);
    if (id) { *id = (uint32_t)ctx->staged.materials.size() - 1; }
    return PTC_OK;
}

int ptc_add_medium(ptc_ctx *ctx, const float sigmaT[3], const float sigmaS[3], uint32_t *id)
{
    if (!ctx || !sigmaT) { return PTC_ERR_INVALID; }
    if (ctx->committed) { CTX_FAIL(ctx, PTC_ERR_STATE, "scene already committed"); }
    Staging::HostMedium m;
    for (int c = 0; c < 3; c++) { m.sigmaT[c] = sigmaT[c]; m.sigmaS[c] = sigmaS ? sigmaS[c] : 0.f; }
    ctx->staged.media.push_back(m);
    if (id) { *id = (uint32_t)ctx->staged.media.size() - 1; }
    return PTC_OK;
}

int ptc_set_internal_medium(ptc_ctx *ctx, uint32_t geom, uint32_t medium)
{
    if (!ctx) { return PTC_ERR_INVALID; }
    if (ctx->committed) { CTX_FAIL(ctx, PTC_ERR_STATE, "scene already committed"); }
    if (geom >= ctx->staged.rootGeometry.size() || ctx->staged.geometries[ctx->staged.rootGeometry[geom]].isInstance) { CTX_FAIL(ctx, PTC_ERR_INVALID, "geometry id %u out of range", geom); }
    if (medium != PTC_NO_MEDIUM && medium >= ctx->staged.media.size()) { CTX_FAIL(ctx, PTC_ERR_INVALID, "medium id %u out of range", medium); }
    ctx->staged.geometries[ctx->staged.rootGeometry[geom]].medium = medium == PTC_NO_MEDIUM ? -1 : (int32_t)medium;
    return PTC_OK;
}

int ptc_set_integrator(ptc_ctx *ctx, int integrator)
{
    if (!ctx) { return PTC_ERR_INVALID; }
    if (integrator != PTC_INTEGRATOR_PATH_TRACER && integrator != PTC_INTEGRATOR_VOLUME_PATH_TRACER) { CTX_FAIL(ctx, PTC_ERR_INVALID, "Unimplemented integrator %d", integrator); }
    ctx->options.integrator = integrator;
    return PTC_OK;
}

// rtcAttachGeometry: the next geometry id of the scene being described
static uint32_t attachGeometry(ptc_ctx *ctx, HostGeometry &g)
{
    g.scene = ctx->staged.sceneStack.empty() ? 0u : ctx->staged.sceneStack.back();
    g.localId = ctx->staged.scenes[g.scene].nGeoms++;
    ctx->staged.scenes[g.scene].members.push_back((uint32_t)ctx->staged.geometries.size());
    if (g.scene == 0) { ctx->staged.rootGeometry.push_back((uint32_t)ctx->staged.geometries.size()); }
    ctx->staged.geometries.push_back(g);
    return g.localId;
}

int ptc_begin_instance(ptc_ctx *ctx, uint32_t *sceneOut)
{
    if (!ctx) { return PTC_ERR_INVALID; }
    if (ctx->committed) { CTX_FAIL(ctx, PTC_ERR_STATE, "scene already committed"); }
    if (ctx->staged.sceneStack.size() >= 8) { CTX_FAIL(ctx, PTC_ERR_INVALID, "instance definitions nested too deeply"); }
    ctx->staged.scenes.push_back(HostScene());
    ctx->staged.sceneStack.push_back((uint32_t)ctx->staged.scenes.size() - 1);
    if (sceneOut) { *sceneOut = ctx->staged.sceneStack.back(); }
    return PTC_OK;
}

int ptc_end_instance(ptc_ctx *ctx)
{
    if (!ctx) { return PTC_ERR_INVALID; }
    if (ctx->committed) { CTX_FAIL(ctx, PTC_ERR_STATE, "scene already committed"); }
    if (ctx->staged.sceneStack.empty()) { CTX_FAIL(ctx, PTC_ERR_STATE, "ptc_end_instance without ptc_begin_instance"); }
    ctx->staged.sceneStack.pop_back();
    return PTC_OK;
}

// Instance::setTransform's world2local0 = rcp(local2world) (ext/embree/kernels/common/scene_instance.cpp:77-85; part of Embree's
// lowest-ISA build: no fused multiply-add).  common/math/affinespace.h:91 and linearspace3.h:57-63: l^-1 = adjoint(l) / det(l) with a
// true division per element, the adjoint's rows = cross products of l's columns, det summed as (x + y) + z, and
// p' = -(p.x * c0 + (p.y * c1 + p.z * c2)) over the columns c of l^-1.  The order matters: the ray origin in the instance's space is
// rounded at the magnitude of the transformed point, so one ulp in this matrix moves t of a short bounce ray by 1e-5 and more.
static void inverseAffine(const float l2w[12], float w2l[12])
{
    const float vx[3] = {l2w[0], l2w[4], l2w[8]}, vy[3] = {l2w[1], l2w[5], l2w[9]}, vz[3] = {l2w[2], l2w[6], l2w[10]};
    auto cross = [](const float *a, const float *b, volatile float *out) { out[0] = a[1] * b[2] - a[2] * b[1]; out[1] = a[2] * b[0] - a[0] * b[2]; out[2] = a[0] * b[1] - a[1] * b[0]; };
    volatile float rows[3][3]; // volatile: every product and sum is rounded to float on its own, whatever the host compiler's contraction setting
    cross(vy, vz, rows[0]); cross(vz, vx, rows[1]); cross(vx, vy, rows[2]);
    volatile float p0 = vx[0] * rows[0][0], p1 = vx[1] * rows[0][1], p2 = vx[2] * rows[0][2];
    volatile float s01 = p0 + p1;
    const float det = s01 + p2;
    for (int i = 0; i < 3; i++) {
        for (int j = 0; j < 3; j++) { w2l[4 * i + j] = rows[i][j] / det; }
        volatile float a = l2w[3] * w2l[4 * i], b = l2w[7] * w2l[4 * i + 1], c = l2w[11] * w2l[4 * i + 2];
        volatile float bc = b + c;
        w2l[4 * i + 3] = -(a + bc);
    }
}

int ptc_add_instance(ptc_ctx *ctx, uint32_t scene, const float m[16], uint32_t *geomId)
{
    if (!ctx || !m) { return PTC_ERR_INVALID; }
    if (ctx->committed) { CTX_FAIL(ctx, PTC_ERR_STATE, "scene already committed"); }
    if (scene == 0 || scene >= ctx->staged.scenes.size()) { CTX_FAIL(ctx, PTC_ERR_INVALID, "unknown instance scene %u", scene); }
    for (uint32_t open : ctx->staged.sceneStack) { if (open == scene) { CTX_FAIL(ctx, PTC_ERR_INVALID, "an instance scene cannot contain itself"); } }
    HostGeometry g;
    g.isInstance = true; g.instanceScene = scene;
    for (int row = 0; row < 3; row++) { for (int col = 0; col < 4; col++) { g.l2w[4 * row + col] = m[4 * col + row]; } } // RTC_FORMAT_FLOAT4X4_COLUMN_MAJOR
    inverseAffine(g.l2w, g.w2l);
    const uint32_t id = attachGeometry(ctx, g);
    if (geomId) { *geomId = id; }
    return PTC_OK;
}

int ptc_add_triangle_mesh(ptc_ctx *ctx, const float *P, const float *N, const float *UV, uint32_t nv, const uint32_t *I,
                          const uint32_t *mat, uint32_t nt, uint32_t *geomId)
{
    if (!ctx || (nv && !P) || (nt && (!I || !mat))) { return PTC_ERR_INVALID; }
    if (ctx->committed) { CTX_FAIL(ctx, PTC_ERR_STATE, "scene already committed"); }
    for (uint32_t t = 0; t < nt; t++) {
        if (mat[t] >= ctx->staged.materials.size()) { CTX_FAIL(ctx, PTC_ERR_INVALID, "material id %u out of range", mat[t]); }
        for (int k = 0; k < 3; k++) { if (I[3 * (size_t)t + k] >= nv) { CTX_FAIL(ctx, PTC_ERR_INVALID, "vertex index out of range in triangle %u", t); } }
    }
    HostGeometry g;
    g.firstVertex = (uint32_t)(ctx->staged.positions4.size() / 4);
    g.nVertices = nv;
    g.firstPrim = (uint32_t)(ctx->staged.prims4.size() / 4);
    g.nPrims = nt;
    const uint32_t geom = ctx->staged.scenes[ctx->staged.sceneStack.empty() ? 0u : ctx->staged.sceneStack.back()].nGeoms; // the id attachGeometry hands out below
    for (uint32_t v = 0; v < nv; v++) {
        ctx->staged.positions4.insert(ctx->staged.positions4.end(), {P[3 * (size_t)v], P[3 * (size_t)v + 1], P[3 * (size_t)v + 2], 0.f});
        if (N) { ctx->staged.normals4.insert(ctx->staged.normals4.end(), {N[3 * (size_t)v], N[3 * (size_t)v + 1], N[3 * (size_t)v + 2], 0.f}); }
        else { ctx->staged.normals4.insert(ctx->staged.normals4.end(), {0.f, 0.f, 0.f, 0.f}); }
        if (UV) { ctx->staged.uvs2.insert(ctx->staged.uvs2.end(), {UV[2 * (size_t)v], UV[2 * (size_t)v + 1]}); }
        else { ctx->staged.uvs2.insert(ctx->staged.uvs2.end(), {0.f, 0.f}); }
    }
    for (uint32_t t = 0; t < nt; t++) {
        ctx->staged.prims4.insert(ctx->staged.prims4.end(), {I[3 * (size_t)t] + g.firstVertex, I[3 * (size_t)t + 1] + g.firstVertex, I[3 * (size_t)t + 2] + g.firstVertex, mat[t]});
        ctx->staged.primIds2.insert(ctx->staged.primIds2.end(), {geom, t});
    }
    attachGeometry(ctx, g);
    if (geomId) { *geomId = geom; }
    return PTC_OK;
}

int ptc_add_sphere(ptc_ctx *ctx, const float cr[4], uint32_t material, uint32_t *geomId)
{
    if (!ctx || !cr) { return PTC_ERR_INVALID; }
    if (ctx->committed) { CTX_FAIL(ctx, PTC_ERR_STATE, "scene already committed"); }
    if (material >= ctx->staged.materials.size()) { CTX_FAIL(ctx, PTC_ERR_INVALID, "material id %u out of range", material); }
    if (!ctx->staged.sceneStack.empty()) { CTX_FAIL(ctx, PTC_ERR_INVALID, "only triangle meshes can be instanced (src/sphere.cpp:46 attaches spheres to the global scene)"); }
    HostGeometry g;
    g.isSphere = true; g.nPrims = 1; memcpy(g.centerRadius, cr, sizeof(g.centerRadius)); g.sphereMaterial = material;
    const uint32_t id = attachGeometry(ctx, g);
    if (geomId) { *geomId = id; }
    return PTC_OK;
}

int ptc_set_environment(ptc_ctx *ctx, const float *rgba, int w, int h, float scale, const float m2w[16], const float w2m[16])
{
    if (!ctx || !rgba || w <= 0 || h <= 0 || !m2w || !w2m) { return PTC_ERR_INVALID; }
    if (w > 65535 || h > 65535) { CTX_FAIL(ctx, PTC_ERR_INVALID, "environment map larger than 65535 texels on a side"); }
    if (ctx->committed) { CTX_FAIL(ctx, PTC_ERR_STATE, "scene already committed"); }
    ctx->staged.envRgba.assign(rgba, rgba + (size_t)w * h * 4);
    ctx->staged.envW = w; ctx->staged.envH = h; ctx->staged.envScale = scale;
    memcpy(ctx->staged.envM2W, m2w, sizeof(ctx->staged.envM2W)); memcpy(ctx->staged.envW2M, w2m, sizeof(ctx->staged.envW2M));
    ctx->staged.hasEnv = true;
    return PTC_OK;
}

int ptc_set_camera(ptc_ctx *ctx, const float o[3], const float t[3], const float up[3], float vfov, int w, int h, int flip)
{
    if (!ctx || !o || !t || !up || w <= 0 || h <= 0) { return PTC_ERR_INVALID; }
    // lookAt, src/transform.cpp:138-164 (host arithmetic in the reference's order)
    auto norm = [](const float v[3], float out[3]) { const float n = sqrtf(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]); out[0] = v[0] / n; out[1] = v[1] / n; out[2] = v[2] / n; };
    auto crossp = [](const float a[3], const float b[3], float out[3]) { out[0] = (a[1] * b[2]) - (a[2] * b[1]); out[1] = (a[2] * b[0]) - (a[0] * b[2]); out[2] = (a[0] * b[1]) - (a[1] * b[0]); };
    const float diff[3] = {o[0] - t[0], o[1] - t[1], o[2] - t[2]};
    float dir[3], upn[3], xr[3], xa[3], ya[3];
    norm(diff, dir);
    if (dir[0] == up[0] && dir[1] == up[1] && dir[2] == up[2]) { CTX_FAIL(ctx, PTC_ERR_INVALID, "Look direction cannot equal up vector"); }
    norm(up, upn); crossp(upn, dir, xr); norm(xr, xa); crossp(dir, xa, ya);
    const float sign = flip ? -1.f : 1.f;
    const float m[12] = {sign * xa[0], ya[0], dir[0], o[0], sign * xa[1], ya[1], dir[1], o[1], sign * xa[2], ya[2], dir[2], o[2]};
    DScene &s = ctx->scene.view; // the camera may be re-aimed after commit
    memcpy(s.camToWorld, m, sizeof(m));
    s.vfov = vfov; s.width = w; s.height = h; ctx->hasCamera = true;
    return PTC_OK;
}

// guide[g] = first i with cdf[i] >= g / G, g = 0 .. G (n - 1 when there is none)
static void buildGuide(const float *cdf, int n, int G, uint16_t *guide)
{
    int i = 0;
    for (int g = 0; g <= G; g++) {
        const float threshold = (float)g / (float)G;
        while (i < n - 1 && cdf[i] < threshold) { i++; }
        guide[g] = (uint16_t)i;
    }
}
static int guideSize(int n)
{
    if (n > 65535) { return 1; }
    int G = 1;
    while (G * 8 <= n && G < 1024) { G *= 2; }
    return G;
}

// src/distribution.cpp:6-33
static bool buildCdf(const float *values, int n, float *cdf)
{
    float sum = 0.f;
    for (int i = 0; i < n; i++) { sum += values[i]; }
    if (sum == 0.f) { for (int i = 0; i < n; i++) { cdf[i] = 0.f; } return true; }
    for (int i = 0; i < n; i++) { cdf[i] = values[i] / sum; if (i > 0) { cdf[i] += cdf[i - 1]; } }
    cdf[n - 1] = 1.f;
    return false;
}

// SURVEY 8(f) N4.  180 GB of HBM make flattening the B200-native form of Embree's two-level instancing: every placement of an
// instance scene becomes world-space boxes of the ONE wide BVH (single-level traversal, no second stack).  The leaf triangles
// keep the instance's LOCAL-space corners and the traversal moves the ray into the placement's space for the triangle test only
// (traverse.cuh: rayToPlacement -- Embree's own arithmetic, so t, u, v round as they do in the reference), and everything
// Scene::testIntersect reads after the hit -- Ng, vertex normals, uvs, the emitter triangle's corners -- stays in LOCAL space as
// well, exactly as the reference leaves it (src/scene.cpp:122-219 never transforms back).
// flat prim = one triangle of the BVH: (local vertex ids, material) | (geomID, primID inside its scene) | (instID[0], instID[1])
struct Flattened {
    std::vector<uint32_t> prims4, ids2, inst2, worldPrims4, tags;
    std::vector<float> worldPos4, placements; // placements: per flattened placement, world-to-local rows of the outer, then of the inner level
};
static const float identity3x4[12] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0};
// Adds the triangles of `scene` placed by T; returns an error message, or null
static const char *flatten(const Staging &st, Flattened &f, uint32_t scene, const float *T, uint32_t inst0, uint32_t inst1, int level,
                           const float *outerW2L, const float *innerW2L)
{
    uint32_t tag = 0; // what the leaf triangles of this placement carry (0: root-scene geometry, tested in world space)
    if (level > 0) {
        f.placements.insert(f.placements.end(), outerW2L, outerW2L + 12);
        f.placements.insert(f.placements.end(), innerW2L ? innerW2L : identity3x4, (innerW2L ? innerW2L : identity3x4) + 12);
        tag = (uint32_t)(f.placements.size() / 24) | (level == 2 ? 0x80000000u : 0u);
    }
    for (uint32_t index : st.scenes[scene].members) {
        const HostGeometry &g = st.geometries[index];
        if (g.isSphere) { continue; }
        if (g.isInstance) {
            if (level >= 2) { return "more than RTC_MAX_INSTANCE_LEVEL_COUNT = 2 instance levels"; }
            float C[12]; // T o g.l2w: the inner placement is applied first
            for (int r = 0; r < 3; r++) {
                for (int c = 0; c < 4; c++) {
                    C[4 * r + c] = T[4 * r] * g.l2w[c] + T[4 * r + 1] * g.l2w[4 + c] + T[4 * r + 2] * g.l2w[8 + c] + (c == 3 ? T[4 * r + 3] : 0.f);
                }
            }
            const char *error = flatten(st, f, g.instanceScene, C, level == 0 ? g.localId : inst0, level == 0 ? PTC_INVALID_ID : g.localId, level + 1,
                                        level == 0 ? g.w2l : outerW2L, level == 0 ? nullptr : g.w2l);
            if (error) { return error; }
            continue;
        }
        const uint32_t base = (uint32_t)(f.worldPos4.size() / 4);
        for (uint32_t v = 0; v < g.nVertices; v++) {
            const float *q = &st.positions4[4 * (size_t)(g.firstVertex + v)];
            f.worldPos4.insert(f.worldPos4.end(), {T[0] * q[0] + T[1] * q[1] + T[2] * q[2] + T[3], T[4] * q[0] + T[5] * q[1] + T[6] * q[2] + T[7],
                                                   T[8] * q[0] + T[9] * q[1] + T[10] * q[2] + T[11], 0.f});
        }
        for (uint32_t t = 0; t < g.nPrims; t++) {
            const uint32_t *ix = &st.prims4[4 * (size_t)(g.firstPrim + t)];
            f.prims4.insert(f.prims4.end(), ix, ix + 4);
            f.worldPrims4.insert(f.worldPrims4.end(), {ix[0] - g.firstVertex + base, ix[1] - g.firstVertex + base, ix[2] - g.firstVertex + base, ix[3]});
            f.ids2.insert(f.ids2.end(), {g.localId, t});
            f.inst2.insert(f.inst2.end(), {inst0, inst1});
            f.tags.push_back(tag);
        }
    }
    return nullptr;
}

// rtcCommitScene: BVH over all triangle geometries; spheres are kept in a flat list.  The geometry goes to the device first:
// the default builder runs there (option "bvh_builder" = 0 selects the host binned-SAH builder instead).  An instanced scene is
// built over world-space copies of its triangles (`buildInputs`) whose leaves are then moved back to local space.
static int buildBvh(ptc_ctx *ctx, const Flattened *flat, const std::vector<uint32_t> &prims4, Committed &c, std::vector<SceneAllocation> &buildInputs)
{
    const Staging &st = ctx->staged; DScene &s = c.view;
    const uint32_t nPrims = (uint32_t)(prims4.size() / 4);
    TRY(upload(ctx, c, (const float4 *)st.positions4.data(), st.positions4.size() / 4, s.positions));
    TRY(upload(ctx, c, (const uint4 *)prims4.data(), prims4.size() / 4, s.prims));
    const float4 *buildPositions = s.positions; const uint4 *buildPrims = s.prims; // what the BVH is built over: world-space triangles
    if (flat) {
        TRY(upload(ctx, buildInputs, (const float4 *)flat->worldPos4.data(), flat->worldPos4.size() / 4, &buildPositions));
        TRY(upload(ctx, buildInputs, (const uint4 *)flat->worldPrims4.data(), flat->worldPrims4.size() / 4, &buildPrims));
        TRY(upload(ctx, c, (const uint2 *)flat->inst2.data(), flat->inst2.size() / 2, s.instIds));
    }
    const auto buildStart = std::chrono::steady_clock::now();
    try {
        if (ctx->options.bvhBuilder == 1) {
            DeviceWideBVH built; void *workspace = nullptr;
            buildWideBVHDevice(buildPositions, buildPrims, nPrims, ctx->stream, built, &workspace);
            c.buildWorkspace = Buffer<uint8_t>((uint8_t *)workspace, 0); // the builder does not report its size
            s.bvh.nodes = built.nodes; s.bvh.triangles = built.triangles; s.bvh.nNodes = built.nNodes;
            if (built.nodes) { c.allocations.push_back({Buffer<uint8_t>((uint8_t *)built.nodes, (size_t)built.nNodes * sizeof(WideNode)), fieldOf(s, &s.bvh.nodes), {}}); }
            if (built.triangles) { c.allocations.push_back({Buffer<uint8_t>((uint8_t *)built.triangles, (size_t)built.nTriangles * sizeof(LeafTriangle)), fieldOf(s, &s.bvh.triangles), {}}); }
            c.bvhTriangles = built.nTriangles; c.bvhDepth = built.maxDepth; c.bvhPlocIterations = built.plocIterations;
        } else {
            WideBVH bvh;
            buildWideBVH((flat ? flat->worldPos4 : st.positions4).data(), (flat ? flat->worldPrims4 : st.prims4).data(), nPrims, bvh);
            TRY(upload(ctx, c, (const float4 *)bvh.nodes.data(), bvh.nodes.size() * 5, s.bvh.nodes));
            TRY(upload(ctx, c, (const float4 *)bvh.triangles.data(), bvh.triangles.size() * 3, s.bvh.triangles));
            s.bvh.nNodes = (uint32_t)bvh.nodes.size(); c.bvhTriangles = (uint32_t)bvh.triangles.size(); c.bvhDepth = bvh.maxDepth;
        }
    } catch (const std::exception &e) { CTX_FAIL(ctx, PTC_ERR_INVALID, "BVH build failed: %s", e.what()); }
    if (flat) { c.placements = flat->placements; }
    if (!c.placements.empty() && c.bvhTriangles) {
        const uint32_t *tags = nullptr;
        TRY(upload(ctx, buildInputs, flat->tags.data(), flat->tags.size(), &tags));
        TRY(upload(ctx, c, (const float4 *)c.placements.data(), c.placements.size() / 4, s.bvh.placements));
        localizeLeavesKernel<<<(c.bvhTriangles + 255) / 256, 256, 0, ctx->stream>>>((LeafTriangle *)s.bvh.triangles, c.bvhTriangles, s.positions, s.prims, tags);
        CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    }
    c.bvhBuildMs = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - buildStart).count();
    return PTC_OK;
}

// packed texels per image, in consecutive allocations
static int uploadTextures(ptc_ctx *ctx, Committed &c)
{
    const uint32_t *texels;
    for (const Staging::HostTexture &t : ctx->staged.textures) { TRY(upload(ctx, c.allocations, t.texels.data(), t.texels.size(), &texels)); }
    return PTC_OK;
}

// the device material table (uploaded by uploadSurfaces) and the material classes present; texture t is c.allocations[firstTexture + t]
static void materialTable(const Staging &st, size_t firstTexture, Committed &c)
{
    c.materials.resize(st.materials.size());
    for (size_t i = 0; i < c.materials.size(); i++) {
        const ptc_material_desc &d = st.materials[i];
        DMaterial &m = c.materials[i]; // zeroed by resize
        c.classMask |= 1u << d.type;
        m.type = d.type; m.distribution = d.distribution; m.albedoKind = d.albedo_kind;
        m.emitter = !(d.emit[0] == 0.f && d.emit[1] == 0.f && d.emit[2] == 0.f);
        for (int k = 0; k < 3; k++) { m.diffuse[k] = d.diffuse[k]; m.emit[k] = d.emit[k]; m.on[k] = d.checker_on[k]; m.off[k] = d.checker_off[k]; }
        const float sigma2 = d.sigma * d.sigma; // OrenNayar::OrenNayar, src/oren_nayar.cpp:11-19
        m.sigmaA = 1.f - (sigma2 / (2.f * (sigma2 + 0.33f)));
        m.sigmaB = (0.45f * sigma2) / (sigma2 + 0.09f);
        m.ior = d.ior; m.alpha = d.alpha; m.resU = d.checker_resolution[0]; m.resV = d.checker_resolution[1];
        if (d.albedo_kind == PTC_ALBEDO_TEXTURE) {
            SceneAllocation &texels = c.allocations[firstTexture + d.texture];
            m.texW = st.textures[d.texture].width; m.texH = st.textures[d.texture].height; m.texels = (const uint32_t *)texels.data.get();
            texels.materials.push_back((uint32_t)i);
        }
    }
}

// the per-surface tables: lights and spheres, vertex attributes, triangle records, ids, the material table and class bytes
static int uploadSurfaces(ptc_ctx *ctx, const std::vector<uint32_t> &prims4, const std::vector<uint32_t> &primIds2, Committed &c)
{
    const Staging &st = ctx->staged; DScene &s = c.view;
    const std::vector<DMaterial> &dm = c.materials;
    // light table: emissive surfaces in registration order, environment light last (src/scene_parser.cpp:173-190); the sphere list
    std::vector<DLight> lights;
    std::vector<float> spheres4; std::vector<uint32_t> sphereIds2;
    for (uint32_t member : st.scenes[0].members) { // only root-scene surfaces become lights (src/scene_parser.cpp:173-182)
        const HostGeometry &ge = st.geometries[member];
        if (ge.isInstance) { continue; }
        if (ge.isSphere) {
            spheres4.insert(spheres4.end(), ge.centerRadius, ge.centerRadius + 4);
            sphereIds2.insert(sphereIds2.end(), {ge.localId, ge.sphereMaterial});
            if (dm[ge.sphereMaterial].emitter) {
                DLight l; memset(&l, 0, sizeof(l)); l.kind = 1;
                memcpy(l.centerRadius, ge.centerRadius, sizeof(l.centerRadius));
                for (int c = 0; c < 3; c++) { l.emit[c] = dm[ge.sphereMaterial].emit[c]; }
                lights.push_back(l);
            }
            continue;
        }
        for (uint32_t p = ge.firstPrim; p < ge.firstPrim + ge.nPrims; p++) {
            const uint32_t *ix = &st.prims4[4 * (size_t)p];
            if (!dm[ix[3]].emitter) { continue; }
            DLight l; memset(&l, 0, sizeof(l)); l.kind = 0;
            for (int c = 0; c < 3; c++) {
                l.p0[c] = st.positions4[4 * (size_t)ix[0] + c]; l.p1[c] = st.positions4[4 * (size_t)ix[1] + c]; l.p2[c] = st.positions4[4 * (size_t)ix[2] + c];
                l.emit[c] = dm[ix[3]].emit[c];
            }
            lights.push_back(l);
        }
    }
    if (st.hasEnv) { DLight l; memset(&l, 0, sizeof(l)); l.kind = 2; lights.push_back(l); }
    TRY(upload(ctx, c, (const float4 *)spheres4.data(), spheres4.size() / 4, s.bvh.spheres));
    s.bvh.nSpheres = (uint32_t)(spheres4.size() / 4);
    TRY(upload(ctx, c, (const float4 *)st.normals4.data(), st.normals4.size() / 4, s.normals));
    TRY(upload(ctx, c, (const float2 *)st.uvs2.data(), st.uvs2.size() / 2, s.uvs));
    const uint32_t nPrims = (uint32_t)(prims4.size() / 4);
    { // per-triangle shading records (shading.cuh: DScene::triShade); Ng = e2 x e1 with the fused multiply-subtracts of triangleNg
        std::vector<float> rec((size_t)nPrims * 20, 0.f);
        for (uint32_t p = 0; p < nPrims; p++) {
            const uint32_t *ix = &prims4[4 * (size_t)p];
            const float *v0 = &st.positions4[4 * (size_t)ix[0]], *v1 = &st.positions4[4 * (size_t)ix[1]], *v2 = &st.positions4[4 * (size_t)ix[2]];
            const float e1x = v0[0] - v1[0], e1y = v0[1] - v1[1], e1z = v0[2] - v1[2];
            const float e2x = v2[0] - v0[0], e2y = v2[1] - v0[1], e2z = v2[2] - v0[2];
            float *r = &rec[(size_t)p * 20];
            r[0] = fmaf(e2y, e1z, -(e2z * e1y)); r[1] = fmaf(e2z, e1x, -(e2x * e1z)); r[2] = fmaf(e2x, e1y, -(e2y * e1x));
            memcpy(&r[3], &ix[3], sizeof(float));
            for (int k = 0; k < 3; k++) {
                const float *n = &st.normals4[4 * (size_t)ix[k]];
                const float *t = &st.uvs2[2 * (size_t)ix[k]];
                r[4 + 3 * k] = n[0]; r[5 + 3 * k] = n[1]; r[6 + 3 * k] = n[2];
                r[13 + 2 * k] = t[0]; r[14 + 2 * k] = t[1];
            }
        }
        TRY(upload(ctx, c, (const float4 *)rec.data(), rec.size() / 4, s.triShade));
    }
    TRY(upload(ctx, c, (const uint2 *)primIds2.data(), primIds2.size() / 2, s.primIds));
    TRY(upload(ctx, c, (const uint2 *)sphereIds2.data(), sphereIds2.size() / 2, s.sphereIds));
    TRY(upload(ctx, c, dm.data(), dm.size(), s.materials));
    // one byte per primitive / sphere for the logic stage: material type | emitter << 3
    std::vector<uint8_t> primClass(nPrims), sphereClass(sphereIds2.size() / 2);
    for (uint32_t p = 0; p < nPrims; p++) { const DMaterial &m = dm[prims4[4 * (size_t)p + 3]]; primClass[p] = (uint8_t)(m.type | (m.emitter ? 8 : 0)); }
    for (size_t i = 0; i < sphereClass.size(); i++) { const DMaterial &m = dm[sphereIds2[2 * i + 1]]; sphereClass[i] = (uint8_t)(m.type | (m.emitter ? 8 : 0)); }
    TRY(upload(ctx, c, primClass.data(), primClass.size(), s.primClass));
    TRY(upload(ctx, c, sphereClass.data(), sphereClass.size(), s.sphereClass));
    TRY(upload(ctx, c, lights.data(), lights.size(), s.lights));
    s.nLights = (uint32_t)lights.size();
    return PTC_OK;
}

// participating media: sigma_t / sigma_s, the internal medium of every geometry, and the occlusion filter's table (a
// Passthrough surface that encloses a medium is not a hit for testOcclusion / the volumetric queries, src/scene.cpp:42-84)
static int uploadMedia(ptc_ctx *ctx, uint32_t nPrims, Committed &c)
{
    const Staging &st = ctx->staged; DScene &s = c.view;
    s.nMedia = (int32_t)st.media.size();
    if (!s.nMedia) { return PTC_OK; }
    std::vector<float> media4;
    for (const Staging::HostMedium &m : st.media) { media4.insert(media4.end(), {m.sigmaT[0], m.sigmaT[1], m.sigmaT[2], 0.f, m.sigmaS[0], m.sigmaS[1], m.sigmaS[2], 0.f}); }
    std::vector<int32_t> geomMedium(st.geometries.size()), primEvent(nPrims, -1), sphereEvent;
    for (size_t g = 0; g < st.geometries.size(); g++) {
        const HostGeometry &ge = st.geometries[g];
        geomMedium[g] = ge.medium;
        if (ge.isSphere) {
            const bool filtered = ge.medium >= 0 && c.materials[ge.sphereMaterial].type == PTC_PASSTHROUGH;
            sphereEvent.push_back(filtered ? ge.medium : -1);
            if (filtered) { s.hasFilter = 1; }
            continue;
        }
        if (ge.medium < 0) { continue; }
        for (uint32_t p = ge.firstPrim; p < ge.firstPrim + ge.nPrims; p++) {
            if (c.materials[st.prims4[4 * (size_t)p + 3]].type == PTC_PASSTHROUGH) { primEvent[p] = ge.medium; s.hasFilter = 1; }
        }
    }
    TRY(upload(ctx, c, (const float4 *)media4.data(), media4.size() / 4, s.media));
    TRY(upload(ctx, c, geomMedium.data(), geomMedium.size(), s.geomMedium));
    TRY(upload(ctx, c, primEvent.data(), primEvent.size(), s.bvh.primEvent));
    return upload(ctx, c, sphereEvent.data(), sphereEvent.size(), s.bvh.sphereEvent);
}

// EnvironmentLight::EnvironmentLight, src/environment_light.cpp:29-53: weight = R+G+B, no sin(theta) (Q9)
static int uploadEnvironment(ptc_ctx *ctx, Committed &c)
{
    const Staging &st = ctx->staged; DScene &s = c.view;
    s.hasEnv = st.hasEnv ? 1 : 0;
    if (!st.hasEnv) { return PTC_OK; }
    const int w = st.envW, h = st.envH;
    std::vector<float> row(w), theta(h), phiCdf((size_t)w * h), thetaCdf(h);
    std::vector<uint8_t> phiEmpty(h);
    for (int t = 0; t < h; t++) {
        float thetaSum = 0.f;
        for (int p = 0; p < w; p++) {
            const float *px = &st.envRgba[4 * ((size_t)t * w + p)];
            float value = 0.f;
            value += px[0]; value += px[1]; value += px[2];
            thetaSum += value; row[p] = value;
        }
        phiEmpty[t] = buildCdf(row.data(), w, &phiCdf[(size_t)t * w]) ? 1 : 0;
        theta[t] = thetaSum;
    }
    s.envThetaEmpty = buildCdf(theta.data(), h, thetaCdf.data()) ? 1 : 0;
    s.envThetaG = guideSize(h); s.envPhiG = guideSize(w);
    std::vector<uint16_t> thetaGuide((size_t)s.envThetaG + 1), phiGuide((size_t)h * (s.envPhiG + 1));
    buildGuide(thetaCdf.data(), h, s.envThetaG, thetaGuide.data());
    for (int t = 0; t < h; t++) { buildGuide(&phiCdf[(size_t)t * w], w, s.envPhiG, &phiGuide[(size_t)t * (s.envPhiG + 1)]); }
    TRY(upload(ctx, c, thetaGuide.data(), thetaGuide.size(), s.envThetaGuide));
    TRY(upload(ctx, c, phiGuide.data(), phiGuide.size(), s.envPhiGuide));
    TRY(upload(ctx, c, (const float4 *)st.envRgba.data(), (size_t)w * h, s.envRgba));
    TRY(upload(ctx, c, thetaCdf.data(), thetaCdf.size(), s.envThetaCdf));
    TRY(upload(ctx, c, phiCdf.data(), phiCdf.size(), s.envPhiCdf));
    TRY(upload(ctx, c, phiEmpty.data(), phiEmpty.size(), s.envPhiEmpty));
    s.envW = w; s.envH = h; s.envScale = st.envScale;
    memcpy(s.envM2W, st.envM2W, sizeof(s.envM2W)); memcpy(s.envW2M, st.envW2M, sizeof(s.envW2M)); // the 3 x 4 rows
    return PTC_OK;
}

// The staged scene becomes a Committed value step by step; the context takes it, and releases the staging, only when every step
// succeeded, so a failed commit leaves no allocation behind
int ptc_commit(ptc_ctx *ctx)
{
    if (!ctx) { return PTC_ERR_INVALID; }
    if (ctx->committed) { CTX_FAIL(ctx, PTC_ERR_STATE, "scene already committed"); }
    if (!ctx->hasCamera) { CTX_FAIL(ctx, PTC_ERR_STATE, "no camera set"); }
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const Staging &st = ctx->staged;
    if (!st.sceneStack.empty()) { CTX_FAIL(ctx, PTC_ERR_STATE, "ptc_begin_instance without ptc_end_instance"); }
    const bool instanced = st.scenes.size() > 1;
    if (instanced && !st.media.empty()) { CTX_FAIL(ctx, PTC_ERR_INVALID, "instancing together with participating media is not supported"); }

    Flattened flat;
    if (const char *error = instanced ? flatten(st, flat, 0, identity3x4, PTC_INVALID_ID, PTC_INVALID_ID, 0, nullptr, nullptr) : nullptr) { CTX_FAIL(ctx, PTC_ERR_INVALID, "%s", error); }
    const std::vector<uint32_t> &prims4 = instanced ? flat.prims4 : st.prims4, &primIds2 = instanced ? flat.ids2 : st.primIds2;
    Committed c; c.view = ctx->scene.view; // the camera
    std::vector<SceneAllocation> buildInputs; // released when the commit returns
    TRY(buildBvh(ctx, instanced ? &flat : nullptr, prims4, c, buildInputs));
    const size_t firstTexture = c.allocations.size();
    TRY(uploadTextures(ctx, c));
    CUDA_TRY(ctx, uploadGammaTable());
    materialTable(st, firstTexture, c);
    TRY(uploadSurfaces(ctx, prims4, primIds2, c));
    TRY(uploadMedia(ctx, (uint32_t)(prims4.size() / 4), c));
    TRY(uploadEnvironment(ctx, c));
    ctx->scene = std::move(c);
    ctx->staged = Staging();
    ctx->committed = true;
    return PTC_OK;
}

#define NEED_COMMIT(ctx) do { if (!(ctx)) { return PTC_ERR_INVALID; } if (!(ctx)->committed) { CTX_FAIL(ctx, PTC_ERR_STATE, "scene not committed"); } } while (0)

// SURVEY 8(e): the scene is parsed, fed and its BVH built ONCE; every further GPU of the spp split gets a copy of the finished
// device data over NVLink (cudaMemcpyPeer) instead of a second feed + build.  Everything ptc_commit uploaded is position-independent
// except the pointers that lead to it, which each allocation records: they are pointed at the copies here.
int ptc_replicate(ptc_ctx *src, int device, ptc_ctx **out)
{
    if (!out) { return PTC_ERR_INVALID; }
    *out = nullptr;
    NEED_COMMIT(src);
    ptc_ctx *dst = nullptr;
    int rc = ptc_create(device, &dst);
    if (rc) { CTX_FAIL(src, rc, "cannot create a context on device %d", device); }
    static_cast<SceneState &>(dst->scene) = src->scene;
    dst->scene.bvhBuildMs = 0.f; // nothing was built here
    dst->options = src->options;
    auto fail = [&](const char *what) { src->error = std::string("ptc_replicate: ") + what + ": " + cudaGetErrorString(cudaGetLastError()); ptc_destroy(dst); return PTC_ERR_CUDA; };
    if (cudaSetDevice(device) != cudaSuccess) { return fail("cudaSetDevice"); }
    for (const SceneAllocation &a : src->scene.allocations) {
        Buffer<uint8_t> copy;
        if (copy.resize(a.data.size()) != cudaSuccess) { return fail("cudaMalloc"); }
        if (cudaMemcpyPeerAsync(copy.get(), device, a.data.get(), src->device, a.data.size(), dst->stream) != cudaSuccess) { return fail("cudaMemcpyPeerAsync"); }
        if (a.field != NO_FIELD) { *(const void **)((char *)&dst->scene.view + a.field) = copy.get(); }
        for (uint32_t m : a.materials) { dst->scene.materials[m].texels = (const uint32_t *)copy.get(); }
        dst->scene.allocations.push_back({std::move(copy), a.field, a.materials});
    }
    const std::vector<DMaterial> &dm = dst->scene.materials;
    if (!dm.empty() && cudaMemcpyAsync((void *)dst->scene.view.materials, dm.data(), dm.size() * sizeof(DMaterial), cudaMemcpyHostToDevice, dst->stream) != cudaSuccess) { return fail("material table"); }
    if (uploadGammaTable() != cudaSuccess) { return fail("gamma table"); }
    // the source's data must be complete before it is read (ptc_commit is synchronous, so it is) and the copies before `dst` is used
    if (cudaStreamSynchronize(dst->stream) != cudaSuccess) { return fail("copy"); }
    dst->committed = true;
    *out = dst;
    return PTC_OK;
}

// Path state for waves of up to `capacity` paths.  The per-path arrays depend on nothing but the capacity (ptc_reserve_paths may ask
// for them before the scene exists); the class queues follow the material classes the committed scene holds.
static int ensurePathBuffers(ptc_ctx *ctx, uint32_t capacity, bool withClassQueues = true)
{
    PathBuffers &pb = ctx->paths;
    if (capacity > ctx->pathCapacity) {
        ctx->pathCapacity = 0;
        struct { void **slot; size_t bytesPerPath; } arrays[] = {
            {(void **)&pb.out, 16}, {(void **)&pb.ray, 32}, {(void **)&pb.nRay, 32}, {(void **)&pb.modThr, 32}, {(void **)&pb.nModThr, 32}, {(void **)&pb.nee, 32},
            {(void **)&pb.hit, 16}, {(void **)&pb.result, 16}, {(void **)&pb.nResult, 16}, {(void **)&pb.occluded, 1}, {(void **)&pb.shadowQueue, 4}};
        // ONE allocation for all the arrays (one driver call instead of eleven; their relative placement no longer depends on what the
        // process allocated and freed before).  Measured: neither the gaps between the arrays (0 ... 2 MB + 9 KB) nor slab vs separate
        // allocations change the throughput (profiles/r02_path_state_layout.txt).
        size_t total = 0;
        for (auto &a : arrays) { total += ((size_t)capacity * a.bytesPerPath + 255u) & ~(size_t)255u; }
        CUDA_TRY(ctx, ctx->pathSlab.reserve(total));
        size_t offset = 0;
        for (auto &a : arrays) { *a.slot = ctx->pathSlab.get() + offset; offset += ((size_t)capacity * a.bytesPerPath + 255u) & ~(size_t)255u; }
        ctx->pathCapacity = capacity;
    }
    if (!withClassQueues) { return PTC_OK; }
    for (int t = 0; t < PTC_MATERIAL_CLASSES; t++) {
        pb.classQueue[t] = nullptr;
        if (!(ctx->scene.classMask & (1u << t))) { continue; }
        CUDA_TRY(ctx, ctx->classQueues[t].reserve(ctx->pathCapacity));
        pb.classQueue[t] = ctx->classQueues[t].get();
    }
    return PTC_OK;
}

int ptc_reserve_paths(ptc_ctx *ctx, uint64_t nPaths)
{
    if (!ctx) { return PTC_ERR_INVALID; }
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const uint64_t capacity = std::min<uint64_t>(std::max<uint64_t>(nPaths, 1), (uint64_t)ctx->options.pathsPerWave);
    return ensurePathBuffers(ctx, (uint32_t)capacity, false);
}

// Which checkpoints the resolve of one wave (global samples F .. F + S - 1 of a render call) snapshots, and after how many of the wave's
// samples: those that fall inside it, plus -- in the first / last wave of the call -- those before / after the call's samples (copies of
// the sums as they were / as they end up: the spp split gives every GPU a block of samples, and a checkpoint is the sum over all GPUs)
struct Checkpoints { const uint32_t *counts = nullptr; uint32_t n = 0; float *const *dst = nullptr; };
static CheckpointPlan planFor(const Checkpoints &cp, uint32_t F, uint32_t S, bool isFirst, bool isLast)
{
    CheckpointPlan plan; plan.n = 0;
    for (uint32_t i = 0; i < cp.n; i++) {
        const uint32_t c = cp.counts[i]; // sample count: the checkpoint holds samples 0 .. c - 1
        const bool inside = c > F && c <= F + S;
        if (!(inside || (isFirst && c <= F) || (isLast && c > F + S))) { continue; }
        plan.at[plan.n] = c <= F ? 0u : std::min(c - F, S);
        plan.dst[plan.n] = cp.dst[i];
        plan.n++;
    }
    return plan;
}

// ptc_render's upload of the caller's sums (through `staging`, page-locked, when that is another buffer) into `device`.  The first
// wave issues it on copyStream behind its other launches, so that it runs while the GPU traces the wave; only the wave's first
// accumulation waits for it.
struct SumsUpload { const float *caller; float *staging, *device; size_t n; };
static int uploadSums(ptc_ctx *ctx, const SumsUpload &u)
{
    if (u.staging != u.caller) { memcpy(u.staging, u.caller, u.n * sizeof(float)); }
    CUDA_TRY(ctx, cudaMemcpyAsync(u.device, u.staging, u.n * sizeof(float), cudaMemcpyHostToDevice, ctx->copyStream));
    CUDA_TRY(ctx, cudaEventRecord(ctx->uploadDone, ctx->copyStream));
    CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream, ctx->uploadDone, 0));
    return PTC_OK;
}

// The arrays of lane `lane`: every array of the wave's path state starts `offset` paths further on
static PathBuffers laneBuffers(const PathBuffers &all, size_t offset)
{
    PathBuffers pb = all;
    pb.ray += 2 * offset; pb.nRay += 2 * offset; pb.modThr += 2 * offset; pb.nModThr += 2 * offset; pb.nee += 2 * offset;
    pb.hit += offset; pb.result += offset; pb.nResult += offset; pb.occluded += offset; pb.out += offset; pb.shadowQueue += offset;
    for (int t = 0; t < PTC_MATERIAL_CLASSES; t++) { if (pb.classQueue[t]) { pb.classQueue[t] += offset; } }
    return pb;
}

static int ensureLanes(ptc_ctx *ctx, int lanes)
{
    CUDA_TRY(ctx, ctx->laneFork.create());
    while ((int)ctx->extraLanes.size() < lanes - 1) {
        ptc_ctx::Lane lane;
        CUDA_TRY(ctx, lane.stream.create());
        CUDA_TRY(ctx, lane.shadowStream.create());
        CUDA_TRY(ctx, lane.shadeDone.create());
        CUDA_TRY(ctx, lane.shadowDone.create());
        CUDA_TRY(ctx, lane.done.create());
        CUDA_TRY(ctx, lane.counters.resize(CNT_STRIDE));
        ctx->extraLanes.push_back(std::move(lane));
    }
    return PTC_OK;
}

static VolumeBuffers laneVolumeBuffers(const VolumeBuffers &all, size_t offset)
{
    VolumeBuffers vb = all;
    if (vb.probeHit) { vb.probeHit += offset; vb.shadowTr += offset; vb.scatter += 3 * offset; vb.scatterTr += offset; vb.extendQueue += offset; vb.scatterQueue += offset; }
    return vb;
}

// VolumePathTracer, wavefront form (volume_wavefront.cuh)
static int ensureVolumeBuffers(ptc_ctx *ctx, uint32_t capacity)
{
    VolumeBuffers &vb = ctx->volumeBuffers;
    struct { void **slot; size_t bytesPerPath; } arrays[] = {
        {(void **)&vb.probeHit, 16}, {(void **)&vb.shadowTr, 16}, {(void **)&vb.scatter, 48}, {(void **)&vb.scatterTr, 16}, {(void **)&vb.extendQueue, 4}, {(void **)&vb.scatterQueue, 4}};
    for (int i = 0; i < 6; i++) {
        CUDA_TRY(ctx, ctx->volumeArrays[i].reserve((size_t)capacity * arrays[i].bytesPerPath));
        *arrays[i].slot = ctx->volumeArrays[i].get();
    }
    return PTC_OK;
}

// A traversal stage of a wave: a traverseKernel, or a volumeTraverseKernel (it also reads the VolumePathTracer's buffers), and its grid
typedef void (*TraverseFn)(DScene, PathBuffers, const uint32_t *, const uint32_t *, uint32_t *, unsigned long long *);
typedef void (*VolumeTraverseFn)(DScene, PathBuffers, VolumeBuffers, const uint32_t *, const uint32_t *, uint32_t *, unsigned long long *);
struct Traversal {
    TraverseFn plain = nullptr; VolumeTraverseFn volume = nullptr; int grid = 0;
    void launch(cudaStream_t stream, const DScene &s, const PathBuffers &pb, const VolumeBuffers &vb, const uint32_t *queue, const uint32_t *count,
                uint32_t *cursor, unsigned long long *work) const
    {
        if (volume) { volume<<<grid, 128, 0, stream>>>(s, pb, vb, queue, count, cursor, work); }
        else { plain<<<grid, 128, 0, stream>>>(s, pb, queue, count, cursor, work); }
    }
};
// extend0: the camera rays; extend: the rays of bounces >= 1; shadow and, in participating media, scatter: the shadow rays of bounces >= 1
struct WaveTraversals { Traversal extend0, extend, shadow, scatter; };
// sharedSMs: the wave is traced as several lanes, whose persistent traversal grids leave room for the CTAs of another lane's stage
// (profiles/r02_sweep_lanes.txt)
static WaveTraversals pickTraversals(const ptc_ctx *ctx, bool volume, bool sharedSMs)
{
    const DScene &s = ctx->scene.view;
    const bool count = ctx->options.countTraversal;
    const int grid = sharedSMs ? ctx->gridTraverseShared : ctx->gridTraverse;
    const int volumeGrid = sharedSMs ? ctx->gridVolumeTraverseShared : ctx->gridVolumeTraverse;
    WaveTraversals t;
    const TraverseFn closest = count ? traverseKernel<false, true> : traverseKernel<false, false>;
    t.extend0 = {s.bvh.placements ? traverseKernel<false, false, false, true> : closest, nullptr, grid}; // instanced: never counted
    if (!volume) {
        t.extend = t.extend0;
        const TraverseFn shadow = s.bvh.placements ? traverseKernel<true, false, false, true> : s.hasFilter ? traverseKernel<true, false, true>
                                  : count ? traverseKernel<true, true> : traverseKernel<true, false>;
        t.shadow = {shadow, nullptr, grid};
        return t;
    }
    // the VolumePathTracer's bounces: probe + continuation ray in one traversal (no container surface: the two rules coincide), both
    // kinds of shadow rays next to them
    if (s.hasFilter) { t.extend = {nullptr, count ? volumeTraverseKernel<VOL_EXTEND, true> : volumeTraverseKernel<VOL_EXTEND, false>, volumeGrid}; }
    else { t.extend = {closest, nullptr, grid}; }
    t.shadow = {nullptr, count ? volumeTraverseKernel<VOL_SHADOW, true> : volumeTraverseKernel<VOL_SHADOW, false>, volumeGrid};
    if (s.nMedia) { t.scatter = {nullptr, count ? volumeTraverseKernel<VOL_SCATTER, true> : volumeTraverseKernel<VOL_SCATTER, false>, volumeGrid}; }
    return t;
}

// The material stage's kernels by class; [LISTED]: the wave's pixels are listed (WaveParams::pixels)
typedef void (*MaterialFn)(DScene, PathBuffers, WaveParams, BounceCounters *, BounceCounters *);
static const MaterialFn materialKernels[2][PTC_MATERIAL_CLASSES] = {
    {materialKernel<PTC_LAMBERTIAN, false>, materialKernel<PTC_OREN_NAYAR, false>, materialKernel<PTC_MIRROR, false>, materialKernel<PTC_GLASS, false>,
     materialKernel<PTC_MICROFACET, false>, materialKernel<PTC_PLASTIC, false>, materialKernel<PTC_PASSTHROUGH, false>},
    {materialKernel<PTC_LAMBERTIAN, true>, materialKernel<PTC_OREN_NAYAR, true>, materialKernel<PTC_MIRROR, true>, materialKernel<PTC_GLASS, true>,
     materialKernel<PTC_MICROFACET, true>, materialKernel<PTC_PLASTIC, true>, materialKernel<PTC_PASSTHROUGH, true>}};
typedef void (*VolumeMaterialFn)(DScene, PathBuffers, VolumeBuffers, WaveParams, BounceCounters *, BounceCounters *);
static const VolumeMaterialFn volumeMaterialKernels[PTC_MATERIAL_CLASSES] = {
    volumeMaterialKernel<PTC_LAMBERTIAN>, volumeMaterialKernel<PTC_OREN_NAYAR>, volumeMaterialKernel<PTC_MIRROR>, volumeMaterialKernel<PTC_GLASS>,
    volumeMaterialKernel<PTC_MICROFACET>, volumeMaterialKernel<PTC_PLASTIC>, volumeMaterialKernel<PTC_PASSTHROUGH>};

// radianceLookup += the samples of one (part-)wave, in sample order; with `moments` also their squares
static void launchAccumulate(ptc_ctx *ctx, cudaStream_t stream, const PathBuffers &pb, const WaveParams &wp, float *accumDevice, float *moments,
                             const CheckpointPlan &plan)
{
    const auto kernel = moments ? accumulateKernel<true> : accumulateKernel<false>;
    kernel<<<gridFor(ctx, wp.nPixels, 256), 256, 0, stream>>>(pb, wp, accumDevice, moments, (uint32_t)ctx->scene.view.width, (uint32_t)ctx->scene.view.height, plan);
    ctx->launches++;
}

// One wave = fixed launch sequence; all queue sizes stay on the device.  The wave's samples are traced as nLanes part-waves (wps[i]:
// consecutive sample blocks, plans[i]: the checkpoints that fall into them) whose launch sequences are issued bounce by bounce on one
// stream per lane, so that the stages of different lanes share the SMs (ptc_ctx::lanes); nLanes = 1 is the plain sequence.
// volume: the VolumePathTracer's stages (volume_wavefront.cuh) -- merged probe / continuation rays, two kinds of shadow rays, its own
// logic and material kernels; bounce 0 is the PathTracer's.  upload: issued behind the wave's other launches (uploadSums).
static int launchWave(ptc_ctx *ctx, const WaveParams *wps, const CheckpointPlan *plans, int nLanes, float *accumDevice, float *moments, cudaStream_t callerStream,
                      bool volume, const SumsUpload *upload)
{
    const DScene &s = ctx->scene.view;
    struct LaneState { PathBuffers pb; VolumeBuffers vb; BounceCounters *cnt; cudaStream_t stream, shadowStream; cudaEvent_t shadeDone, shadowDone; };
    LaneState lanes[PTC_MAX_LANES];
    if (nLanes > 1) {
        const int rc = ensureLanes(ctx, nLanes);
        if (rc) { return rc; }
        CUDA_TRY(ctx, cudaEventRecord(ctx->laneFork, callerStream)); // the other lanes start behind whatever the caller's stream holds so far
    }
    const WaveTraversals traversals = pickTraversals(ctx, volume, nLanes > 1);
    size_t offset = 0;
    for (int i = 0; i < nLanes; i++) {
        LaneState &l = lanes[i];
        l.pb = laneBuffers(ctx->paths, offset); // by value: the current / next buffers swap after every bounce
        l.vb = laneVolumeBuffers(ctx->volumeBuffers, offset);
        offset += (size_t)wps[i].nPixels * wps[i].sppWave;
        if (i == 0) { l.cnt = ctx->counters.get(); l.stream = callerStream; l.shadowStream = ctx->shadowStream; l.shadeDone = ctx->shadeDone; l.shadowDone = ctx->shadowDone; }
        else {
            const ptc_ctx::Lane &x = ctx->extraLanes[(size_t)i - 1];
            l.cnt = x.counters.get(); l.stream = x.stream; l.shadowStream = x.shadowStream; l.shadeDone = x.shadeDone; l.shadowDone = x.shadowDone;
            CUDA_TRY(ctx, cudaStreamWaitEvent(l.stream, ctx->laneFork, 0));
        }
        CUDA_TRY(ctx, cudaMemsetAsync(l.cnt, 0, CNT_STRIDE * sizeof(BounceCounters), l.stream));
        const uint32_t nPaths = wps[i].nPixels * wps[i].sppWave;
        {
            StageTimer t(ctx, l.stream, STAGE_OTHER);
            generateKernel<<<gridFor(ctx, nPaths, 256), 256, 0, l.stream>>>(s, l.pb, wps[i], l.cnt);
        }
        ctx->launches++;
    }
    unsigned long long *work = ctx->totals.get() + 2;
    const int lastBounce = wps[0].lastBounce;
    // ray k leaves vertex k (k = 0: camera ray).  Ray k feeds direct() of vertex k and creates vertex k + 1, so rays
    // 0 .. lastBounce are traced; shadow rays cast at vertex k are traced alongside ray k.
    for (int k = 0; k <= lastBounce; k++) {
        for (int i = 0; i < nLanes; i++) {
            LaneState &l = lanes[i];
            const WaveParams &wp = wps[i];
            PathBuffers &pb = l.pb;
            const VolumeBuffers &vb = l.vb;
            cudaStream_t stream = l.stream;
            BounceCounters *bc = l.cnt + k;
            // shadow rays cast at vertex k (queued by material(k - 1)) go to the second stream, behind everything enqueued so far
            const bool overlap = ctx->options.overlapShadow && k > 0;
            cudaStream_t shadowOn = overlap ? l.shadowStream : stream;
            if (overlap) {
                CUDA_TRY(ctx, cudaEventRecord(l.shadeDone, stream));
                CUDA_TRY(ctx, cudaStreamWaitEvent(l.shadowStream, l.shadeDone, 0));
            }
            {
                // the rays of bounce k are the current buffers' slots 0 .. extendCount - 1: no queue (camera rays of either integrator:
                // Scene::testIntersect), except the VolumePathTracer's bounces
                StageTimer t(ctx, stream, STAGE_EXTEND);
                (k > 0 ? traversals.extend : traversals.extend0).launch(stream, s, pb, vb, volume && k > 0 ? vb.extendQueue : nullptr, &bc->extendCount, &bc->extendCursor, work);
            }
            ctx->launches++;
            if (k > 0) {
                StageTimer t(ctx, shadowOn, STAGE_SHADOW);
                traversals.shadow.launch(shadowOn, s, pb, vb, pb.shadowQueue, &bc->shadowCount, &bc->shadowCursor, work + 2);
                ctx->launches++;
                if (traversals.scatter.volume) {
                    traversals.scatter.launch(shadowOn, s, pb, vb, vb.scatterQueue, &bc->scatterCount, &bc->scatterCursor, work + 2);
                    ctx->launches++;
                }
            }
            if (overlap) { // the logic stage reads the occlusion bytes / shadow outcomes
                CUDA_TRY(ctx, cudaEventRecord(l.shadowDone, l.shadowStream));
                CUDA_TRY(ctx, cudaStreamWaitEvent(stream, l.shadowDone, 0));
            }
            {
                StageTimer t(ctx, stream, STAGE_SHADE);
                if (volume && k > 0) { volumeLogicKernel<<<ctx->gridVolumeLogic, 256, 0, stream>>>(s, pb, vb, wp, bc, ctx->scene.classMask); }
                else { // k = 0 of the VolumePathTracer: SampleIntegrator::samplePixel's own terms, as in the PathTracer wavefront
                    logicKernel<<<ctx->gridLogic, 256, 0, stream>>>(s, pb, wp, bc, ctx->scene.classMask, k);
                    if (k == 0 && s.hasFilter) { containerKernel<<<ctx->gridShade, 128, 0, stream>>>(s, pb, wp, bc); ctx->launches++; }
                }
                ctx->launches++;
                for (int c = 0; c < PTC_MATERIAL_CLASSES; c++) {
                    if (!(ctx->scene.classMask & (1u << c))) { continue; }
                    if (volume) { volumeMaterialKernels[c]<<<ctx->gridVolumeShade, 128, 0, stream>>>(s, pb, vb, wp, bc, bc + 1); }
                    else { materialKernels[wp.pixels != nullptr][c]<<<ctx->gridShade, 128, 0, stream>>>(s, pb, wp, bc, bc + 1); }
                    ctx->launches++;
                }
            }
            // the material stage moved every surviving path to its slot of bounce k + 1 in the `next` buffers
            std::swap(pb.ray, pb.nRay); std::swap(pb.modThr, pb.nModThr); std::swap(pb.result, pb.nResult);
        }
    }
    if (upload) { const int rc = uploadSums(ctx, *upload); if (rc) { return rc; } }
    // radianceLookup += in sample order: the lanes' samples are added one lane after the other on the caller's stream
    for (int i = 0; i < nLanes; i++) {
        if (i > 0) {
            const ptc_ctx::Lane &x = ctx->extraLanes[(size_t)i - 1];
            CUDA_TRY(ctx, cudaEventRecord(x.done, x.stream));
            CUDA_TRY(ctx, cudaStreamWaitEvent(callerStream, x.done, 0));
        }
        StageTimer t(ctx, callerStream, STAGE_OTHER);
        launchAccumulate(ctx, callerStream, lanes[i].pb, wps[i], accumDevice, moments, plans[i]);
        tallyKernel<<<1, 32, 0, callerStream>>>(lanes[i].cnt, ctx->totals.get());
        ctx->launches++;
    }
    if (ctx->pending.size() > 4096) { collectTimings(ctx); }
    CUDA_TRY(ctx, cudaGetLastError());
    return PTC_OK;
}

// The pixels of an adaptive pass (ptc_adaptive_pass): `count` pixels, listed on the device (null list: the whole image in slotToPixel's
// order), whose accumulation also adds the squared samples into `moments`.  moments = null: a plain render of every pixel.
struct PassPixels { const uint32_t *list = nullptr; uint32_t count = 0; float *moments = nullptr; };

// One wave of the VolumePathTracer as one thread per path: a volumePathKernel launch over pixels x sppWave paths, then the same
// in-order accumulation
static int volumeWave(ptc_ctx *ctx, const WaveParams &wp, const CheckpointPlan &plan, float *accumDevice, float *moments, cudaStream_t stream, const SumsUpload *upload)
{
    PathBuffers pb = ctx->paths;
    pb.out = ctx->volumeOut.get();
    uint32_t *cursor = ctx->volumeCursor.get();
    CUDA_TRY(ctx, cudaMemsetAsync(cursor, 0, sizeof(uint32_t), stream));
    {
        StageTimer t(ctx, stream, STAGE_SHADE);
        const auto kernel = ctx->options.countTraversal ? volumePathKernel<true> : volumePathKernel<false>;
        kernel<<<ctx->gridVolume, 128, 0, stream>>>(ctx->scene.view, pb.out, wp, cursor, ctx->totals.get());
        ctx->launches++;
    }
    if (upload) { const int rc = uploadSums(ctx, *upload); if (rc) { return rc; } }
    {
        StageTimer t(ctx, stream, STAGE_OTHER);
        launchAccumulate(ctx, stream, pb, wp, accumDevice, moments, plan);
    }
    CUDA_TRY(ctx, cudaGetLastError());
    return PTC_OK;
}

static int renderInternal(ptc_ctx *ctx, uint64_t seed, uint32_t firstSample, uint32_t nSpp, int start, int last, float *accumDevice, cudaStream_t stream,
                          const Checkpoints &checkpoints = Checkpoints(), const PassPixels &pass = PassPixels(), const SumsUpload *upload = nullptr)
{
    if (start < 0 || (last != -1 && start > last)) { CTX_FAIL(ctx, PTC_ERR_INVALID, "bad bounce window [%d, %d]", start, last); }
    if (last == -1 || last > PTC_MAX_BOUNCES) { last = PTC_MAX_BOUNCES; }
    const uint32_t nPixels = pass.moments ? pass.count : (uint32_t)ctx->scene.view.width * (uint32_t)ctx->scene.view.height;
    uint32_t sppWave = (uint32_t)std::max<int64_t>(1, ctx->options.pathsPerWave / (int64_t)nPixels);
    sppWave = std::min(sppWave, std::max(nSpp, 1u));
    const bool volume = ctx->options.integrator == PTC_INTEGRATOR_VOLUME_PATH_TRACER;
    // the one-thread-per-path kernel stays for instanced scenes (the volume traversal kernels test world-space leaves only) and as an option
    const bool megakernel = volume && (ctx->options.volumeMegakernel || ctx->scene.view.bvh.placements);
    if (megakernel) {
        CUDA_TRY(ctx, ctx->volumeOut.reserve((size_t)nPixels * sppWave));
        CUDA_TRY(ctx, ctx->volumeCursor.resize(1));
    } else {
        int rc = ensurePathBuffers(ctx, nPixels * sppWave);
        if (rc) { return rc; }
        if (volume && (rc = ensureVolumeBuffers(ctx, nPixels * sppWave))) { return rc; }
    }
    for (uint32_t done = 0; done < nSpp; done += sppWave) {
        WaveParams wp;
        wp.seed = seed; wp.firstSample = firstSample + done; wp.sppWave = std::min(sppWave, nSpp - done); wp.nPixels = nPixels; wp.groupShift = groupShiftFor(wp.sppWave);
        wp.startBounce = start; wp.lastBounce = last; wp.pixels = pass.list;
        // lanes: consecutive blocks of the wave's samples.  Two lanes, four when the wave is small (measured on five scenes,
        // profiles/r02_sweep_lanes.txt); one for the megakernel, and while a stage or traversal counter pass describes one launch
        // sequence at a time
        int nLanes = ctx->options.lanes > 0 ? ctx->options.lanes : ((uint64_t)nPixels * wp.sppWave <= (1u << 25) ? 4 : 2);
        if (megakernel || ctx->options.stageTiming || ctx->options.countTraversal) { nLanes = 1; }
        nLanes = (int)std::min<uint32_t>((uint32_t)nLanes, wp.sppWave);
        WaveParams wps[PTC_MAX_LANES]; CheckpointPlan plans[PTC_MAX_LANES];
        const uint32_t perLane = (wp.sppWave + (uint32_t)nLanes - 1) / (uint32_t)nLanes;
        int used = 0;
        for (uint32_t at = 0; at < wp.sppWave; at += perLane, used++) {
            WaveParams &w = wps[used]; w = wp;
            w.firstSample = wp.firstSample + at; w.sppWave = std::min(perLane, wp.sppWave - at); w.groupShift = groupShiftFor(w.sppWave);
            plans[used] = planFor(checkpoints, w.firstSample, w.sppWave, done == 0 && at == 0, done + sppWave >= nSpp && at + perLane >= wp.sppWave);
        }
        const SumsUpload *waveUpload = done == 0 ? upload : nullptr;
        const int rc = megakernel ? volumeWave(ctx, wps[0], plans[0], accumDevice, pass.moments, stream, waveUpload)
                                  : launchWave(ctx, wps, plans, used, accumDevice, pass.moments, stream, volume, waveUpload);
        if (rc) { return rc; }
    }
    if (ctx->pending.size() > 4096) { collectTimings(ctx); } // launchWave also collects after every wave
    ctx->samples += (uint64_t)nPixels * nSpp;
    return PTC_OK;
}

int ptc_render_device(ptc_ctx *ctx, uint64_t seed, uint32_t firstSample, uint32_t nSpp, int start, int last, float *accumDevice, void *stream)
{
    NEED_COMMIT(ctx);
    if (!accumDevice) { CTX_FAIL(ctx, PTC_ERR_INVALID, "null accumulation buffer"); }
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    return renderInternal(ctx, seed, firstSample, nSpp, start, last, accumDevice, (cudaStream_t)stream);
}

int ptc_render(ptc_ctx *ctx, uint64_t seed, uint32_t firstSample, uint32_t nSpp, int start, int last, float *accum)
{
    NEED_COMMIT(ctx);
    if (!accum) { CTX_FAIL(ctx, PTC_ERR_INVALID, "null accumulation buffer"); }
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const size_t n = (size_t)3 * ctx->scene.view.width * ctx->scene.view.height;
    CUDA_TRY(ctx, ctx->accumScratch.reserve(n));
    CUDA_TRY(ctx, ctx->pinned.reserve(n));
    float *accumDevice = ctx->accumScratch.get();
    // A radianceLookup in page-locked memory (cudaHostAlloc / cudaHostRegister by the caller) is copied from and to directly; a pageable
    // one goes through the context's pinned staging buffer (two host copies of the framebuffer more per call).
    cudaPointerAttributes attr;
    const bool callerPinned = cudaPointerGetAttributes(&attr, accum) == cudaSuccess && attr.type == cudaMemoryTypeHost;
    cudaGetLastError(); // older drivers report unregistered host memory as an error
    float *hostSide = callerPinned ? accum : ctx->pinned.get();
    // radianceLookup is accumulated, not overwritten (src/sample_integrator.cpp:61-63): upload, add, download.  The sums are first
    // needed by the accumulation at the end of the first wave, so the host copy into pinned memory and the upload are issued on a second
    // stream AFTER the wave's other launches (they are asynchronous) and run while the GPU traces the wave.
    CUDA_TRY(ctx, cudaEventRecord(ctx->evStart, ctx->stream));
    const SumsUpload upload = {accum, hostSide, accumDevice, n};
    int rc = renderInternal(ctx, seed, firstSample, nSpp, start, last, accumDevice, ctx->stream, Checkpoints(), PassPixels(), &upload);
    if (!rc && nSpp == 0) { rc = uploadSums(ctx, upload); } // no wave at all: the sums pass through
    if (rc) { return rc; }
    CUDA_TRY(ctx, cudaMemcpyAsync(hostSide, accumDevice, n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaEventRecord(ctx->evStop, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    cudaEventElapsedTime(&ctx->lastRenderMs, ctx->evStart, ctx->evStop);
    if (hostSide != accum) { memcpy(accum, hostSide, n * sizeof(float)); }
    return PTC_OK;
}

// The framebuffer at the camera's resolution; a new one starts at zero
static int ensureFramebuffer(ptc_ctx *ctx)
{
    const size_t n = (size_t)3 * ctx->scene.view.width * ctx->scene.view.height;
    if (ctx->framebuffer.size() == n) { return PTC_OK; }
    CUDA_TRY(ctx, ctx->framebuffer.resize(n));
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->framebuffer.get(), 0, n * sizeof(float), ctx->stream));
    CUDA_TRY(ctx, ctx->framebufferReady.create());
    return PTC_OK;
}

int ptc_framebuffer_clear(ptc_ctx *ctx)
{
    NEED_COMMIT(ctx);
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const int rc = ensureFramebuffer(ctx);
    if (rc) { return rc; }
    const size_t n = ctx->framebuffer.size();
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->framebuffer.get(), 0, n * sizeof(float), ctx->stream));
    // with the option on the moments exist from here, so that a context that gets no samples still has (zero) moments to gather
    if (ctx->options.framebufferMoments) {
        CUDA_TRY(ctx, ctx->moments.resize(n));
        CUDA_TRY(ctx, cudaMemsetAsync(ctx->moments.get(), 0, n * sizeof(float), ctx->stream));
    }
    ctx->momentsComplete = ctx->options.framebufferMoments;
    ctx->adaptive.on = false;
    return PTC_OK;
}

int ptc_framebuffer_render(ptc_ctx *ctx, uint64_t seed, uint32_t firstSample, uint32_t nSpp, int start, int last)
{
    return ptc_framebuffer_render_checkpoints(ctx, seed, firstSample, nSpp, start, last, nullptr, 0);
}

int ptc_framebuffer_render_checkpoints(ptc_ctx *ctx, uint64_t seed, uint32_t firstSample, uint32_t nSpp, int start, int last, const uint32_t *sampleCounts, uint32_t nCounts)
{
    NEED_COMMIT(ctx);
    if (nCounts > PTC_MAX_CHECKPOINTS || (nCounts && !sampleCounts)) { CTX_FAIL(ctx, PTC_ERR_INVALID, "bad checkpoint list (at most %d)", PTC_MAX_CHECKPOINTS); }
    for (uint32_t i = 1; i < nCounts; i++) { if (sampleCounts[i] <= sampleCounts[i - 1]) { CTX_FAIL(ctx, PTC_ERR_INVALID, "checkpoint sample counts must ascend"); } }
    if (ctx->adaptive.on) { CTX_FAIL(ctx, PTC_ERR_STATE, "the framebuffer holds an adaptive render: ptc_framebuffer_clear first"); }
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    int rc = ensureFramebuffer(ctx);
    if (rc) { return rc; }
    const size_t n = ctx->framebuffer.size();
    const bool withMoments = ctx->options.framebufferMoments;
    // the moments need room behind the sums, and a new resolution new buffers
    if (nCounts && ((withMoments && !ctx->snapshotsHoldMoments) || ctx->snapshotSize != n)) {
        CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream)); // gathers that read the old snapshots are ordered before this stream's work
        ctx->snapshots.clear(); ctx->snapshotsHoldMoments = withMoments; ctx->snapshotSize = n;
    }
    while (ctx->snapshots.size() < nCounts) {
        Buffer<float> buffer;
        CUDA_TRY(ctx, buffer.resize((ctx->snapshotsHoldMoments ? 2 : 1) * n));
        ctx->snapshots.push_back(std::move(buffer));
    }
    if (!withMoments) { ctx->momentsComplete = false; }
    else if (ctx->moments.size() != n) { // a new buffer starts at zero, like a new framebuffer
        CUDA_TRY(ctx, ctx->moments.resize(n));
        CUDA_TRY(ctx, cudaMemsetAsync(ctx->moments.get(), 0, n * sizeof(float), ctx->stream));
    }
    ctx->snapshotMomentsComplete.assign(ctx->snapshots.size(), false);
    float *dst[PTC_MAX_CHECKPOINTS];
    for (uint32_t i = 0; i < nCounts; i++) { ctx->snapshotMomentsComplete[i] = withMoments && ctx->momentsComplete; dst[i] = ctx->snapshots[i].get(); }
    if (nSpp == 0) { // no samples for this context in the wave: every snapshot is the framebuffer (and its moments) as it stands
        for (uint32_t i = 0; i < nCounts; i++) {
            CUDA_TRY(ctx, cudaMemcpyAsync(dst[i], ctx->framebuffer.get(), n * sizeof(float), cudaMemcpyDeviceToDevice, ctx->stream));
            if (withMoments) { CUDA_TRY(ctx, cudaMemcpyAsync(dst[i] + n, ctx->moments.get(), n * sizeof(float), cudaMemcpyDeviceToDevice, ctx->stream)); }
        }
        return PTC_OK;
    }
    Checkpoints cp; cp.counts = sampleCounts; cp.n = nCounts; cp.dst = dst;
    PassPixels pass; // every pixel, no list; with the moments option the accumulation also adds the squared samples (the sums are the same)
    if (withMoments) { pass.count = (uint32_t)(n / 3); pass.moments = ctx->moments.get(); }
    return renderInternal(ctx, seed, firstSample, nSpp, start, last, ctx->framebuffer.get(), ctx->stream, cp, pass);
}

} // extern "C"

// What a gather reads on context c for a framebuffer of n floats: the sums of checkpoint snapshot i, or of the framebuffer when i < 0,
// or with `moments` the second moments that cover every sample those sums hold; null when there are none
static const float *gatherInput(const ptc_ctx *c, int i, size_t n, bool moments)
{
    if (i < 0 && !moments) { return c->framebuffer.get(); }
    if (i < 0) { return c->momentsComplete && c->moments.size() == n ? c->moments.get() : nullptr; }
    if ((size_t)i >= c->snapshots.size() || c->snapshotSize != n) { return nullptr; }
    if (!moments) { return c->snapshots[i].get(); }
    return c->snapshotsHoldMoments && c->snapshotMomentsComplete[i] ? c->snapshots[i].get() + n : nullptr;
}

// The buffers a gather over root + peers reads: set k = sources[k](root), then sources[k] of every peer as root's device reads it --
// the peer's own pointer on the same device or through an NVLink peer mapping, else a copy staged into root->gatherStage.  Root's
// stream is first ordered behind each peer's pending work.  PTC_ERR_STATE for a peer without a buffer or of another size.
typedef std::function<const float *(ptc_ctx *)> GatherSource;
static int gatherSets(ptc_ctx *root, ptc_ctx *const *peers, uint32_t nPeers, const GatherSource *sources, int nSets, FramebufferSet *sets)
{
    const size_t n = root->framebuffer.size();
    for (int k = 0; k < nSets; k++) { sets[k].fb[0] = sources[k](root); sets[k].count = 1; }
    size_t staged = 0;
    for (uint32_t g = 0; g < nPeers; g++) {
        ptc_ctx *peer = peers[g];
        bool present = peer && peer->committed && peer->framebuffer.size() == n;
        for (int k = 0; present && k < nSets; k++) { present = sources[k](peer) != nullptr; }
        if (!present) { CTX_FAIL(root, PTC_ERR_STATE, "peer %u has no framebuffer (or snapshot, or moments) of the same size", g); }
        // order the gather after the peer's pending renders
        CUDA_TRY(root, cudaSetDevice(peer->device));
        CUDA_TRY(root, cudaEventRecord(peer->framebufferReady, peer->stream));
        CUDA_TRY(root, cudaSetDevice(root->device));
        CUDA_TRY(root, cudaStreamWaitEvent(root->stream, peer->framebufferReady, 0));
        bool direct = peer->device == root->device;
        int canAccess = 0;
        if (!direct) { cudaDeviceCanAccessPeer(&canAccess, root->device, peer->device); }
        if (canAccess) {
            const cudaError_t e = cudaDeviceEnablePeerAccess(peer->device, 0);
            direct = e == cudaSuccess || e == cudaErrorPeerAccessAlreadyEnabled;
            cudaGetLastError();
        }
        for (int k = 0; k < nSets; k++) {
            if (direct) { sets[k].fb[sets[k].count++] = sources[k](peer); continue; }
            // no peer mapping: stage the peer's buffer into local memory first
            if (root->gatherStage.size() < (size_t)nSets * nPeers * n) {
                CUDA_TRY(root, cudaStreamSynchronize(root->stream)); // earlier gathers may still read the old buffer
                CUDA_TRY(root, root->gatherStage.reserve((size_t)nSets * nPeers * n));
            }
            float *slot = root->gatherStage.get() + staged * n; staged++;
            CUDA_TRY(root, cudaMemcpyPeerAsync(slot, root->device, sources[k](peer), peer->device, n * sizeof(float), root->stream));
            sets[k].fb[sets[k].count++] = slot;
        }
    }
    return PTC_OK;
}

// A free result slot of root (device buffer + pinned host buffer + event), allocated on first use
static int takeGatherSlot(ptc_ctx *root, uint32_t *ticketOut)
{
    uint32_t ticket = 0;
    while (ticket < root->gathers.size() && root->gathers[ticket].busy) { ticket++; }
    if (ticket == root->gathers.size()) { root->gathers.emplace_back(); }
    ptc_ctx::Gather &slot = root->gathers[ticket];
    // sized on first use, and again when the camera's resolution changed
    CUDA_TRY(root, slot.device.resize(root->framebuffer.size()));
    CUDA_TRY(root, slot.pinned.resize(root->framebuffer.size()));
    CUDA_TRY(root, slot.done.create());
    *ticketOut = ticket;
    return PTC_OK;
}

// After the kernels that read the contexts' buffers and wrote slot `ticket`'s device buffer: later work on the peers waits for those
// reads, the result goes to the slot's pinned buffer, and ptc_framebuffer_gather_end hands it out
static int finishGather(ptc_ctx *root, ptc_ctx *const *peers, uint32_t nPeers, uint32_t ticket)
{
    CUDA_TRY(root, cudaGetLastError());
    // renders that follow on any of the contexts must not overwrite what the kernels read
    CUDA_TRY(root, root->gatherRead.create());
    CUDA_TRY(root, cudaEventRecord(root->gatherRead, root->stream));
    for (uint32_t g = 0; g < nPeers; g++) { CUDA_TRY(root, cudaStreamWaitEvent(peers[g]->stream, root->gatherRead, 0)); }
    ptc_ctx::Gather &slot = root->gathers[ticket];
    CUDA_TRY(root, cudaMemcpyAsync(slot.pinned.get(), slot.device.get(), slot.device.size() * sizeof(float), cudaMemcpyDeviceToHost, root->stream));
    CUDA_TRY(root, cudaEventRecord(slot.done, root->stream));
    slot.busy = true;
    return PTC_OK;
}

extern "C" {

int ptc_framebuffer_gather_begin(ptc_ctx *root, ptc_ctx *const *peers, uint32_t nPeers, int snapshot, uint32_t divisor, uint32_t *ticketOut)
{
    NEED_COMMIT(root);
    if (!ticketOut || !divisor || (nPeers && !peers) || nPeers > PTC_MAX_PEERS) { CTX_FAIL(root, PTC_ERR_INVALID, "bad gather arguments"); }
    CUDA_TRY(root, cudaSetDevice(root->device));
    int rc = ensureFramebuffer(root);
    if (rc) { return rc; }
    const size_t n = root->framebuffer.size();
    // PTC_GATHER_MOMENTS: the second moments of an adaptive render or of the framebuffer renders
    const bool moments = snapshot == PTC_GATHER_MOMENTS;
    const GatherSource source = [&](ptc_ctx *c) { return gatherInput(c, snapshot, n, moments); };
    if (!source(root)) {
        if (moments) {
            CTX_FAIL(root, PTC_ERR_STATE, "no second moments of every sample on this context (option framebuffer_moments on since the last clear, or an adaptive render)");
        }
        CTX_FAIL(root, PTC_ERR_STATE, "no snapshot %d was rendered", snapshot);
    }
    FramebufferSet set;
    if ((rc = gatherSets(root, peers, nPeers, &source, 1, &set))) { return rc; }
    uint32_t ticket = 0;
    if ((rc = takeGatherSlot(root, &ticket))) { return rc; }
    gatherResolveKernel<<<std::min<uint32_t>((uint32_t)((n / 4 + 255) / 256) + 1, (uint32_t)root->gridSimple * 4), 256, 0, root->stream>>>(set, root->gathers[ticket].device.get(), (uint32_t)n, divisor);
    root->launches++;
    if ((rc = finishGather(root, peers, nPeers, ticket))) { return rc; }
    *ticketOut = ticket;
    return PTC_OK;
}

int ptc_framebuffer_gather_end(ptc_ctx *root, uint32_t ticket, float *out)
{
    NEED_COMMIT(root);
    if (!out || ticket >= root->gathers.size() || !root->gathers[ticket].busy) { CTX_FAIL(root, PTC_ERR_INVALID, "no gather in flight under ticket %u", ticket); }
    CUDA_TRY(root, cudaSetDevice(root->device));
    ptc_ctx::Gather &slot = root->gathers[ticket];
    CUDA_TRY(root, cudaEventSynchronize(slot.done));
    memcpy(out, slot.pinned.get(), root->framebuffer.size() * sizeof(float));
    slot.busy = false;
    return PTC_OK;
}

int ptc_framebuffer_gather(ptc_ctx *root, ptc_ctx *const *peers, uint32_t nPeers, uint32_t divisor, float *out)
{
    if (!out) { return PTC_ERR_INVALID; }
    uint32_t ticket = 0;
    const int rc = ptc_framebuffer_gather_begin(root, peers, nPeers, -1, divisor, &ticket);
    return rc ? rc : ptc_framebuffer_gather_end(root, ticket, out);
}

int ptc_adaptive_begin(ptc_ctx *ctx, const ptc_adaptive_desc *desc)
{
    NEED_COMMIT(ctx);
    if (!desc || !(desc->threshold > 0.f) || desc->min_spp < 2 || desc->step_spp < 1 || desc->max_spp < desc->min_spp) {
        CTX_FAIL(ctx, PTC_ERR_INVALID, "bad adaptive sampling descriptor (threshold > 0, min_spp >= 2, step_spp >= 1, max_spp >= min_spp)");
    }
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const int rc = ensureFramebuffer(ctx);
    if (rc) { return rc; }
    ptc_ctx::Adaptive &a = ctx->adaptive;
    const size_t pixels = (size_t)ctx->scene.view.width * ctx->scene.view.height;
    a.pixels = 0; // until every buffer is sized for `pixels`
    CUDA_TRY(ctx, ctx->moments.resize(3 * pixels));
    CUDA_TRY(ctx, a.counts.resize(pixels));
    CUDA_TRY(ctx, a.list.resize(pixels));
    CUDA_TRY(ctx, a.next.resize(pixels));
    CUDA_TRY(ctx, a.selected.resize(1));
    CUDA_TRY(ctx, a.selectedHost.resize(1));
    size_t scratchBytes = 0;
    CUDA_TRY(ctx, cub::DeviceSelect::If(nullptr, scratchBytes, a.next.get(), a.list.get(), a.selected.get(), (int)pixels, StillActive(), ctx->stream));
    CUDA_TRY(ctx, a.scratch.resize(std::max<size_t>(scratchBytes, 1)));
    a.pixels = pixels;
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->framebuffer.get(), 0, ctx->framebuffer.size() * sizeof(float), ctx->stream));
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->moments.get(), 0, 3 * pixels * sizeof(float), ctx->stream));
    CUDA_TRY(ctx, cudaMemsetAsync(a.counts.get(), 0, pixels * sizeof(uint32_t), ctx->stream));
    a.desc = *desc; a.n = 0; a.active = (uint32_t)pixels; a.on = true;
    ctx->momentsComplete = true; // the passes add the squares of every sample they add to the framebuffer
    return PTC_OK;
}

// One pass: samples n .. n + k - 1 of the active pixels (k = min_spp for the first pass, then min(step_spp, max_spp - n)), in
// one or more waves over the pixel list, then the stopping test and the stable selection of the pixels that go on.  The host
// needs the survivor count to size the next pass: one synchronisation per pass.
int ptc_adaptive_pass(ptc_ctx *ctx, uint64_t seed, int start, int last, uint32_t *activeOut, uint32_t *sppOut)
{
    NEED_COMMIT(ctx);
    ptc_ctx::Adaptive &a = ctx->adaptive;
    if (!a.on) { CTX_FAIL(ctx, PTC_ERR_STATE, "no adaptive render on this context: ptc_adaptive_begin first"); }
    if (a.pixels != (size_t)ctx->scene.view.width * ctx->scene.view.height || ctx->framebuffer.size() != 3 * a.pixels) {
        CTX_FAIL(ctx, PTC_ERR_STATE, "the resolution changed during the adaptive render");
    }
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    if (a.active) {
        const uint32_t k = a.n == 0 ? a.desc.min_spp : std::min(a.desc.step_spp, a.desc.max_spp - a.n);
        PassPixels pass; pass.list = a.n == 0 ? nullptr : a.list.get(); pass.count = a.active; pass.moments = ctx->moments.get();
        const int rc = renderInternal(ctx, seed, a.n, k, start, last, ctx->framebuffer.get(), ctx->stream, Checkpoints(), pass);
        if (rc) { return rc; }
        const uint32_t n = a.n + k;
        WaveParams wp; memset(&wp, 0, sizeof(wp));
        wp.nPixels = a.active; wp.pixels = pass.list;
        const double tau = (double)a.desc.threshold;
        adaptiveTestKernel<<<gridFor(ctx, a.active, 256), 256, 0, ctx->stream>>>(
            wp, ctx->framebuffer.get(), ctx->moments.get(), a.counts.get(), a.next.get(), (uint32_t)ctx->scene.view.width, (uint32_t)ctx->scene.view.height, tau * tau, n, a.desc.max_spp);
        CUDA_TRY(ctx, cudaGetLastError());
        size_t bytes = a.scratch.size();
        CUDA_TRY(ctx, cub::DeviceSelect::If(a.scratch.get(), bytes, a.next.get(), a.list.get(), a.selected.get(), (int)a.active, StillActive(), ctx->stream));
        CUDA_TRY(ctx, cudaMemcpyAsync(a.selectedHost.get(), a.selected.get(), sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
        ctx->launches += 2;
        a.n = n; a.active = *a.selectedHost.get();
    }
    if (activeOut) { *activeOut = a.active; }
    if (sppOut) { *sppOut = a.n; }
    return PTC_OK;
}

int ptc_adaptive_state(ptc_ctx *ctx, uint32_t *sppPerPixel, float *secondMoment)
{
    NEED_COMMIT(ctx);
    const ptc_ctx::Adaptive &a = ctx->adaptive;
    if (!a.on) { CTX_FAIL(ctx, PTC_ERR_STATE, "no adaptive render on this context: ptc_adaptive_begin first"); }
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    if (sppPerPixel) { CUDA_TRY(ctx, cudaMemcpyAsync(sppPerPixel, a.counts.get(), a.pixels * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream)); }
    if (secondMoment) { CUDA_TRY(ctx, cudaMemcpyAsync(secondMoment, ctx->moments.get(), 3 * a.pixels * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream)); }
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return PTC_OK;
}

int ptc_resolve_device(ptc_ctx *ctx, const float *accum, float *out, uint32_t spp, void *stream)
{
    NEED_COMMIT(ctx);
    if (!accum || !out || !spp) { CTX_FAIL(ctx, PTC_ERR_INVALID, "bad resolve arguments"); }
    const uint32_t n = 3u * (uint32_t)ctx->scene.view.width * (uint32_t)ctx->scene.view.height;
    resolveKernel<<<gridFor(ctx, n, 256), 256, 0, (cudaStream_t)stream>>>(accum, out, n, spp);
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
    return PTC_OK;
}

} // extern "C"

// ------------------------------------------------------------------------------------------------ queries (host buffers)
// A host array of a query, `n` elements, and its device scratch.  An input is uploaded before the launch, an output downloaded after
// it; an optional output with a null pointer is not downloaded (the kernel still writes its scratch).
template <typename T> struct HostArray { T *host; size_t n; bool up, down; Buffer<T> device; };
namespace host {
template <typename T> static HostArray<T> in(const T *p, size_t n) { return {const_cast<T *>(p), n, true, false}; } // never written
template <typename T> static HostArray<T> out(T *p, size_t n) { return {p, n, false, true}; }
template <typename T> static HostArray<T> inout(T *p, size_t n) { return {p, n, true, true}; }
template <typename T> static HostArray<T> optionalOut(T *p, size_t n) { return {p, n, false, p != nullptr}; }
}

// One query on host arrays, on the context's device and stream: scratch of at least one element per array (n = 0 works), the inputs
// uploaded, launch(the arrays' device pointers, in order) -- one kernel --, every output downloaded, one synchronisation.
// PTC_ERR_NOMEM when the scratch cannot be allocated, PTC_ERR_CUDA for any other failure.
template <typename Launch, typename... T>
static int query(ptc_ctx *ctx, Launch launch, HostArray<T>... a)
{
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    cudaError_t e = cudaSuccess;
    if (!(((e = a.device.resize(std::max<size_t>(a.n, 1))) == cudaSuccess) && ...)) { CTX_FAIL(ctx, PTC_ERR_NOMEM, "query scratch: %s", cudaGetErrorString(e)); }
    if (!((!a.up || !a.n || (e = cudaMemcpyAsync(a.device.get(), a.host, a.n * sizeof(T), cudaMemcpyHostToDevice, ctx->stream)) == cudaSuccess) && ...)) {
        CTX_FAIL(ctx, PTC_ERR_CUDA, "query upload: %s", cudaGetErrorString(e));
    }
    launch(a.device.get()...);
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
    if (!((!a.down || !a.n || (e = cudaMemcpyAsync(a.host, a.device.get(), a.n * sizeof(T), cudaMemcpyDeviceToHost, ctx->stream)) == cudaSuccess) && ...)) {
        CTX_FAIL(ctx, PTC_ERR_CUDA, "query download: %s", cudaGetErrorString(e));
    }
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return PTC_OK;
}

// ------------------------------------------------------------------------------------------------ denoising (denoise.cuh)
static int checkDenoiseDesc(ptc_ctx *ctx, const ptc_denoise_desc *desc)
{
    auto positive = [](float v) { return v > 0.f && std::isfinite(v); };
    if (!desc || desc->iterations > 10 || !positive(desc->sigma_l) || !(desc->sigma_n >= 0.f && std::isfinite(desc->sigma_n)) ||
        !positive(desc->sigma_z) || !positive(desc->sigma_a) || !positive(desc->eps)) {
        CTX_FAIL(ctx, PTC_ERR_INVALID, "bad denoise descriptor (iterations <= 10, sigma_l, sigma_z, sigma_a, eps > 0, sigma_n >= 0)");
    }
    return PTC_OK;
}

// The a-trous levels over ctx->denoise.colour[0] (the prepared colour records) on the context's stream; the result is in
// colour[desc->iterations & 1]
static int denoiseAtrous(ptc_ctx *ctx, const ptc_denoise_desc *desc, const float4 *guide)
{
    ptc_ctx::Denoise &d = ctx->denoise;
    const int width = ctx->scene.view.width, height = ctx->scene.view.height;
    DenoiseParams dp;
    dp.sigmaL = desc->sigma_l; dp.sigmaN = desc->sigma_n; dp.sigmaZ = desc->sigma_z; dp.sigmaA = desc->sigma_a; dp.eps = desc->eps;
    const dim3 block(32, 8), grid((unsigned)(width + 31) / 32, (unsigned)(height + 7) / 8);
    for (uint32_t i = 0; i < desc->iterations; i++) {
        denoiseAtrousKernel<<<grid, block, 0, ctx->stream>>>(d.colour[i & 1].get(), d.colour[(i + 1) & 1].get(), guide, width, height, 1 << i, dp);
        ctx->launches++;
        CUDA_TRY(ctx, cudaGetLastError());
    }
    return PTC_OK;
}

extern "C" {

int ptc_intersect(ptc_ctx *ctx, const ptc_ray *rays, uint32_t n, ptc_hit *hits)
{
    NEED_COMMIT(ctx);
    if (n && (!rays || !hits)) { return PTC_ERR_INVALID; }
    return query(ctx, [&](const ptc_ray *r, ptc_hit *h) { intersectKernel<<<gridFor(ctx, n), 128, 0, ctx->stream>>>(ctx->scene.view, r, n, h, nullptr); },
                 host::in(rays, n), host::out(hits, n));
}
int ptc_intersect_instanced(ptc_ctx *ctx, const ptc_ray *rays, uint32_t n, ptc_hit *hits, uint32_t *instIds)
{
    NEED_COMMIT(ctx);
    if (n && (!rays || !hits || !instIds)) { return PTC_ERR_INVALID; }
    return query(ctx, [&](const ptc_ray *r, ptc_hit *h, uint32_t *inst) { intersectKernel<<<gridFor(ctx, n), 128, 0, ctx->stream>>>(ctx->scene.view, r, n, h, (uint2 *)inst); },
                 host::in(rays, n), host::out(hits, n), host::out(instIds, (size_t)2 * n));
}
int ptc_intersect_full(ptc_ctx *ctx, const ptc_ray *rays, uint32_t n, ptc_isect *out)
{
    NEED_COMMIT(ctx);
    if (n && (!rays || !out)) { return PTC_ERR_INVALID; }
    return query(ctx, [&](const ptc_ray *r, ptc_isect *o) { intersectFullKernel<<<gridFor(ctx, n), 128, 0, ctx->stream>>>(ctx->scene.view, r, n, o); },
                 host::in(rays, n), host::out(out, n));
}
int ptc_occluded(ptc_ctx *ctx, const ptc_ray *rays, const float *maxT, uint32_t n, uint8_t *occluded)
{
    NEED_COMMIT(ctx);
    if (n && (!rays || !maxT || !occluded)) { return PTC_ERR_INVALID; }
    return query(ctx, [&](const ptc_ray *r, const float *t, uint8_t *o) { occludedKernel<<<gridFor(ctx, n), 128, 0, ctx->stream>>>(ctx->scene.view, r, t, n, o); },
                 host::in(rays, n), host::in(maxT, n), host::out(occluded, n));
}
// the volumetric queries' per-ray event lists are optional outputs
int ptc_occluded_volumetric(ptc_ctx *ctx, const ptc_ray *rays, const float *maxT, uint32_t n, uint8_t *occluded, uint32_t *nEvents, float *eventT, uint32_t *eventMedium)
{
    NEED_COMMIT(ctx);
    if (n && (!rays || !maxT || !occluded)) { return PTC_ERR_INVALID; }
    return query(ctx,
                 [&](const ptc_ray *r, const float *t, uint8_t *o, uint32_t *en, float *et, uint32_t *em) {
                     occludedVolumetricKernel<<<gridFor(ctx, n), 128, 0, ctx->stream>>>(ctx->scene.view, r, t, n, o, en, et, em);
                 },
                 host::in(rays, n), host::in(maxT, n), host::out(occluded, n), host::optionalOut(nEvents, n),
                 host::optionalOut(eventT, (size_t)n * PTC_MAX_EVENTS), host::optionalOut(eventMedium, (size_t)n * PTC_MAX_EVENTS));
}
int ptc_intersect_volumetric(ptc_ctx *ctx, const ptc_ray *rays, uint32_t n, ptc_isect *out, uint32_t *nEvents, float *eventT, uint32_t *eventMedium)
{
    NEED_COMMIT(ctx);
    if (n && (!rays || !out)) { return PTC_ERR_INVALID; }
    return query(ctx,
                 [&](const ptc_ray *r, ptc_isect *o, uint32_t *en, float *et, uint32_t *em) {
                     intersectVolumetricKernel<<<gridFor(ctx, n), 128, 0, ctx->stream>>>(ctx->scene.view, r, n, o, en, et, em);
                 },
                 host::in(rays, n), host::out(out, n), host::optionalOut(nEvents, n), host::optionalOut(eventT, (size_t)n * PTC_MAX_EVENTS),
                 host::optionalOut(eventMedium, (size_t)n * PTC_MAX_EVENTS));
}
int ptc_intersect_device(ptc_ctx *ctx, const ptc_ray *rays, uint32_t n, ptc_hit *hits, void *stream)
{
    NEED_COMMIT(ctx);
    intersectKernel<<<gridFor(ctx, n), 128, 0, (cudaStream_t)stream>>>(ctx->scene.view, rays, n, hits, nullptr);
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
    return PTC_OK;
}
int ptc_occluded_device(ptc_ctx *ctx, const ptc_ray *rays, const float *maxT, uint32_t n, uint8_t *occluded, void *stream)
{
    NEED_COMMIT(ctx);
    occludedKernel<<<gridFor(ctx, n), 128, 0, (cudaStream_t)stream>>>(ctx->scene.view, rays, maxT, n, occluded);
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
    return PTC_OK;
}
int ptc_camera_rays(ptc_ctx *ctx, const float *rowCol, uint32_t n, ptc_ray *rays)
{
    NEED_COMMIT(ctx);
    return query(ctx, [&](const float *rc, ptc_ray *r) { cameraRaysKernel<<<gridFor(ctx, n), 128, 0, ctx->stream>>>(ctx->scene.view, rc, n, r); },
                 host::in(rowCol, (size_t)2 * n), host::out(rays, n));
}
// Guide buffers (denoise.cuh: aovKernel): the caller's sums go up, the kernel adds to them, they come back
int ptc_render_aovs(ptc_ctx *ctx, uint64_t seed, uint32_t firstSample, uint32_t nSpp, float *albedo, float *normal, float *depth, uint32_t *hits)
{
    NEED_COMMIT(ctx);
    if (!albedo || !normal || !depth || !hits) { CTX_FAIL(ctx, PTC_ERR_INVALID, "null guide buffer"); }
    if (!nSpp) { return PTC_OK; } // no samples: the sums stay as they are
    const size_t pixels = (size_t)ctx->scene.view.width * ctx->scene.view.height;
    return query(ctx,
                 [&](float *a, float *nrm, float *z, uint32_t *h) {
                     aovKernel<<<gridFor(ctx, (uint32_t)pixels), 128, 0, ctx->stream>>>(ctx->scene.view, seed, firstSample, nSpp, a, nrm, z, h);
                 },
                 host::inout(albedo, 3 * pixels), host::inout(normal, 3 * pixels), host::inout(depth, pixels), host::inout(hits, pixels));
}

// The same guide sums from zero into the context's device buffers, then the guide records of ptc_denoise's prepare step
int ptc_framebuffer_guides(ptc_ctx *ctx, uint64_t seed, uint32_t firstSample, uint32_t nSpp, float *albedo, float *normal, float *depth, uint32_t *hits)
{
    NEED_COMMIT(ctx);
    if (!nSpp) { CTX_FAIL(ctx, PTC_ERR_INVALID, "n_spp must be > 0: the guide records are means over the samples"); }
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const size_t pixels = (size_t)ctx->scene.view.width * ctx->scene.view.height;
    CUDA_TRY(ctx, ctx->aovs.resize(8 * pixels));
    ptc_ctx::Guides &g = ctx->guides;
    g.aovSpp = 0; // no guides until this call has enqueued them
    CUDA_TRY(ctx, g.records.resize(2 * pixels));
    float *d = ctx->aovs.get();
    float *dAlbedo = d, *dNormal = d + 3 * pixels, *dDepth = d + 6 * pixels;
    uint32_t *dHits = (uint32_t *)(d + 7 * pixels);
    CUDA_TRY(ctx, cudaMemsetAsync(d, 0, 8 * pixels * sizeof(float), ctx->stream));
    aovKernel<<<gridFor(ctx, (uint32_t)pixels), 128, 0, ctx->stream>>>(ctx->scene.view, seed, firstSample, nSpp, dAlbedo, dNormal, dDepth, dHits);
    denoiseGuideKernel<<<gridFor(ctx, (uint32_t)pixels, 256), 256, 0, ctx->stream>>>(dAlbedo, dNormal, dDepth, dHits, nSpp, (uint32_t)pixels, g.records.get());
    ctx->launches += 2;
    CUDA_TRY(ctx, cudaGetLastError());
    const struct { void *dst; const void *src; size_t bytes; } fetches[] = {
        {albedo, dAlbedo, 3 * pixels * 4}, {normal, dNormal, 3 * pixels * 4}, {depth, dDepth, pixels * 4}, {hits, dHits, pixels * 4}};
    bool fetched = false;
    for (const auto &f : fetches) {
        if (f.dst) { CUDA_TRY(ctx, cudaMemcpyAsync(f.dst, f.src, f.bytes, cudaMemcpyDeviceToHost, ctx->stream)); fetched = true; }
    }
    if (fetched) { CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream)); }
    g.aovSpp = nSpp; g.width = ctx->scene.view.width; g.height = ctx->scene.view.height;
    return PTC_OK;
}

// The filter (denoise.cuh): inputs staged in one device buffer, one kernel that builds the colour and guide records, one a-trous
// launch per iteration between the two colour buffers, the last one's colours copied back
int ptc_denoise(ptc_ctx *ctx, const ptc_denoise_desc *desc, const ptc_denoise_input *in, float *out)
{
    NEED_COMMIT(ctx);
    int rc = checkDenoiseDesc(ctx, desc);
    if (rc) { return rc; }
    if (!in || !out || !in->sums || !in->moments || !in->albedo_rgb || !in->normal_xyz || !in->depth || !in->hits) {
        CTX_FAIL(ctx, PTC_ERR_INVALID, "missing denoise input");
    }
    if (!in->aov_spp) { CTX_FAIL(ctx, PTC_ERR_INVALID, "aov_spp must be > 0"); }
    const int width = ctx->scene.view.width, height = ctx->scene.view.height;
    const size_t pixels = (size_t)width * height;
    if (in->counts) {
        for (size_t p = 0; p < pixels; p++) { if (in->counts[p] < 2) { CTX_FAIL(ctx, PTC_ERR_INVALID, "pixel %zu has %u samples: the variance needs 2", p, in->counts[p]); } }
    } else if (in->spp < 2) { CTX_FAIL(ctx, PTC_ERR_INVALID, "spp must be >= 2: the variance needs 2 samples"); }
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    ptc_ctx::Denoise &d = ctx->denoise;
    CUDA_TRY(ctx, d.inputs.resize(15 * pixels));
    CUDA_TRY(ctx, d.guide.resize(2 * pixels));
    CUDA_TRY(ctx, d.colour[0].resize(pixels));
    CUDA_TRY(ctx, d.colour[1].resize(pixels));
    DenoiseInputs di;
    float *f = d.inputs.get();
    di.sums = f; di.moments = f + 3 * pixels; di.albedo = f + 6 * pixels; di.normal = f + 9 * pixels; di.depth = f + 12 * pixels;
    di.hits = (const uint32_t *)(f + 13 * pixels); di.counts = in->counts ? (const uint32_t *)(f + 14 * pixels) : nullptr;
    di.spp = in->spp; di.aovSpp = in->aov_spp; di.nPixels = (uint32_t)pixels;
    const struct { void *dst; const void *src; size_t bytes; } uploads[] = {
        {f, in->sums, 3 * pixels * 4}, {f + 3 * pixels, in->moments, 3 * pixels * 4}, {f + 6 * pixels, in->albedo_rgb, 3 * pixels * 4},
        {f + 9 * pixels, in->normal_xyz, 3 * pixels * 4}, {f + 12 * pixels, in->depth, pixels * 4}, {f + 13 * pixels, in->hits, pixels * 4},
        {f + 14 * pixels, in->counts, in->counts ? pixels * 4 : 0}};
    for (const auto &u : uploads) { if (u.bytes) { CUDA_TRY(ctx, cudaMemcpyAsync(u.dst, u.src, u.bytes, cudaMemcpyHostToDevice, ctx->stream)); } }
    denoisePrepareKernel<<<gridFor(ctx, (uint32_t)pixels, 256), 256, 0, ctx->stream>>>(di, d.colour[0].get(), d.guide.get());
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
    if ((rc = denoiseAtrous(ctx, desc, d.guide.get()))) { return rc; }
    std::vector<float4> result(pixels);
    CUDA_TRY(ctx, cudaMemcpyAsync(result.data(), d.colour[desc->iterations & 1].get(), pixels * sizeof(float4), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    for (size_t p = 0; p < pixels; p++) { out[3 * p] = result[p].x; out[3 * p + 1] = result[p].y; out[3 * p + 2] = result[p].z; }
    return PTC_OK;
}

// ptc_denoise on what the contexts hold: the colour records straight from the (peer-read) sums and moments, the guide records of
// ptc_framebuffer_guides, the same a-trous levels, and the image out through a gather slot
int ptc_framebuffer_denoise_begin(ptc_ctx *root, ptc_ctx *const *peers, uint32_t nPeers, int snapshot, uint32_t spp, const ptc_denoise_desc *desc,
                                  uint32_t *ticketOut)
{
    NEED_COMMIT(root);
    int rc = checkDenoiseDesc(root, desc);
    if (rc) { return rc; }
    if (!ticketOut || (nPeers && !peers) || nPeers > PTC_MAX_PEERS) { CTX_FAIL(root, PTC_ERR_INVALID, "bad denoise arguments"); }
    const ptc_ctx::Adaptive &a = root->adaptive;
    if (!a.on && spp < 2) { CTX_FAIL(root, PTC_ERR_INVALID, "spp must be >= 2: the variance needs 2 samples"); }
    CUDA_TRY(root, cudaSetDevice(root->device));
    if ((rc = ensureFramebuffer(root))) { return rc; }
    const size_t n = root->framebuffer.size(), pixels = n / 3;
    if (!root->guides.aovSpp || root->guides.width != root->scene.view.width || root->guides.height != root->scene.view.height || 2 * pixels != root->guides.records.size()) { CTX_FAIL(root, PTC_ERR_STATE, "no guides of this resolution: ptc_framebuffer_guides first"); }
    if (a.on && a.n == 0) { CTX_FAIL(root, PTC_ERR_STATE, "the adaptive render has no pass yet"); }
    if (a.on && snapshot >= 0) { CTX_FAIL(root, PTC_ERR_STATE, "an adaptive render keeps no checkpoint snapshots"); }
    const GatherSource sources[2] = {[&](ptc_ctx *c) { return gatherInput(c, snapshot, n, false); }, [&](ptc_ctx *c) { return gatherInput(c, snapshot, n, true); }};
    if (!sources[0](root)) { CTX_FAIL(root, PTC_ERR_STATE, "no snapshot %d was rendered", snapshot); }
    if (!sources[1](root)) {
        CTX_FAIL(root, PTC_ERR_STATE, "no second moments of every sample of this image (option framebuffer_moments on since the last clear, or an adaptive render)");
    }
    FramebufferSet sets[2];
    if ((rc = gatherSets(root, peers, nPeers, sources, 2, sets))) { return rc; }
    ptc_ctx::Denoise &d = root->denoise;
    CUDA_TRY(root, d.colour[0].resize(pixels));
    CUDA_TRY(root, d.colour[1].resize(pixels));
    uint32_t ticket = 0;
    if ((rc = takeGatherSlot(root, &ticket))) { return rc; }
    const uint32_t grid = gridFor(root, (uint32_t)pixels, 256);
    denoiseGatherKernel<<<grid, 256, 0, root->stream>>>(sets[0], sets[1], a.on ? a.counts.get() : nullptr, spp, (uint32_t)pixels, d.colour[0].get());
    root->launches++;
    CUDA_TRY(root, cudaGetLastError());
    if ((rc = denoiseAtrous(root, desc, root->guides.records.get()))) { return rc; }
    denoisePackKernel<<<grid, 256, 0, root->stream>>>(d.colour[desc->iterations & 1].get(), root->gathers[ticket].device.get(), (uint32_t)pixels);
    root->launches++;
    if ((rc = finishGather(root, peers, nPeers, ticket))) { return rc; }
    *ticketOut = ticket;
    return PTC_OK;
}

int ptc_philox4x32_10(ptc_ctx *ctx, const uint32_t *counters, const uint32_t *keys, uint32_t n, uint32_t *out)
{
    if (!ctx || (n && (!counters || !keys || !out))) { return PTC_ERR_INVALID; }
    return query(ctx, [&](const uint32_t *c, const uint32_t *k, uint32_t *o) { philoxKernel<<<std::max(1u, (n + 127) / 128), 128, 0, ctx->stream>>>(c, k, n, o); },
                 host::in(counters, (size_t)4 * n), host::in(keys, (size_t)2 * n), host::out(out, (size_t)4 * n));
}
int ptc_uniforms(ptc_ctx *ctx, uint64_t seed, const uint32_t *streams, uint32_t nStreams, uint32_t draws, float *out)
{
    if (!ctx || (nStreams && draws && (!streams || !out))) { return PTC_ERR_INVALID; }
    return query(ctx, [&](const uint32_t *s, float *o) { uniformsKernel<<<std::max(1u, (nStreams + 127) / 128), 128, 0, ctx->stream>>>(seed, s, nStreams, draws, o); },
                 host::in(streams, (size_t)3 * nStreams), host::out(out, (size_t)nStreams * draws));
}
int ptc_bsdf_eval(ptc_ctx *ctx, uint32_t material, const ptc_isect *isects, const float *wi, uint32_t n, float *f, float *pdf)
{
    NEED_COMMIT(ctx);
    if (material >= ctx->scene.materials.size()) { CTX_FAIL(ctx, PTC_ERR_INVALID, "material id out of range"); }
    return query(ctx,
                 [&](const ptc_isect *is, const float *w, float *fo, float *p) {
                     bsdfEvalKernel<<<gridFor(ctx, n), 128, 0, ctx->stream>>>(ctx->scene.view, material, is, w, n, fo, p);
                 },
                 host::in(isects, n), host::in(wi, (size_t)3 * n), host::out(f, (size_t)3 * n), host::out(pdf, n));
}
int ptc_bsdf_sample(ptc_ctx *ctx, uint32_t material, const ptc_isect *isects, const float *xi, uint32_t n, float *wi, float *pdf, float *thr)
{
    NEED_COMMIT(ctx);
    if (material >= ctx->scene.materials.size()) { CTX_FAIL(ctx, PTC_ERR_INVALID, "material id out of range"); }
    return query(ctx,
                 [&](const ptc_isect *is, const float *x, float *w, float *p, float *t) {
                     bsdfSampleKernel<<<gridFor(ctx, n), 128, 0, ctx->stream>>>(ctx->scene.view, material, is, x, n, w, p, t);
                 },
                 host::in(isects, n), host::in(xi, (size_t)3 * n), host::out(wi, (size_t)3 * n), host::out(pdf, n), host::out(thr, (size_t)3 * n));
}
int ptc_light_sample(ptc_ctx *ctx, const float *ref, const float *xi, uint32_t n, ptc_light_sample_t *out)
{
    NEED_COMMIT(ctx);
    if (!ctx->scene.view.nLights) { CTX_FAIL(ctx, PTC_ERR_STATE, "scene has no lights"); }
    return query(ctx, [&](const float *r, const float *x, ptc_light_sample_t *o) { lightSampleKernel<<<gridFor(ctx, n), 128, 0, ctx->stream>>>(ctx->scene.view, r, x, n, o); },
                 host::in(ref, (size_t)3 * n), host::in(xi, (size_t)3 * n), host::out(out, n));
}
int ptc_light_pdf(ptc_ctx *ctx, const ptc_ray *rays, uint32_t n, float *pdf)
{
    NEED_COMMIT(ctx);
    return query(ctx, [&](const ptc_ray *r, float *p) { lightPdfKernel<<<gridFor(ctx, n), 128, 0, ctx->stream>>>(ctx->scene.view, r, n, p); },
                 host::in(rays, n), host::out(pdf, n));
}
int ptc_environment_radiance(ptc_ctx *ctx, const float *dirs, uint32_t n, float *rgb)
{
    NEED_COMMIT(ctx);
    return query(ctx, [&](const float *d, float *o) { envRadianceKernel<<<gridFor(ctx, n), 128, 0, ctx->stream>>>(ctx->scene.view, d, n, o); },
                 host::in(dirs, (size_t)3 * n), host::out(rgb, (size_t)3 * n));
}
int ptc_radiance_replay(ptc_ctx *ctx, const ptc_ray *rays, const float *xi, uint32_t stride, uint32_t n, int start, int last, float *rgb)
{
    NEED_COMMIT(ctx);
    if (last == -1 || last > PTC_MAX_BOUNCES) { last = PTC_MAX_BOUNCES; }
    const auto kernel = ctx->options.integrator == PTC_INTEGRATOR_VOLUME_PATH_TRACER ? volumeReplayKernel : radianceReplayKernel;
    return query(ctx, [&](const ptc_ray *r, const float *x, float *o) { kernel<<<gridFor(ctx, n), 128, 0, ctx->stream>>>(ctx->scene.view, r, x, stride, n, start, last, o); },
                 host::in(rays, n), host::in(xi, (size_t)n * stride), host::out(rgb, (size_t)3 * n));
}

int ptc_num_lights(ptc_ctx *ctx, uint32_t *out) { NEED_COMMIT(ctx); *out = ctx->scene.view.nLights; return PTC_OK; }

int ptc_get_stats(ptc_ctx *ctx, ptc_stats *out)
{
    if (!ctx || !out) { return PTC_ERR_INVALID; }
    memset(out, 0, sizeof(*out));
    unsigned long long totals[6] = {0, 0, 0, 0, 0, 0};
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    collectTimings(ctx);
    cudaMemcpy(totals, ctx->totals.get(), sizeof(totals), cudaMemcpyDeviceToHost);
    out->closest_rays = totals[0]; out->shadow_rays = totals[1]; out->samples = ctx->samples; out->kernel_launches = ctx->launches;
    out->extend_inner_visits = totals[2]; out->extend_triangle_tests = totals[3];
    out->shadow_inner_visits = totals[4]; out->shadow_triangle_tests = totals[5];
    const Committed &sc = ctx->scene; // before ptc_commit: zeros
    out->bvh_nodes = sc.view.bvh.nNodes; out->bvh_triangles = sc.bvhTriangles;
    out->bvh_bytes = (size_t)sc.view.bvh.nNodes * sizeof(WideNode) + (size_t)sc.bvhTriangles * sizeof(LeafTriangle);
    out->extend_launches = ctx->stageLaunches[STAGE_EXTEND]; out->shadow_launches = ctx->stageLaunches[STAGE_SHADOW];
    out->shade_launches = ctx->stageLaunches[STAGE_SHADE];
    out->extend_ms = (float)ctx->stageMs[STAGE_EXTEND]; out->shadow_ms = (float)ctx->stageMs[STAGE_SHADOW];
    out->shade_ms = (float)ctx->stageMs[STAGE_SHADE]; out->other_ms = (float)ctx->stageMs[STAGE_OTHER];
    out->last_render_ms = ctx->lastRenderMs;
    out->bvh_build_ms = sc.bvhBuildMs; out->bvh_builder = (uint32_t)ctx->options.bvhBuilder; out->bvh_depth = sc.bvhDepth;
    out->bvh_ploc_iterations = sc.bvhPlocIterations;
    return PTC_OK;
}

int ptc_get_wave_counts(ptc_ctx *ctx, uint32_t *extend, uint32_t *shadow, uint32_t capacity)
{
    if (!ctx || !extend || !shadow) { return PTC_ERR_INVALID; }
    std::vector<BounceCounters> host(CNT_STRIDE);
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    if (cudaMemcpy(host.data(), ctx->counters.get(), CNT_STRIDE * sizeof(BounceCounters), cudaMemcpyDeviceToHost) != cudaSuccess) { CTX_FAIL(ctx, PTC_ERR_CUDA, "cudaMemcpy failed"); }
    for (uint32_t k = 0; k < capacity && k < CNT_STRIDE; k++) { extend[k] = host[k].extendCount; shadow[k] = host[k].shadowCount + host[k].scatterCount; }
    return PTC_OK;
}

int ptc_reset_stats(ptc_ctx *ctx)
{
    if (!ctx) { return PTC_ERR_INVALID; }
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    collectTimings(ctx);
    cudaMemset(ctx->totals.get(), 0, 6 * sizeof(unsigned long long));
    ctx->samples = 0; ctx->launches = 0;
    for (int i = 0; i < 4; i++) { ctx->stageMs[i] = 0; ctx->stageLaunches[i] = 0; }
    return PTC_OK;
}

int ptc_set_option(ptc_ctx *ctx, const char *name, int64_t value)
{
    if (!ctx || !name) { return PTC_ERR_INVALID; }
    if (!strcmp(name, "paths_per_wave")) { // path indices are 32-bit
        if (value < 1024 || value > (int64_t)1 << 30) { CTX_FAIL(ctx, PTC_ERR_INVALID, "paths_per_wave must be in [1024, 2^30]"); }
        ctx->options.pathsPerWave = value; return PTC_OK;
    }
    if (!strcmp(name, "stage_timing")) { ctx->options.stageTiming = value != 0; return PTC_OK; }
    if (!strcmp(name, "overlap_shadow")) { ctx->options.overlapShadow = value != 0; return PTC_OK; }
    if (!strcmp(name, "lanes")) { // part-waves traced side by side (ptc_ctx::lanes)
        if (value < 0 || value > PTC_MAX_LANES) { CTX_FAIL(ctx, PTC_ERR_INVALID, "lanes must be in [0, %d] (0: chosen per wave)", PTC_MAX_LANES); }
        ctx->options.lanes = (int)value; return PTC_OK;
    }
    if (!strcmp(name, "count_traversal")) { ctx->options.countTraversal = value != 0; return PTC_OK; }
    if (!strcmp(name, "volume_megakernel")) { ctx->options.volumeMegakernel = value != 0; return PTC_OK; }
    if (!strcmp(name, "framebuffer_moments")) { // takes effect for the moments at the next ptc_framebuffer_clear
        ctx->options.framebufferMoments = value != 0;
        if (!ctx->options.framebufferMoments && !ctx->adaptive.on) { ctx->momentsComplete = false; } // an adaptive render's moments stay complete
        return PTC_OK;
    }
    if (!strcmp(name, "bvh_builder")) { // before ptc_commit; 1 = device (default), 0 = host binned SAH
        if (ctx->committed) { CTX_FAIL(ctx, PTC_ERR_STATE, "bvh_builder must be set before ptc_commit"); }
        if (value != 0 && value != 1) { CTX_FAIL(ctx, PTC_ERR_INVALID, "bvh_builder must be 0 (host) or 1 (device)"); }
        ctx->options.bvhBuilder = (int)value; return PTC_OK;
    }
    CTX_FAIL(ctx, PTC_ERR_INVALID, "unknown option %s", name);
}

int ptc_count_traversal(ptc_ctx *ctx, const ptc_ray *rays, uint32_t n, uint64_t *inner, uint64_t *tris)
{
    NEED_COMMIT(ctx);
    if (!ctx->hostBvh) { // host copy of the device-resident BVH for the scalar traversal
        cudaSetDevice(ctx->device);
        const Committed &sc = ctx->scene;
        WideBVH bvh;
        bvh.nodes.resize(sc.view.bvh.nNodes); bvh.triangles.resize(sc.bvhTriangles); bvh.placements = sc.placements;
        if (sc.view.bvh.nNodes) {
            CUDA_TRY(ctx, cudaMemcpy(bvh.nodes.data(), sc.view.bvh.nodes, bvh.nodes.size() * sizeof(WideNode), cudaMemcpyDeviceToHost));
            CUDA_TRY(ctx, cudaMemcpy(bvh.triangles.data(), sc.view.bvh.triangles, bvh.triangles.size() * sizeof(LeafTriangle), cudaMemcpyDeviceToHost));
        }
        ctx->hostBvh = std::move(bvh);
    }
    TraversalCounts c;
    for (uint32_t i = 0; i < n; i++) { traverseReference(*ctx->hostBvh, rays[i].origin, rays[i].direction, PTC_TNEAR, PTC_TFAR, false, nullptr, nullptr, &c); }
    if (inner) { *inner = c.innerVisits; }
    if (tris) { *tris = c.triangleTests; }
    return PTC_OK;
}

int ptc_bvh_selfcheck(const float *P, uint32_t nv, const uint32_t *I, uint32_t nt, const ptc_ray *rays, uint32_t nRays, float *tBvh,
                      uint32_t *primBvh, float *tBrute, uint32_t *primBrute, uint64_t stats[6])
{
    double cost = 0;
    return ptc_bvh_selfcheck_builder(0, P, nv, I, nt, rays, nRays, tBvh, primBvh, tBrute, primBrute, stats, &cost);
}

int ptc_bvh_selfcheck_builder(int builder, const float *P, uint32_t nv, const uint32_t *I, uint32_t nt, const ptc_ray *rays, uint32_t nRays,
                              float *tBvh, uint32_t *primBvh, float *tBrute, uint32_t *primBrute, uint64_t stats[6], double *sahCost)
{
    if (builder != 0 && builder != 1) { return PTC_ERR_INVALID; }
    if (!P || !I || !stats || (nRays && (!rays || !tBvh || !primBvh))) { return PTC_ERR_INVALID; }
    std::vector<float> positions4((size_t)nv * 4, 0.f);
    std::vector<uint32_t> prims4((size_t)nt * 4, 0u);
    for (uint32_t v = 0; v < nv; v++) { for (int a = 0; a < 3; a++) { positions4[4 * (size_t)v + a] = P[3 * (size_t)v + a]; } }
    for (uint32_t t = 0; t < nt; t++) {
        for (int a = 0; a < 3; a++) { if (I[3 * (size_t)t + a] >= nv) { return PTC_ERR_INVALID; } prims4[4 * (size_t)t + a] = I[3 * (size_t)t + a]; }
    }
    WideBVH bvh;
    try {
        if (builder == 1) { buildWideBVHEmulated(positions4.data(), prims4.data(), nt, bvh); }
        else { buildWideBVH(positions4.data(), prims4.data(), nt, bvh); }
    } catch (const std::exception &) { return PTC_ERR_INVALID; }
    if (sahCost) { *sahCost = wideBVHCost(bvh); }
    uint64_t slots = 0;
    for (const WideNode &n : bvh.nodes) { for (int s = 0; s < 8; s++) { slots += n.meta[s] ? 1 : 0; } }
    TraversalCounts counts;
    for (uint32_t r = 0; r < nRays; r++) {
        const float *o = rays[r].origin, *d = rays[r].direction;
        tBvh[r] = PTC_TFAR; primBvh[r] = PTC_MISS;
        traverseReference(bvh, o, d, PTC_TNEAR, PTC_TFAR, false, &tBvh[r], &primBvh[r], &counts);
        if (!tBrute || !primBrute) { continue; } // statistics only
        float best = PTC_TFAR; uint32_t bestPrim = PTC_MISS; bool found = false;
        for (const LeafTriangle &tri : bvh.triangles) {
            const float4 a = make_float4(tri.v0[0], tri.v0[1], tri.v0[2], 0.f), b = make_float4(tri.e1[0], tri.e1[1], tri.e1[2], 0.f),
                         c = make_float4(tri.e2[0], tri.e2[1], tri.e2[2], 0.f);
            float t, u, v;
            if (triangleTest(a, b, c, o[0], o[1], o[2], d[0], d[1], d[2], PTC_TNEAR, best, t, u, v)) {
                if (!(found && t == best && tri.prim < bestPrim)) { best = t; bestPrim = tri.prim; }
                found = true;
            }
        }
        tBrute[r] = best; primBrute[r] = bestPrim;
    }
    stats[0] = bvh.nodes.size(); stats[1] = bvh.triangles.size(); stats[2] = slots; stats[3] = bvh.maxDepth;
    stats[4] = counts.innerVisits; stats[5] = counts.triangleTests;
    return PTC_OK;
}

} // extern "C"
