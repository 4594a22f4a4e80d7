// VolumePathTracer as wavefront stages (SURVEY 8(f) N3, src/volume_path_tracer.cpp:14-131): the same loop as volume.cuh's
// one-thread-per-path volumeRadiance, cut where it traces rays, so that rays are traced by persistent traversal warps with lane
// refill and the shading runs per material class over dense path slots -- the layout of the PathTracer wavefront (pathed_cuda.cu).
// Included by pathed_cuda.cu after the PathTracer kernels (uses PathBuffers, BounceCounters, warpAppend, finishPath, ...).
//
// What makes the reference's loop wavefront-shaped after all:
//  * The MIS probe ray of DirectLightingHelper::Ld (src/direct_lighting_helper.cpp:139-187; containers are skipped) and the
//    continuation ray of VolumePathTracer::L (src/volume_path_tracer.cpp:52-53; containers are hit) are the SAME ray with two
//    acceptance rules.  ONE traversal answers both: it runs with the filtered rule (the farther interval) and keeps, next to the
//    filtered closest hit, the closest candidate of ALL surfaces under the plain rule (`PlainBest`: Embree's own interval test
//    T <= |den| * tfar against the plain hit distance, ties to the larger primitive index as in traverse.cuh).  Every surface in
//    front of the plain hit is in front of the filtered hit as well, so the filtered traversal meets it.  16.3 -> 12.3 rays per
//    sample on cornell-medium, bit-identical hits.
//  * Both kinds of shadow rays (light sampling at a surface vertex, :75-137, and at a scatter point inside a medium,
//    src/volume_helper.cpp:12-70) need the volume events of an unoccluded ray only to turn them into ONE transmittance; the
//    traversal warp does that when the ray ends (it holds origin, direction and the events) and stores 16 bytes, so no event list
//    leaves the kernel.  Only the count (0, 1, 2, more) and the two nearest distinct distances matter (rayTransmission applies
//    nothing to more than two events, volumeDirectLights applies zero), so three events per lane are kept.
//  * The random numbers of vertex b -- scatter distance, scatter light sample, BSDF sample, light sample, in that order -- are all
//    drawn in the material stage of vertex b, one thread, one Philox stream (pixel, sample, b).
// Per bounce k >= 1:  merged extend (queue) | shadow (S1 queue) | scatter shadow (S2 queue)  ->  volumeLogic(k)  ->  volumeMaterial<class>(k).
// Bounce 0 (camera ray) is SampleIntegrator::samplePixel, shared with the PathTracer: traverseKernel, logicKernel(0), containerKernel.
//
// The light-sampling terms are multiplied by their transmittance AFTER the other factors ((((Le w) f) cos / pdf) tr instead of
// ((((Le tr) w) f) cos) / pdf): bit-identical when tr = 1 (no event on the shadow ray), within 2 ulp otherwise.
#pragma once

#define FLAG_SCATTER 0x1000u /* a scatter-point shadow ray (S2) of the segment that arrived at this vertex is pending */
#define FLAG_LAST 0x2000u    /* the path ends after this bounce's logic stage (bounce limit reached or modulation black) */
#define FLAG_TRACED 0x4000u  /* the merged probe / continuation ray of this slot was traced */

struct VolumeBuffers {
    float4 *probeHit;       // filtered closest hit of the merged ray (t, u, v, prim); written only for scenes with containers
    float4 *shadowTr;       // outcome of S1 by slot: transmittance rgb, w = 1 when occluded
    float4 *scatter;        // S2 by slot, 3 float4: origin xyz, distance | direction xyz, medium | contribution rgb (x modulation, without tr)
    float4 *scatterTr;      // outcome of S2 by slot
    uint32_t *extendQueue;  // slots whose merged ray is traced
    uint32_t *scatterQueue; // slots with a pending S2
};

enum { VOL_EXTEND = 0, VOL_SHADOW = 1, VOL_SCATTER = 2 };

struct PlainBest { float t, U, V, den; uint32_t prim; bool found; };
struct Events3 { uint32_t count; float t0, t1, t2; int32_t m0, m1; };

__device__ __forceinline__ void events3Add(Events3 &ev, float t, int32_t medium) // eventAdd (volume.cuh) with three slots, no indexing
{
    if ((ev.count >= 1u && ev.t0 == t) || (ev.count >= 2u && ev.t1 == t) || (ev.count >= 3u && ev.t2 == t)) { return; }
    if (ev.count == 0u) { ev.t0 = t; ev.m0 = medium; }
    else if (ev.count == 1u) { ev.t1 = t; ev.m1 = medium; }
    else if (ev.count == 2u) { ev.t2 = t; }
    ev.count++;
}

// One triangle of the pending group under the rules of the volume rays (filteredTriangle of volume.cuh + the plain rule)
template <int MODE, bool COUNT>
__device__ __forceinline__ bool volumeTriangle(const DScene &s, TraversalState &st, PlainBest &pl, Events3 &ev, TraverseCounters &tc)
{
    const uint32_t bit = highestBit(st.tgroup.y);
    st.tgroup.y &= ~(1u << bit);
    const float4 *tri = s.bvh.triangles + (size_t)(st.tgroup.x + bit) * 3;
    const float4 a = loadNodeWord(tri), b = loadNodeWord(tri + 1), c = loadNodeWord(tri + 2);
    if (COUNT) { tc.tris++; }
    float T, U, V, absDen;
    if (!triangleTestRaw(a, b, c, st.ox, st.oy, st.oz, st.dx, st.dy, st.dz, st.tnear, st.hit.t, T, U, V, absDen)) { return false; }
    const float t = divIeee(T, absDen);
    const uint32_t prim = f2u(a.w);
    const int32_t medium = s.bvh.primEvent ? __ldg(s.bvh.primEvent + prim) : -1;
    if (MODE == VOL_EXTEND) {
        if (T <= absDen * pl.t) { // Scene::testIntersect's ray: every surface is a hit (traversalTriangle's rule against the plain distance)
            if (!(pl.found && t == pl.t && prim < pl.prim)) { pl.t = t; pl.U = U; pl.V = V; pl.den = absDen; pl.prim = prim; }
            pl.found = true;
        }
        if (medium >= 0) { return false; }
    } else if (medium >= 0) { events3Add(ev, t, medium); return false; }
    if (!(st.found && t == st.hit.t && prim < st.hit.prim)) { st.hit.t = t; st.hit.u = U; st.hit.v = V; st.hitDen = absDen; st.hit.prim = prim; }
    st.found = true;
    return true;
}

__device__ __forceinline__ V3 transmittanceBetween(const DScene &s, int32_t medium, V3 O, V3 D, float ta, float tb)
{
    return mediumTransmittance(s, medium, O + D * ta, O + D * tb);
}

// Persistent warps with lane refill (the loop of traverseKernel) over a queue of slots.
//  VOL_EXTEND  ray = the slot's (origin, direction); writes the plain closest hit to pb.hit and the filtered one to vb.probeHit
//  VOL_SHADOW  ray = slot origin + the NEE record's direction / distance, medium = the one the path was in when Ld was evaluated
//  VOL_SCATTER ray = the slot's scatter record
// 64 registers -> 8 resident CTAs, as the PathTracer's traversal kernel has them (72-80 registers / 6 CTAs without the bound: merged
// extend 55.5 -> 53.6 ms per 4 steps on cornell-medium)
#ifndef PTC_VOLUME_TRAVERSE_MIN_BLOCKS
#define PTC_VOLUME_TRAVERSE_MIN_BLOCKS 8
#endif
#define PTC_VOLUME_TRAVERSE_BOUNDS __launch_bounds__(128, PTC_VOLUME_TRAVERSE_MIN_BLOCKS)
template <int MODE, bool COUNT>
__global__ void PTC_VOLUME_TRAVERSE_BOUNDS volumeTraverseKernel(const __grid_constant__ DScene scene, PathBuffers pb, VolumeBuffers vb, const uint32_t *queue, const uint32_t *count,
                                                            uint32_t *cursor, unsigned long long *work)
{
    constexpr bool ANY = MODE != VOL_EXTEND;
    __shared__ uint2 fastStack[(PTC_FAST_STACK > 0 ? PTC_FAST_STACK : 1) * PTC_FAST_STRIDE];
    uint2 *const fast = fastStack + threadIdx.x;
    const uint32_t n = *count;
    const uint32_t lane = threadIdx.x & 31u;
    TraverseCounters tc = {0, 0};
    TraversalState st;
    PlainBest pl = {0.f, 0.f, 0.f, 1.f, PTC_MISS, false};
    Events3 ev = {0u, 0.f, 0.f, 0.f, -1, -1};
    int32_t medium = -1;
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
                    p = streamLoad(queue + item);
                    if (MODE == VOL_EXTEND) {
                        const Rec32 r = loadRec(pb.ray, p);
                        traversalInit(st, r.a.x, r.a.y, r.a.z, r.b.x, r.b.y, r.b.z, PTC_TNEAR, PTC_TFAR);
                        pl.t = PTC_TFAR; pl.prim = PTC_MISS; pl.found = false; pl.U = pl.V = 0.f; pl.den = 1.f;
                    } else if (MODE == VOL_SHADOW) { // DirectLightingHelper::directSampleLights' shadow ray, src/direct_lighting_helper.cpp:100-113
                        const float4 o = streamLoad(pb.ray + 2 * (size_t)p);
                        const Rec32 ne = loadRec(pb.nee, p);
                        traversalInit(st, o.x, o.y, o.z, ne.b.x, ne.b.y, ne.b.z, PTC_TNEAR, ne.b.w - 1e-3f);
                        medium = (int32_t)__float_as_uint(ne.a.w);
                        ev.count = 0u;
                    } else {                         // VolumeHelper::directSampleLights' shadow ray, src/volume_helper.cpp:30-44
                        const float4 a = streamLoad(vb.scatter + 3 * (size_t)p), b = streamLoad(vb.scatter + 3 * (size_t)p + 1);
                        traversalInit(st, a.x, a.y, a.z, b.x, b.y, b.z, PTC_TNEAR, a.w - 1e-3f);
                        medium = (int32_t)__float_as_uint(b.w);
                        ev.count = 0u;
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
            if (busy && hasNodes && st.tgroup.y == 0u) { traversalNode<COUNT>(scene.bvh, st, &tc, fast); }
            bool done = false;
            for (int round = 0; round < (ANY ? PTC_TRI_ROUNDS_ANY : PTC_TRI_ROUNDS); round++) {
                const bool pending = busy && !done && st.tgroup.y != 0u;
                if (__ballot_sync(0xFFFFFFFFu, pending) == 0u) { break; }
                if (pending && volumeTriangle<MODE, COUNT>(scene, st, pl, ev, tc) && ANY) { done = true; }
            }
            if (busy && (done || (st.tgroup.y == 0u && traversalPop(st, fast)))) {
                const V3 O = mk(st.ox, st.oy, st.oz), D = mk(st.dx, st.dy, st.dz);
                if (MODE == VOL_EXTEND) {
                    // plain rule: traversalSpheres<false>; filtered rule: the sphere loop of traverseFiltered<false> (container spheres are skipped)
                    if (pl.found) { pl.U = divIeee(pl.U, pl.den); pl.V = divIeee(pl.V, pl.den); }
                    if (st.found) { st.hit.u = divIeee(st.hit.u, st.hitDen); st.hit.v = divIeee(st.hit.v, st.hitDen); }
                    for (uint32_t i = 0; i < scene.bvh.nSpheres; i++) {
                        const float4 sp = loadNodeWord(scene.bvh.spheres + i);
                        float t, nx, ny, nz;
                        if (sphereTest(sp, st.ox, st.oy, st.oz, st.dx, st.dy, st.dz, st.tnear, pl.t, t, nx, ny, nz)) {
                            pl.t = t; pl.U = 0.f; pl.V = 0.f; pl.prim = PTC_SPHERE_FLAG | i; pl.found = true;
                        }
                        if (sphereTest(sp, st.ox, st.oy, st.oz, st.dx, st.dy, st.dz, st.tnear, st.hit.t, t, nx, ny, nz)) {
                            const int32_t m = scene.bvh.sphereEvent ? __ldg(scene.bvh.sphereEvent + i) : -1;
                            if (m < 0) { st.hit.t = t; st.hit.u = 0.f; st.hit.v = 0.f; st.hit.prim = PTC_SPHERE_FLAG | i; st.found = true; }
                        }
                    }
                    streamStore(pb.hit + p, make_float4(pl.t, pl.U, pl.V, __uint_as_float(pl.prim)));
                    streamStore(vb.probeHit + p, make_float4(st.hit.t, st.hit.u, st.hit.v, __uint_as_float(st.hit.prim)));
                } else {
                    if (!st.found) {
                        for (uint32_t i = 0; i < scene.bvh.nSpheres; i++) {
                            float t, nx, ny, nz;
                            if (sphereTest(loadNodeWord(scene.bvh.spheres + i), st.ox, st.oy, st.oz, st.dx, st.dy, st.dz, st.tnear, st.hit.t, t, nx, ny, nz)) {
                                const int32_t m = scene.bvh.sphereEvent ? __ldg(scene.bvh.sphereEvent + i) : -1;
                                if (m >= 0) { events3Add(ev, t, m); continue; }
                                st.found = true;
                                break;
                            }
                        }
                    }
                    V3 tr = mk(1.f, 1.f, 1.f);
                    if (!st.found) {
                        // eventsSort: only the order of the first two of at most two events is ever used
                        float ta = ev.t0, tb = ev.t1; int32_t ma = ev.m0;
                        if (ev.count == 2u && ta > tb) { ta = ev.t1; tb = ev.t0; ma = ev.m1; }
                        if (MODE == VOL_SHADOW) { // VolumeHelper::rayTransmission, src/volume_helper.cpp:72-123
                            const int32_t m = medium >= 0 ? medium : ma;
                            if (ev.count == 1u) { tr = transmittanceBetween(scene, m, O, D, 0.f, ta); }
                            else if (ev.count == 2u) { tr = transmittanceBetween(scene, m, O, D, ta, tb); }
                        } else {                  // src/volume_helper.cpp:46-66: zero unless one or two events
                            tr = mk(0.f, 0.f, 0.f);
                            if (ev.count == 1u) { tr = transmittanceBetween(scene, medium, O, D, 0.f, ta); }
                            else if (ev.count == 2u) { tr = transmittanceBetween(scene, medium, O, D, ta, tb); }
                        }
                    }
                    streamStore((MODE == VOL_SHADOW ? vb.shadowTr : vb.scatterTr) + p, make_float4(tr.x, tr.y, tr.z, st.found ? 1.f : 0.f));
                }
                busy = false;
            }
            active = __ballot_sync(0xFFFFFFFFu, busy);
            if (active == 0u || (more && __popc(active) <= PTC_REFILL_BELOW)) { break; }
        }
    }
    if (COUNT) { flushCounters(tc, work); }
}

// Everything of VolumePathTracer::L that waits for the rays traced at bounce k >= 1 (they left vertex k): the in-scattered light of
// the segment that arrived at vertex k (:54-55), Ld of vertex k (:36 -> DirectLightingHelper::Ld), and whether the path goes on (:52-53).
#ifndef PTC_VOLUME_LOGIC_MIN_BLOCKS
#define PTC_VOLUME_LOGIC_MIN_BLOCKS 3
#endif
__global__ void __launch_bounds__(256, PTC_VOLUME_LOGIC_MIN_BLOCKS) volumeLogicKernel(const __grid_constant__ DScene scene, PathBuffers pb, VolumeBuffers vb, WaveParams wp,
                                                                                BounceCounters *bc, uint32_t classMask)
{
    const uint32_t n = bc->slotCount;
    const uint32_t lane = threadIdx.x & 31u;
    for (uint32_t base = (blockIdx.x * blockDim.x + threadIdx.x) & ~31u; base < n; base += gridDim.x * blockDim.x) {
        const uint32_t p = base + lane;
        int cls = -1;
        if (p < n) {
            const float4 res4 = streamLoad(pb.result + p);
            const uint32_t flags = __float_as_uint(res4.w);
            const Rec32 mt = loadRec(pb.modThr, p);
            V3 result = mk(res4.x, res4.y, res4.z);
            if (flags & FLAG_SCATTER) { // result += Ls * modulation
                const float4 tr = streamLoad(vb.scatterTr + p);
                if (tr.w == 0.f) {
                    const float4 c = streamLoad(vb.scatter + 3 * (size_t)p + 2);
                    result = result + mk(c.x, c.y, c.z) * mk(tr.x, tr.y, tr.z);
                }
            }
            float4 hc = make_float4(0.f, 0.f, 0.f, __uint_as_float(PTC_MISS));
            if (flags & FLAG_TRACED) { hc = streamLoad(pb.hit + p); }
            Rec32 ray; ray.a = ray.b = make_float4(0.f, 0.f, 0.f, 0.f);
            bool haveRay = false;
            if (flags & FLAG_DIRECT) {
                V3 Ld = mk(0.f, 0.f, 0.f);
                if (flags & FLAG_NEE) {
                    const float4 tr = streamLoad(vb.shadowTr + p);
                    if (tr.w == 0.f) {
                        const float4 ne = streamLoad(pb.nee + 2 * (size_t)p);
                        Ld = Ld + mk(ne.x, ne.y, ne.z) * mk(tr.x, tr.y, tr.z);
                    }
                }
                // directSampleBSDF, src/direct_lighting_helper.cpp:139-187: the probe hit (containers skipped); emitter hits and
                // environment misses only, either side of the emitter, no transmittance
                const float4 hp = scene.hasFilter ? streamLoad(vb.probeHit + p) : hc;
                const uint32_t prim = __float_as_uint(hp.w);
                const bool isHit = prim != PTC_MISS;
                uint32_t surface = 0;
                if (isHit) { surface = (prim & PTC_SPHERE_FLAG) ? __ldg(scene.sphereClass + (prim & ~PTC_SPHERE_FLAG)) : __ldg(scene.primClass + prim); }
                if (!isHit || (surface & 8u)) {
                    ray = loadRec(pb.ray, p); haveRay = true;
                    const V3 O = mk(ray.a.x, ray.a.y, ray.a.z), D = mk(ray.b.x, ray.b.y, ray.b.z);
                    Isect bi;
                    if (isHit) { RayHit hit; hit.t = hp.x; hit.u = hp.y; hit.v = hp.z; hit.prim = prim; makeIsect(scene, O, D, hit, bi); }
                    Ld = Ld + directBsdf(scene, O, mt.b.w, D, mt.a.w, mk(mt.b.x, mt.b.y, mt.b.z), (flags & FLAG_DELTA) != 0, isHit, &bi, false);
                }
                result = result + Ld * mk(mt.a.x, mt.a.y, mt.a.z);
            }
            const uint32_t primC = __float_as_uint(hc.w);
            const bool alive = !(flags & FLAG_LAST) && primC != PTC_MISS;
            if (alive) {
                if (flags & (FLAG_DIRECT | FLAG_SCATTER)) { streamStore(pb.result + p, make_float4(result.x, result.y, result.z, res4.w)); }
                cls = (int)(((primC & PTC_SPHERE_FLAG) ? __ldg(scene.sphereClass + (primC & ~PTC_SPHERE_FLAG)) : __ldg(scene.primClass + primC)) & 7u);
            } else {
                const uint32_t origin = haveRay ? __float_as_uint(ray.a.w) : __float_as_uint(streamLoad(&pb.ray[2 * (size_t)p].w));
                finishPath(pb, origin, flags, result);
            }
        }
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

// Vertex b = k + 1 of every path whose continuation ray k hit a surface of material class TYPE: the rest of loop iteration k of
// VolumePathTracer::L (:52-61: Intersection, modulation, scatter, transmittance, black test) and the head of iteration b (:33-50:
// BSDF sample, Ld set-up, medium change).  k = 0: the camera hit (:21-31 are the same statements with modulation = 1).
// Occupancy sweep on cornell-medium (profiles/r02_sweep_volume_wavefront.txt, Msamples/s): 8 CTAs of 128 per SM 333, 6 CTAs 342-345,
// 5 CTAs 377, 4 CTAs 386-394, 3 CTAs 385, 2 CTAs 386 -- unlike the PathTracer's material kernels (best at 8 CTAs with ~170 B of
// spills) this one carries the scatter record and the medium next to the BSDF state, and its spills cost more than the occupancy gives
#ifndef PTC_VOLUME_MATERIAL_MIN_BLOCKS
#define PTC_VOLUME_MATERIAL_MIN_BLOCKS 4
#endif
template <int TYPE>
__global__ void __launch_bounds__(128, PTC_VOLUME_MATERIAL_MIN_BLOCKS) volumeMaterialKernel(const __grid_constant__ DScene scene, PathBuffers pb, VolumeBuffers vb, WaveParams wp,
                                                                                             BounceCounters *bc, BounceCounters *next)
{
    const uint32_t n = bc->classCount[TYPE];
    const uint32_t *queue = pb.classQueue[TYPE];
    for (uint32_t base = (blockIdx.x * blockDim.x + threadIdx.x) & ~31u; base < n; base += gridDim.x * blockDim.x) {
        const uint32_t item = base + (threadIdx.x & 31u);
        bool push = false, pushShadow = false, pushScatter = false, pushExtend = false;
        float4 nO = make_float4(0.f, 0.f, 0.f, 0.f), nD = nO, nMod = nO, nThr = nO, nRes = nO, nNee = nO, nSh = nO, sA = nO, sB = nO, sC = nO;
        if (item < n) {
            const uint32_t p = streamLoad(queue + item);
            const Rec32 ray = loadRec(pb.ray, p);
            const float4 h4 = streamLoad(pb.hit + p), res4 = streamLoad(pb.result + p);
            const uint32_t origin = __float_as_uint(ray.a.w);
            const uint32_t flags = __float_as_uint(res4.w);
            const int k = (int)(flags & FLAG_BOUNCE_MASK);
            const int b = k + 1;
            const V3 O = mk(ray.a.x, ray.a.y, ray.a.z), D = mk(ray.b.x, ray.b.y, ray.b.z);
            RayHit hit; hit.t = h4.x; hit.u = h4.y; hit.v = h4.z; hit.prim = __float_as_uint(h4.w);
            Isect bi;
            makeIsect(scene, O, D, hit, bi);
            const DMaterial &m = scene.materials[bi.material];
            Rng rng;
            uint32_t oq, os;
            slotToPixelSample(origin, wp, oq, os);
            rng.initPhilox(wp.seed, wavePixel(oq, wp, (uint32_t)scene.width, (uint32_t)scene.height), wp.firstSample + os);
            rng.beginVertex((uint32_t)b);
            V3 modulation = mk(1.f, 1.f, 1.f);
            int32_t medium = -1;
            bool dead = false;
            if (k > 0) {
                const Rec32 mt = loadRec(pb.modThr, p);
                modulation = advanceModulation(mt.a, mt.b);
                medium = (int32_t)__float_as_uint(ray.b.w);
                if (medium >= 0) {
                    // VolumePathTracer::scatter -> HomogeneousMedium::integrate -> VolumeHelper::directSampleLights
                    const float sigmaT = __ldg(scene.media + 2 * medium).x;
                    const V3 travel = bi.point - O;
                    const float distance = length(travel);
                    const float xi = rng.next();
                    const float sampleT = -logHost(1 - xi) / sigmaT;
                    if (sampleT < distance && scene.nLights != 0u) {
                        const V3 samplePoint = O + normalize(travel) * sampleT;
                        SurfSample ls;
                        const DLight *light = sampleDirectLights(scene, samplePoint, rng, ls);
                        const V3 sd = ls.point - samplePoint;
                        const V3 wi = normalize(sd);
                        if (!(dot(ls.normal, wi) >= 0.f)) {
                            const float dist = length(sd);
                            const float pdf = solidAnglePdf(ls, samplePoint);
                            const V3 lwo = -normalize(sd);
                            const V3 Le = __ldg(&light->kind) == 2 ? envRadiance(scene, -lwo) : mk(__ldg(&light->emit[0]), __ldg(&light->emit[1]), __ldg(&light->emit[2]));
                            const V3 Ls = ((Le * 1.f) / (float)(4.f * PTC_PI_D)) / pdf;
                            const V3 c = Ls * modulation;
                            sA = make_float4(samplePoint.x, samplePoint.y, samplePoint.z, dist);
                            sB = make_float4(wi.x, wi.y, wi.z, __uint_as_float((uint32_t)medium));
                            sC = make_float4(c.x, c.y, c.z, 0.f);
                            pushScatter = true;
                        }
                    }
                    modulation = modulation * mediumTransmittance(scene, medium, O, bi.point);
                }
                if (isBlack(modulation)) { dead = true; }
            }
            uint32_t nf = (uint32_t)b | (flags & FLAG_BASE) | (pushScatter ? FLAG_SCATTER : 0u);
            if (!dead) {
                BsdfSample bs;
                bsdfSample<TYPE>(m, bi, rng, bs);
                // DirectLightingHelper::Ld returns 0 for containers and emitters before it traces anything (:47-52)
                const bool wantDirect = checkCounts(wp.startBounce, wp.lastBounce, b) && TYPE != PTC_PASSTHROUGH && !__ldg(&m.emitter);
                if (wantDirect) {
                    V3 contribution, sd; float maxT;
                    if (directLightsSetup<TYPE>(scene, m, bi, bs, rng, contribution, sd, maxT) && !isBlack(contribution)) {
                        nNee = make_float4(contribution.x, contribution.y, contribution.z, __uint_as_float((uint32_t)medium));
                        nSh = make_float4(sd.x, sd.y, sd.z, maxT);
                        pushShadow = true;
                    }
                }
                const bool wantNext = !checkDone(wp.lastBounce, b + 1);
                if (wantNext && dot(bi.wo, bs.wi) < 0.f) { // refraction: the medium changes (:42-50)
                    medium = dot(bi.n, bs.wi) < 0.f ? internalMedium(scene, bi.prim) : -1;
                }
                pushExtend = wantDirect || wantNext;
                nO = make_float4(bi.point.x, bi.point.y, bi.point.z, ray.a.w);
                nD = make_float4(bs.wi.x, bs.wi.y, bs.wi.z, __uint_as_float((uint32_t)medium));
                nMod = make_float4(modulation.x, modulation.y, modulation.z, bs.pdf);
                nThr = make_float4(bs.thr.x, bs.thr.y, bs.thr.z, fabsf(dot(bi.ns, bs.wi)));
                nf |= (bs.delta ? FLAG_DELTA : 0u) | (wantDirect ? FLAG_DIRECT : 0u) | (pushShadow ? FLAG_NEE : 0u) | (wantNext ? 0u : FLAG_LAST) | (pushExtend ? FLAG_TRACED : 0u);
            } else {
                nO = make_float4(bi.point.x, bi.point.y, bi.point.z, ray.a.w);
                nf |= FLAG_LAST;
            }
            push = pushExtend || pushScatter;
            nRes = make_float4(res4.x, res4.y, res4.z, __uint_as_float(nf));
            if (!push) { finishPath(pb, origin, flags, mk(res4.x, res4.y, res4.z)); }
        }
        const uint32_t e = warpAppend(&next->slotCount, push);
        if (push) {
            storeRec(pb.nRay, e, nO, nD);
            storeRec(pb.nModThr, e, nMod, nThr);
            streamStore(pb.nResult + e, nRes);
            if (pushShadow) { storeRec(pb.nee, e, nNee, nSh); }
            if (pushScatter) { streamStore(vb.scatter + 3 * (size_t)e, sA); streamStore(vb.scatter + 3 * (size_t)e + 1, sB); streamStore(vb.scatter + 3 * (size_t)e + 2, sC); }
        }
        const uint32_t x = warpAppend(&next->extendCount, pushExtend);
        if (pushExtend) { streamStore(vb.extendQueue + x, e); }
        const uint32_t sh = warpAppend(&next->shadowCount, pushShadow);
        if (pushShadow) { streamStore(pb.shadowQueue + sh, e); }
        const uint32_t sc = warpAppend(&next->scatterCount, pushScatter);
        if (pushScatter) { streamStore(vb.scatterQueue + sc, e); }
    }
}

