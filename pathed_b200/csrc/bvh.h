// Host-side BVH builder: binned-SAH binary tree collapsed into an 8-wide BVH whose nodes are stored in the
// compressed 80-byte layout (quantised child boxes) the sm_100a traversal kernels read.
// Replaces Embree's builder (ext/embree/kernels/bvh/bvh_builder_sah.cpp, builders/heuristic_binning.h) behind
// rtcCommitScene (src/scene.cpp:39).
#pragma once

#include <cuda_runtime.h>

#include <cstdint>
#include <vector>

namespace ptc {

// 80-byte compressed wide node (5 x 16 B).  Child boxes are 8-bit offsets from `origin` on a per-axis
// power-of-two grid: lo = origin + qlo * 2^e, hi = origin + qhi * 2^e (rounded outwards, so conservative).
struct alignas(16) WideNode {
    float origin[3];
    uint8_t exponent[3]; // biased fp32 exponents of the grid scale
    uint8_t imask;       // bit i: slot i is an inner node
    uint32_t childBase;  // index of the first inner child (children are contiguous, in slot order)
    uint32_t triBase;    // index of the first leaf triangle referenced by this node
    uint8_t meta[8];     // inner: 0b001xxxxx with xxxxx = 24 + slot; leaf: unary triangle count << 5 | triangle offset; empty: 0
    uint8_t qlox[8], qloy[8], qloz[8];
    uint8_t qhix[8], qhiy[8], qhiz[8];
};
static_assert(sizeof(WideNode) == 80, "WideNode must be 80 bytes");

// 48-byte leaf triangle in Embree's Triangle4 form (ext/embree/kernels/geometry/triangle.h:53-54):
// v0, e1 = v0 - v1, e2 = v2 - v0; w of the first float4 carries the global primitive index.
struct alignas(16) LeafTriangle {
    float v0[3];
    uint32_t prim;
    float e1[3];
    uint32_t pad0;
    float e2[3];
    uint32_t pad1;
};
static_assert(sizeof(LeafTriangle) == 48, "LeafTriangle must be 48 bytes");

struct WideBVH {
    std::vector<WideNode> nodes;         // nodes[0] is the root
    std::vector<LeafTriangle> triangles; // in leaf order
    std::vector<float> placements;       // instanced scenes: 24 floats per flattened placement (traverse.cuh: BvhView::placements)
    uint32_t maxDepth = 0;
};

// positions: float4 per vertex (xyz used); indices: 4 uint32 per primitive (i0, i1, i2, material)
void buildWideBVH(const float *positions4, const uint32_t *indices4, uint32_t nPrims, WideBVH &out);

// Device builder (bvh_build_gpu.cu; SURVEY §8(f) N2): Morton sort -> PLOC clustering -> the same SAH-optimal 8-wide collapse and
// node encoding, all in kernels on `stream`.  Inputs and outputs are device pointers; `nodes` / `triangles` are cudaMalloc'ed
// and owned by the caller.  Throws std::runtime_error on CUDA errors.
struct DeviceWideBVH {
    float4 *nodes = nullptr;     // 5 float4 per node
    float4 *triangles = nullptr; // 3 float4 per triangle
    uint32_t nNodes = 0, nTriangles = 0, maxDepth = 0, plocIterations = 0;
    float buildMs[4] = {0, 0, 0, 0}; // boxes + sort, clustering, emission, total (host clock around synchronised phases)
};
// workspaceOut (optional): the build's working set (one allocation, ~480 B per primitive) is handed to the caller instead of being
// released -- cudaFree of a few hundred MB that kernels have just written was measured at 37 ms, five times the build itself; the
// caller frees it when nothing waits for it (ptc_destroy).
void buildWideBVHDevice(const float4 *dPositions, const uint4 *dPrims, uint32_t nPrims, cudaStream_t stream, DeviceWideBVH &out, void **workspaceOut = nullptr);
// The device builder's per-element code run serially on the host (ptc_bvh_selfcheck_builder: CPU tests of the algorithm).
// Never used by ptc_commit.
void buildWideBVHEmulated(const float *positions4, const uint32_t *indices4, uint32_t nPrims, WideBVH &out);
// SAH cost of a wide BVH: sum over nodes of area(node) * 1.0 + sum over leaf slots of area(slot box) * 0.4 * triangles, divided
// by the root area (the collapse's own cost model)
double wideBVHCost(const WideBVH &bvh);

// Scalar reference traversal of the wide BVH (same node/triangle decoding as the kernels) that counts work:
// SURVEY §8(d) defines the algorithmic bytes per ray from these counts.  Returns true on a hit.
struct TraversalCounts { uint64_t innerVisits = 0, triangleTests = 0; };
bool traverseReference(const WideBVH &bvh, const float origin[3], const float direction[3], float tnear, float tfar,
                       bool anyHit, float *tOut, uint32_t *primOut, TraversalCounts *counts);

} // namespace ptc
