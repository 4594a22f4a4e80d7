// Device BVH builder (SURVEY §8(f) N2): replaces the host SAH builder behind ptc_commit / rtcCommitScene (src/scene.cpp:39,
// Embree's ext/embree/kernels/bvh/bvh_builder_sah.cpp) with a build that runs entirely on the B200:
//
//   1. primitive boxes, centroid bounds                        (one pass, block reduce + ordered-int atomics)
//   2. 63-bit Morton codes of the centroids, radix sort        (cub::DeviceRadixSort)
//   3. PLOC (parallel locally-ordered clustering, Meister & Bittner 2018): every cluster looks for the neighbour within
//      +-PLOC_RADIUS positions of the Morton order that gives the smallest merged surface area; mutual nearest neighbours
//      merge; the cluster list is compacted with a prefix sum; repeat until PLOC_TOP_CLUSTERS clusters are left.  The top of the
//      tree (visited by every ray) is then built over those clusters top-down with a binned SAH.  The SAH-optimal 8-wide
//      collapse table C(n, 1..7) of Ylitie et al. 2017 is computed at the moment a node is created (its children are final).
//   4. level-by-level emission of the compressed 80-byte nodes: children chosen from the collapse table, octant-ordered slot
//      assignment, outward quantisation, leaf triangles in Embree's (v0, e1, e2) form.  Node and triangle indices come from
//      prefix sums, so the layout is deterministic (breadth first, children of a node contiguous).
//
// Every per-element step is a functor over an index that compiles for the device and for the host.  The kernels run the
// functors one element per thread; ptc_bvh_selfcheck_builder runs the very same functors in a serial loop so that the CPU test
// suite can check the algorithm (tree validity, exact hits, SAH quality) without a GPU.  ptc_commit only ever uses the kernels.
#include "bvh.h"
#include "traverse.cuh"

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <stdexcept>
#include <string>
#include <vector>

namespace ptc {

namespace {

#ifndef PLOC_RADIUS
#define PLOC_RADIUS 16
#endif
#ifndef PLOC_TOP_CLUSTERS
#define PLOC_TOP_CLUSTERS 512
#endif
constexpr uint32_t kInvalid = 0xFFFFFFFFu;
#ifndef PTC_COST_PRIM
#define PTC_COST_PRIM 0.4f
#endif
constexpr float kCostNode = 1.0f, kCostPrim = PTC_COST_PRIM; // same constants as the host builder's collapse
constexpr uint32_t kMaxLeaf = 3;
constexpr float kInf = 3.0e38f;

// ---- collapse table entry of one binary node (32 B) ------------------------------------------------------------------
// info: bits 0..3 primitive count (saturating at 15), bit 4 "a wide-BVH root made from this node is a leaf",
//       bits 8..28 the seven 3-bit split decisions k of C_distribute(n, j), j = 2..8
struct NodeDP {
    float c[7];
    uint32_t info;
};
PTC_HD uint32_t dpPrimCount(uint32_t info) { return info & 15u; }
PTC_HD bool dpRootIsLeaf(uint32_t info) { return (info >> 4) & 1u; }
PTC_HD uint32_t dpSplit(uint32_t info, int j) { return (info >> (8 + 3 * (j - 2))) & 7u; }

PTC_HD float halfArea(float lx, float ly, float lz, float hx, float hy, float hz)
{
    const float x = hx - lx, y = hy - ly, z = hz - lz;
    return x < 0.f ? 0.f : x * y + y * z + z * x;
}

// order-preserving float <-> uint map for atomicMin / atomicMax on floats
PTC_HD uint32_t orderedBits(float f) { const uint32_t u = f2u(f); return (u & 0x80000000u) ? ~u : (u | 0x80000000u); }
PTC_HD float orderedFloat(uint32_t u) { return u2f((u & 0x80000000u) ? (u & 0x7FFFFFFFu) : ~u); }

PTC_HD uint64_t spread21(uint32_t v) // 21 bits -> every third bit of 63
{
    uint64_t x = v & 0x1FFFFFu;
    x = (x | (x << 32)) & 0x1F00000000FFFFull;
    x = (x | (x << 16)) & 0x1F0000FF0000FFull;
    x = (x | (x << 8)) & 0x100F00F00F00F00Full;
    x = (x | (x << 4)) & 0x10C30C30C30C30C3ull;
    x = (x | (x << 2)) & 0x1249249249249249ull;
    return x;
}

// All arrays of one build.  The same struct describes device memory (kernels) and host memory (emulation).
struct BuildArrays {
    const float4 *positions; // xyz per vertex
    const uint4 *prims;      // i0, i1, i2, material
    uint32_t nPrims;
    float4 *primLo, *primHi; // per primitive box
    uint32_t *bounds;        // 6 ordered-int words: centroid lo xyz, hi xyz
    uint64_t *keys[2];
    uint32_t *order[2];      // primitive index per sorted position
    // binary tree: nodes [0, nPrims) are the leaves in Morton order, inner nodes follow in creation order
    float4 *nodeLo, *nodeHi; // w: left child / right child (leaf: primitive index / kInvalid)
    NodeDP *dp;
    // PLOC cluster list, double buffered; w of lo = node index
    float4 *clusterLo[2], *clusterHi[2];
    uint32_t *nearest;
    uint64_t *scanIn, *scanOut; // packed counters: high word / low word scanned together
    // top-level SAH pass: one segment (first cluster, cluster count, node index) per inner node, level after level; per segment and
    // axis the best split (cost, bin, lower centroid bound, bins per unit length); state = {segments appended so far, next free node index}
    uint4 *topSegments;
    float4 *topAxis;
    uint32_t *topMid, *topState;
    // emission
    uint32_t *items[2];     // binary node of every wide node of the current / next level
    uint32_t *itemChildren; // 8 per item, slot order, kInvalid = empty
    WideNode *wideNodes;
    LeafTriangle *leafTriangles;
    float costPrim; // cost of a triangle test relative to a node visit in the collapse (runBuild)
};

// ---- step 1: boxes ---------------------------------------------------------------------------------------------------
struct PrimBoxOp {
    BuildArrays a;
    PTC_HD void operator()(uint32_t p) const
    {
        const uint4 ix = a.prims[p];
        const float4 v0 = a.positions[ix.x], v1 = a.positions[ix.y], v2 = a.positions[ix.z];
        a.primLo[p] = make_float4(fminf(v0.x, fminf(v1.x, v2.x)), fminf(v0.y, fminf(v1.y, v2.y)), fminf(v0.z, fminf(v1.z, v2.z)), 0.f);
        a.primHi[p] = make_float4(fmaxf(v0.x, fmaxf(v1.x, v2.x)), fmaxf(v0.y, fmaxf(v1.y, v2.y)), fmaxf(v0.z, fmaxf(v1.z, v2.z)), 0.f);
    }
};

PTC_HD void centroidOf(const float4 lo, const float4 hi, float c[3])
{
    c[0] = 0.5f * (lo.x + hi.x); c[1] = 0.5f * (lo.y + hi.y); c[2] = 0.5f * (lo.z + hi.z);
}

// ---- step 2: Morton codes ----------------------------------------------------------------------------------------------
struct MortonOp {
    BuildArrays a;
    PTC_HD void operator()(uint32_t p) const
    {
        float c[3];
        centroidOf(a.primLo[p], a.primHi[p], c);
        uint64_t key = 0;
        for (int axis = 0; axis < 3; axis++) {
            const float lo = orderedFloat(a.bounds[axis]), hi = orderedFloat(a.bounds[3 + axis]);
            const float extent = hi - lo;
            float f = extent > 0.f ? (c[axis] - lo) / extent : 0.f;
            f = fminf(fmaxf(f, 0.f), 1.f);
            uint32_t q = (uint32_t)(f * 2097152.f);
            if (q > 2097151u) { q = 2097151u; }
            key |= spread21(q) << (2 - axis);
        }
        a.keys[0][p] = key;
        a.order[0][p] = p;
    }
};

// leaves of the binary tree = sorted primitives; they are also the first cluster list
struct LeafOp {
    BuildArrays a;
    const uint32_t *sorted;
    PTC_HD void operator()(uint32_t i) const
    {
        const uint32_t p = sorted[i];
        const float4 lo = a.primLo[p], hi = a.primHi[p];
        a.nodeLo[i] = make_float4(lo.x, lo.y, lo.z, u2f(p));
        a.nodeHi[i] = make_float4(hi.x, hi.y, hi.z, u2f(kInvalid));
        NodeDP d;
        const float cost = halfArea(lo.x, lo.y, lo.z, hi.x, hi.y, hi.z) * a.costPrim;
        for (int k = 0; k < 7; k++) { d.c[k] = cost; }
        d.info = 1u | (1u << 4);
        a.dp[i] = d;
        a.clusterLo[0][i] = make_float4(lo.x, lo.y, lo.z, u2f(i));
        a.clusterHi[0][i] = hi;
    }
};

// ---- step 3: PLOC ------------------------------------------------------------------------------------------------------
struct NearestOp {
    BuildArrays a;
    int buffer;
    uint32_t nClusters, radius;
    PTC_HD void operator()(uint32_t i) const
    {
        const float4 *lo = a.clusterLo[buffer], *hi = a.clusterHi[buffer];
        const float4 l = lo[i], h = hi[i];
        const uint32_t first = i > radius ? i - radius : 0u;
        const uint32_t last = i + radius < nClusters - 1u ? i + radius : nClusters - 1u;
        float best = kInf; uint32_t bestJ = kInvalid;
        for (uint32_t j = first; j <= last; j++) {
            if (j == i) { continue; }
            const float4 l2 = lo[j], h2 = hi[j];
            // symmetric in (i, j): min / max commute, so both sides of a pair see the same distance
            const float d = halfArea(fminf(l.x, l2.x), fminf(l.y, l2.y), fminf(l.z, l2.z), fmaxf(h.x, h2.x), fmaxf(h.y, h2.y), fmaxf(h.z, h2.z));
            if (d < best) { best = d; bestJ = j; } // ties: the lowest index wins, so the globally closest pair is always mutual
        }
        a.nearest[i] = bestJ;
    }
};

// per cluster: high word = 1 if this cluster creates a node (the lower index of a mutual pair), low word = 1 if it survives
struct MergeFlagOp {
    BuildArrays a;
    PTC_HD void operator()(uint32_t i) const
    {
        const uint32_t j = a.nearest[i];
        const bool mutual = j != kInvalid && a.nearest[j] == i;
        const uint64_t creates = (mutual && i < j) ? 1u : 0u, survives = (mutual && i > j) ? 0u : 1u;
        a.scanIn[i] = (creates << 32) | survives;
    }
};

// collapse table of a new inner node from its children's tables (Ylitie et al. 2017, section 3.1; the host builder's recurrences)
PTC_HD NodeDP combineDP(const NodeDP &l, const NodeDP &r, float area, float costPrim)
{
    NodeDP d;
    float distribute[9];
    uint32_t splits = 0;
    for (int j = 2; j <= 8; j++) {
        float best = kInf; int bestK = 1;
        for (int k = 1; k < j; k++) {
            if (k > 7 || j - k > 7) { continue; }
            const float v = l.c[k - 1] + r.c[j - k - 1];
            if (v < best) { best = v; bestK = k; }
        }
        distribute[j] = best;
        splits |= (uint32_t)bestK << (3 * (j - 2));
    }
    const uint32_t sum = dpPrimCount(l.info) + dpPrimCount(r.info);
    const uint32_t count = sum > 15u ? 15u : sum;
    const float internal = distribute[8] + area * kCostNode;
    const float leaf = count <= kMaxLeaf ? area * (float)count * costPrim : kInf;
    const bool rootIsLeaf = leaf <= internal;
    d.c[0] = fminf(leaf, internal);
    for (int i = 2; i <= 7; i++) { d.c[i - 1] = fminf(distribute[i], d.c[i - 2]); }
    d.info = count | (rootIsLeaf ? 16u : 0u) | (splits << 8);
    return d;
}

struct MergeOp {
    BuildArrays a;
    int buffer;
    uint32_t nClusters, firstNewNode;
    PTC_HD void operator()(uint32_t i) const
    {
        const uint32_t j = a.nearest[i];
        const bool mutual = j != kInvalid && a.nearest[j] == i;
        if (mutual && i > j) { return; } // absorbed by cluster j
        const uint64_t prefix = a.scanOut[i];
        const uint32_t slot = (uint32_t)(prefix & 0xFFFFFFFFu);
        float4 lo = a.clusterLo[buffer][i], hi = a.clusterHi[buffer][i];
        if (mutual) {
            const uint32_t node = firstNewNode + (uint32_t)(prefix >> 32);
            const float4 lo2 = a.clusterLo[buffer][j], hi2 = a.clusterHi[buffer][j];
            const uint32_t left = f2u(lo.w), right = f2u(lo2.w);
            lo = make_float4(fminf(lo.x, lo2.x), fminf(lo.y, lo2.y), fminf(lo.z, lo2.z), 0.f);
            hi = make_float4(fmaxf(hi.x, hi2.x), fmaxf(hi.y, hi2.y), fmaxf(hi.z, hi2.z), 0.f);
            a.nodeLo[node] = make_float4(lo.x, lo.y, lo.z, u2f(left));
            a.nodeHi[node] = make_float4(hi.x, hi.y, hi.z, u2f(right));
            a.dp[node] = combineDP(a.dp[left], a.dp[right], halfArea(lo.x, lo.y, lo.z, hi.x, hi.y, hi.z), a.costPrim);
            lo.w = u2f(node);
        }
        a.clusterLo[buffer ^ 1][slot] = lo;
        a.clusterHi[buffer ^ 1][slot] = hi;
    }
};

// ---- step 3b: top of the tree ----------------------------------------------------------------------------------------------
// Agglomerative clustering decides well near the leaves but the last few hundred merges (the top of the tree, visited by every
// ray) are taken between whatever clusters happen to be left.  So PLOC stops at `count` clusters and the top is built over them
// top-down with a 16-bin SAH over all three axes (the host builder's split rule), level by level: every inner node of the top is a
// segment [first, first + count) of the cluster list.  Per level
//   TopAxisOp   one thread per (segment, axis): centroid bounds, binning, sweep -> the best split on that axis
//   TopSplitOp  one thread per segment: picks the axis, partitions the segment's clusters in place
//   TopEmitOp   one thread: numbers the children (root = last node index, the others downwards in creation order, so that a level's
//               nodes are consecutive), links them, appends the segments of the next level
// and once the segments have run out TopFinishOp, one thread per node, deepest level first: box and collapse table from the children.
// The serial chain is one pass over the largest segment per level (512 + 256 + ... clusters) instead of one thread walking every
// segment of every level.
constexpr int kTopBins = 16;

struct TopAxisOp {
    BuildArrays a;
    int buffer;
    uint32_t segBase;
    PTC_HD void operator()(uint32_t i) const
    {
        const uint4 seg = a.topSegments[segBase + i / 3u];
        const int axis = (int)(i % 3u);
        const float4 *lo = a.clusterLo[buffer], *hi = a.clusterHi[buffer];
        const uint32_t first = seg.x, end = seg.x + seg.y;
        float cl = kInf, ch = -kInf;
        for (uint32_t c = first; c < end; c++) {
            const float4 l = lo[c], h = hi[c];
            const float v = 0.5f * (axis == 0 ? l.x + h.x : (axis == 1 ? l.y + h.y : l.z + h.z));
            cl = fminf(cl, v); ch = fmaxf(ch, v);
        }
        float bestCost = kInf; int bestBin = -1;
        const float extent = ch - cl;
        const float scale = extent > 0.f ? (float)kTopBins / extent : 0.f;
        if (extent > 0.f) {
            float bl[kTopBins][3], bh[kTopBins][3]; uint32_t bn[kTopBins];
            for (int b = 0; b < kTopBins; b++) { bn[b] = 0; for (int k = 0; k < 3; k++) { bl[b][k] = kInf; bh[b][k] = -kInf; } }
            for (uint32_t c = first; c < end; c++) {
                const float4 l = lo[c], h = hi[c];
                const float v = 0.5f * (axis == 0 ? l.x + h.x : (axis == 1 ? l.y + h.y : l.z + h.z));
                int b = (int)((v - cl) * scale);
                b = b < 0 ? 0 : (b >= kTopBins ? kTopBins - 1 : b);
                bn[b]++;
                bl[b][0] = fminf(bl[b][0], l.x); bl[b][1] = fminf(bl[b][1], l.y); bl[b][2] = fminf(bl[b][2], l.z);
                bh[b][0] = fmaxf(bh[b][0], h.x); bh[b][1] = fmaxf(bh[b][1], h.y); bh[b][2] = fmaxf(bh[b][2], h.z);
            }
            float rightArea[kTopBins]; uint32_t rightCount[kTopBins];
            float al[3] = {kInf, kInf, kInf}, ah[3] = {-kInf, -kInf, -kInf}; uint32_t m = 0;
            for (int b = kTopBins - 1; b > 0; b--) {
                for (int k = 0; k < 3; k++) { al[k] = fminf(al[k], bl[b][k]); ah[k] = fmaxf(ah[k], bh[b][k]); }
                m += bn[b]; rightArea[b] = halfArea(al[0], al[1], al[2], ah[0], ah[1], ah[2]); rightCount[b] = m;
            }
            for (int k = 0; k < 3; k++) { al[k] = kInf; ah[k] = -kInf; }
            m = 0;
            for (int b = 0; b < kTopBins - 1; b++) {
                for (int k = 0; k < 3; k++) { al[k] = fminf(al[k], bl[b][k]); ah[k] = fmaxf(ah[k], bh[b][k]); }
                m += bn[b];
                if (m == 0 || rightCount[b + 1] == 0) { continue; }
                // clusters are not unit cost: weigh a side by its count (every cluster holds a similar number of primitives)
                const float cost = halfArea(al[0], al[1], al[2], ah[0], ah[1], ah[2]) * (float)m + rightArea[b + 1] * (float)rightCount[b + 1];
                if (cost < bestCost) { bestCost = cost; bestBin = b; }
            }
        }
        a.topAxis[3u * (segBase + i / 3u) + (uint32_t)axis] = make_float4(bestCost, u2f((uint32_t)bestBin), cl, scale);
    }
};

struct TopSplitOp {
    BuildArrays a;
    int buffer;
    uint32_t segBase;
    PTC_HD void operator()(uint32_t i) const
    {
        const uint4 seg = a.topSegments[segBase + i];
        float4 *lo = a.clusterLo[buffer], *hi = a.clusterHi[buffer];
        const uint32_t first = seg.x, end = seg.x + seg.y;
        float bestCost = kInf; int bestAxis = -1; float4 best = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int axis = 0; axis < 3; axis++) { // the first axis with the lowest cost, as one loop over axes and bins would find it
            const float4 c = a.topAxis[3u * (segBase + i) + (uint32_t)axis];
            if ((int)f2u(c.y) >= 0 && c.x < bestCost) { bestCost = c.x; bestAxis = axis; best = c; }
        }
        uint32_t mid = first + seg.y / 2; // identical centroids: split by index
        if (bestAxis >= 0) {
            const int bestBin = (int)f2u(best.y);
            uint32_t c = first, j = end;
            while (c < j) {
                const float4 l = lo[c], h = hi[c];
                const float v = 0.5f * (bestAxis == 0 ? l.x + h.x : (bestAxis == 1 ? l.y + h.y : l.z + h.z));
                int b = (int)((v - best.z) * best.w);
                b = b < 0 ? 0 : (b >= kTopBins ? kTopBins - 1 : b);
                if (b <= bestBin) { c++; }
                else { j--; lo[c] = lo[j]; hi[c] = hi[j]; lo[j] = l; hi[j] = h; }
            }
            if (c != first && c != end) { mid = c; }
        }
        a.topMid[segBase + i] = mid;
    }
};

struct TopEmitOp {
    BuildArrays a;
    int buffer;
    uint32_t segBase, segCount;
    PTC_HD void operator()(uint32_t) const
    {
        const float4 *lo = a.clusterLo[buffer];
        uint32_t appended = a.topState[0], nextFree = a.topState[1];
        for (uint32_t i = 0; i < segCount; i++) {
            const uint4 seg = a.topSegments[segBase + i];
            const uint32_t mid = a.topMid[segBase + i], end = seg.x + seg.y;
            uint32_t child[2];
            const uint32_t firstOf[2] = {seg.x, mid}, countOf[2] = {mid - seg.x, end - mid};
            for (int side = 0; side < 2; side++) {
                if (countOf[side] == 1u) { child[side] = f2u(lo[firstOf[side]].w); continue; } // a PLOC cluster: its node exists
                child[side] = nextFree--;
                a.topSegments[appended++] = make_uint4(firstOf[side], countOf[side], child[side], 0u);
            }
            a.nodeLo[seg.z].w = u2f(child[0]);
            a.nodeHi[seg.z].w = u2f(child[1]);
        }
        a.topState[0] = appended; a.topState[1] = nextFree;
    }
};

struct TopFinishOp {
    BuildArrays a;
    uint32_t segBase;
    PTC_HD void operator()(uint32_t i) const
    {
        const uint32_t node = a.topSegments[segBase + i].z;
        const uint32_t left = f2u(a.nodeLo[node].w), right = f2u(a.nodeHi[node].w);
        const float4 l0 = a.nodeLo[left], h0 = a.nodeHi[left], l1 = a.nodeLo[right], h1 = a.nodeHi[right];
        const float4 l = make_float4(fminf(l0.x, l1.x), fminf(l0.y, l1.y), fminf(l0.z, l1.z), u2f(left));
        const float4 h = make_float4(fmaxf(h0.x, h1.x), fmaxf(h0.y, h1.y), fmaxf(h0.z, h1.z), u2f(right));
        a.nodeLo[node] = l; a.nodeHi[node] = h;
        a.dp[node] = combineDP(a.dp[left], a.dp[right], halfArea(l.x, l.y, l.z, h.x, h.y, h.z), a.costPrim);
    }
};

// ---- step 4: emission ------------------------------------------------------------------------------------------------
PTC_HD bool isBinaryLeaf(const BuildArrays &a, uint32_t n) { return f2u(a.nodeHi[n].w) == kInvalid; }

// children of the wide node made from binary node n: follow the recorded decisions (the host builder's Collector)
PTC_HD int collectChildren(const BuildArrays &a, uint32_t n, uint32_t child[8])
{
    int count = 0;
    const uint32_t rootInfo = a.dp[n].info;
    if (isBinaryLeaf(a, n) || dpRootIsLeaf(rootInfo)) { child[count++] = n; return count; } // a single-leaf scene still needs an inner root
    uint32_t stackNode[16]; int stackI[16]; int sp = 0;
    // distribute(n, 8)
    {
        const int k = (int)dpSplit(rootInfo, 8);
        stackNode[sp] = f2u(a.nodeHi[n].w); stackI[sp++] = 8 - k;
        stackNode[sp] = f2u(a.nodeLo[n].w); stackI[sp++] = k;
    }
    while (sp) {
        const uint32_t m = stackNode[--sp]; int i = stackI[sp];
        if (isBinaryLeaf(a, m)) { child[count++] = m; continue; }
        const NodeDP d = a.dp[m];
        while (i > 1 && d.c[i - 1] == d.c[i - 2]) { i--; } // C(m, i) took the C(m, i-1) branch
        if (i == 1) { child[count++] = m; continue; }
        const int k = (int)dpSplit(d.info, i);
        stackNode[sp] = f2u(a.nodeHi[m].w); stackI[sp++] = i - k;
        stackNode[sp] = f2u(a.nodeLo[m].w); stackI[sp++] = k;
    }
    return count;
}

PTC_HD uint32_t leafPrimsOf(const BuildArrays &a, uint32_t c)
{
    if (isBinaryLeaf(a, c)) { return 1u; }
    const uint32_t info = a.dp[c].info;
    return dpRootIsLeaf(info) ? dpPrimCount(info) : 0u;
}

// pass A: choose the children of every wide node of this level and assign them to octant-ordered slots; count what to allocate
struct EmitPlanOp {
    BuildArrays a;
    int buffer;
    PTC_HD void operator()(uint32_t item) const
    {
        const uint32_t n = a.items[buffer][item];
        uint32_t child[8];
        const int count = collectChildren(a, n, child);
        const float4 lo = a.nodeLo[n], hi = a.nodeHi[n];
        float center[3];
        centroidOf(lo, hi, center);
        // slot assignment: child -> slot minimising (centroid - node centroid) . octant direction, greedily, so that visiting
        // slots in (slot ^ ray octant) order approximates front-to-back
        float slotCost[8][8];
        for (int c = 0; c < count; c++) {
            float cc[3];
            centroidOf(a.nodeLo[child[c]], a.nodeHi[child[c]], cc);
            for (int s = 0; s < 8; s++) {
                const float dsx = (s & 4) ? -1.f : 1.f, dsy = (s & 2) ? -1.f : 1.f, dsz = (s & 1) ? -1.f : 1.f;
                float v = 0.f;
                v += (cc[0] - center[0]) * dsx; v += (cc[1] - center[1]) * dsy; v += (cc[2] - center[2]) * dsz;
                slotCost[c][s] = v;
            }
        }
        int slotOf[8]; uint32_t slotUsed = 0, childDone = 0;
        for (int c = 0; c < 8; c++) { slotOf[c] = -1; }
        for (int round = 0; round < count; round++) {
            float bestCost = kInf; int bc = -1, bs = -1;
            for (int c = 0; c < count; c++) {
                if (childDone & (1u << c)) { continue; }
                for (int s = 0; s < 8; s++) { if (!(slotUsed & (1u << s)) && slotCost[c][s] < bestCost) { bestCost = slotCost[c][s]; bc = c; bs = s; } }
            }
            if (bc < 0) { // non-finite coordinates: any free slot
                for (int c = 0; c < count && bc < 0; c++) { if (!(childDone & (1u << c))) { bc = c; } }
                for (int s = 0; s < 8 && bs < 0; s++) { if (!(slotUsed & (1u << s))) { bs = s; } }
            }
            slotOf[bc] = bs; slotUsed |= 1u << bs; childDone |= 1u << bc;
        }
        uint32_t inSlot[8];
        for (int s = 0; s < 8; s++) { inSlot[s] = kInvalid; }
        for (int c = 0; c < count; c++) { inSlot[slotOf[c]] = child[c]; }
        uint64_t inner = 0, tris = 0;
        for (int s = 0; s < 8; s++) {
            a.itemChildren[8 * (size_t)item + s] = inSlot[s];
            if (inSlot[s] == kInvalid) { continue; }
            const uint32_t lp = leafPrimsOf(a, inSlot[s]);
            if (lp) { tris += lp; } else { inner++; }
        }
        a.scanIn[item] = (inner << 32) | tris;
    }
};

PTC_HD uint8_t exponentForExtent(float extent)
{
    // smallest power of two 2^e with 255 * 2^e >= extent
    if (!(extent > 0.f)) { return 1; }
    int e;
    frexpf(extent / 255.f, &e);
    int biased = e + 127;
    if (biased < 1) { biased = 1; }
    if (biased > 254) { biased = 254; }
    return (uint8_t)biased;
}

// pass B: write the compressed node, its leaf triangles and the next level's work items
struct EmitWriteOp {
    BuildArrays a;
    int buffer;
    uint32_t levelBase;     // wide-node index of item 0 of this level
    uint32_t nextLevelBase; // wide-node index of the first node of the next level
    uint32_t triBaseLevel;  // leaf triangles emitted before this level
    PTC_HD void operator()(uint32_t item) const
    {
        const uint32_t n = a.items[buffer][item];
        const uint64_t prefix = a.scanOut[item];
        const uint32_t innerBefore = (uint32_t)(prefix >> 32), trisBefore = (uint32_t)(prefix & 0xFFFFFFFFu);
        const float4 lo = a.nodeLo[n], hi = a.nodeHi[n];
        WideNode node;
        memset(&node, 0, sizeof(node));
        node.origin[0] = lo.x; node.origin[1] = lo.y; node.origin[2] = lo.z;
        node.exponent[0] = exponentForExtent(hi.x - lo.x); node.exponent[1] = exponentForExtent(hi.y - lo.y);
        node.exponent[2] = exponentForExtent(hi.z - lo.z);
        node.childBase = nextLevelBase + innerBefore;
        node.triBase = triBaseLevel + trisBefore;
        uint32_t innerCount = 0, triCount = 0;
        for (int s = 0; s < 8; s++) {
            const uint32_t c = a.itemChildren[8 * (size_t)item + s];
            if (c == kInvalid) { continue; }
            const float4 clo = a.nodeLo[c], chi = a.nodeHi[c];
            const float cl[3] = {clo.x, clo.y, clo.z}, ch[3] = {chi.x, chi.y, chi.z};
            // quantise outwards and verify against the fp32 decode origin + q * 2^e
            for (int axis = 0; axis < 3; axis++) {
                const float scale = u2f((uint32_t)node.exponent[axis] << 23);
                const float o = node.origin[axis];
                int qlo = (int)floorf((cl[axis] - o) / scale), qhi = (int)ceilf((ch[axis] - o) / scale);
                qlo = qlo < 0 ? 0 : (qlo > 255 ? 255 : qlo); qhi = qhi < 0 ? 0 : (qhi > 255 ? 255 : qhi);
                while (qlo > 0 && o + (float)qlo * scale > cl[axis]) { qlo--; }
                while (qhi < 255 && o + (float)qhi * scale < ch[axis]) { qhi++; }
                uint8_t *ql = axis == 0 ? node.qlox : (axis == 1 ? node.qloy : node.qloz);
                uint8_t *qh = axis == 0 ? node.qhix : (axis == 1 ? node.qhiy : node.qhiz);
                ql[s] = (uint8_t)qlo; qh[s] = (uint8_t)qhi;
            }
            const uint32_t leafPrims = leafPrimsOf(a, c);
            if (leafPrims == 0) {
                node.imask |= (uint8_t)(1u << s);
                node.meta[s] = (uint8_t)((1u << 5) | (24u + (uint32_t)s));
                a.items[buffer ^ 1][innerBefore + innerCount] = c;
                innerCount++;
            } else {
                const uint32_t unary = leafPrims == 1 ? 1u : (leafPrims == 2 ? 3u : 7u);
                node.meta[s] = (uint8_t)((unary << 5) | triCount);
                // the primitives of a collapsed subtree (at most 3): walk it, left first
                uint32_t stack[8]; int sp = 0;
                stack[sp++] = c;
                while (sp) {
                    const uint32_t m = stack[--sp];
                    if (!isBinaryLeaf(a, m)) { stack[sp++] = f2u(a.nodeHi[m].w); stack[sp++] = f2u(a.nodeLo[m].w); continue; }
                    const uint32_t p = f2u(a.nodeLo[m].w);
                    const uint4 ix = a.prims[p];
                    const float4 v0 = a.positions[ix.x], v1 = a.positions[ix.y], v2 = a.positions[ix.z];
                    LeafTriangle t;
                    t.v0[0] = v0.x; t.v0[1] = v0.y; t.v0[2] = v0.z; t.prim = p;
                    t.e1[0] = v0.x - v1.x; t.e1[1] = v0.y - v1.y; t.e1[2] = v0.z - v1.z; t.pad0 = 0;
                    t.e2[0] = v2.x - v0.x; t.e2[1] = v2.y - v0.y; t.e2[2] = v2.z - v0.z; t.pad1 = 0;
                    a.leafTriangles[node.triBase + triCount] = t;
                    triCount++;
                }
            }
        }
        a.wideNodes[levelBase + item] = node;
    }
};

// ---- execution policies --------------------------------------------------------------------------------------------------
#if defined(__CUDACC__)
template <class Op>
__global__ void __launch_bounds__(256) forEachKernel(uint32_t n, Op op)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { op(i); }
}

// centroid bounds of all primitives: warp shuffle reduce, one ordered-int atomic per warp and component
__global__ void __launch_bounds__(256) centroidBoundsKernel(BuildArrays a)
{
    float lo[3] = {kInf, kInf, kInf}, hi[3] = {-kInf, -kInf, -kInf};
    for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < a.nPrims; p += gridDim.x * blockDim.x) {
        float c[3];
        centroidOf(a.primLo[p], a.primHi[p], c);
        for (int k = 0; k < 3; k++) { lo[k] = fminf(lo[k], c[k]); hi[k] = fmaxf(hi[k], c[k]); }
    }
    for (int k = 0; k < 3; k++) {
        for (int offset = 16; offset; offset >>= 1) {
            lo[k] = fminf(lo[k], __shfl_xor_sync(0xFFFFFFFFu, lo[k], offset));
            hi[k] = fmaxf(hi[k], __shfl_xor_sync(0xFFFFFFFFu, hi[k], offset));
        }
    }
    if ((threadIdx.x & 31) == 0) {
        for (int k = 0; k < 3; k++) { atomicMin(&a.bounds[k], orderedBits(lo[k])); atomicMax(&a.bounds[3 + k], orderedBits(hi[k])); }
    }
}
#endif

struct DeviceExec {
    cudaStream_t stream;
    std::vector<void *> owned;
    void *scratch = nullptr; size_t scratchBytes = 0;

    static void check(cudaError_t e, const char *what)
    {
        if (e != cudaSuccess) { throw std::runtime_error(std::string(what) + ": " + cudaGetErrorString(e)); }
    }
    // The working set (436 B per primitive in ~25 arrays) comes out of ONE allocation: every cudaMalloc / cudaFree is a driver call
    // of 0.1-0.5 ms that synchronises the device, which cost as much as the sort.  Requests that do not fit fall back to cudaMalloc.
    char *arena = nullptr; size_t arenaBytes = 0, arenaUsed = 0;
    void reserve(size_t bytes)
    {
        if (arena || cudaMalloc((void **)&arena, bytes) != cudaSuccess) { cudaGetLastError(); return; }
        arenaBytes = bytes; arenaUsed = 0;
    }
    template <class T> T *alloc(size_t n)
    {
        const size_t bytes = (std::max<size_t>(n, 1) * sizeof(T) + 255u) & ~(size_t)255u;
        if (arena && arenaUsed + bytes <= arenaBytes) { void *p = arena + arenaUsed; arenaUsed += bytes; return (T *)p; }
        void *p = nullptr;
        check(cudaMalloc(&p, bytes), "cudaMalloc (BVH build)");
        owned.push_back(p);
        return (T *)p;
    }
    void releaseAll()
    {
        for (void *p : owned) { cudaFree(p); }
        owned.clear();
        if (scratch) { cudaFree(scratch); scratch = nullptr; }
        if (arena) { cudaFree(arena); arena = nullptr; arenaBytes = arenaUsed = 0; }
    }
    void needScratch(size_t bytes)
    {
        if (bytes <= scratchBytes) { return; }
        const size_t rounded = (bytes + 255u) & ~(size_t)255u;
        if (arena && arenaUsed + rounded <= arenaBytes) { scratchFromArena = true; scratchPtr = arena + arenaUsed; arenaUsed += rounded; scratchBytes = bytes; return; }
        if (scratch) { cudaFree(scratch); }
        check(cudaMalloc(&scratch, bytes), "cudaMalloc (scan scratch)");
        scratchPtr = scratch; scratchFromArena = false;
        scratchBytes = bytes;
    }
    void *scratchPtr = nullptr; bool scratchFromArena = false;
    template <class Op> void forEach(uint32_t n, const Op &op)
    {
        if (!n) { return; }
        forEachKernel<<<(n + 255u) / 256u, 256, 0, stream>>>(n, op);
        check(cudaGetLastError(), "BVH build kernel launch");
    }
    void centroidBounds(const BuildArrays &a)
    {
        uint32_t init[6];
        for (int k = 0; k < 3; k++) { init[k] = 0xFFFFFFFFu; init[3 + k] = 0u; }
        check(cudaMemcpyAsync(a.bounds, init, sizeof(init), cudaMemcpyHostToDevice, stream), "bounds init");
        const uint32_t blocks = std::min<uint32_t>((a.nPrims + 255u) / 256u, 148u * 8u);
        centroidBoundsKernel<<<blocks, 256, 0, stream>>>(a);
        check(cudaGetLastError(), "centroidBoundsKernel");
    }
    // returns the buffer index (0 / 1) that holds the sorted keys and values
    int sortPairs(BuildArrays &a)
    {
        cub::DoubleBuffer<uint64_t> keys(a.keys[0], a.keys[1]);
        cub::DoubleBuffer<uint32_t> values(a.order[0], a.order[1]);
        size_t bytes = 0;
        check(cub::DeviceRadixSort::SortPairs(nullptr, bytes, keys, values, (int)a.nPrims, 0, 63, stream), "radix sort size");
        needScratch(bytes);
        check(cub::DeviceRadixSort::SortPairs(scratchPtr, bytes, keys, values, (int)a.nPrims, 0, 63, stream), "radix sort");
        return values.selector;
    }
    // exclusive sum of packed counters; returns the total (sum of all n inputs)
    uint64_t scan(const BuildArrays &a, uint32_t n)
    {
        size_t bytes = 0;
        check(cub::DeviceScan::ExclusiveSum(nullptr, bytes, a.scanIn, a.scanOut, (int)n, stream), "scan size");
        needScratch(bytes);
        check(cub::DeviceScan::ExclusiveSum(scratchPtr, bytes, a.scanIn, a.scanOut, (int)n, stream), "scan");
        uint64_t tail[2];
        check(cudaMemcpyAsync(&tail[0], a.scanIn + (n - 1), 8, cudaMemcpyDeviceToHost, stream), "scan tail");
        check(cudaMemcpyAsync(&tail[1], a.scanOut + (n - 1), 8, cudaMemcpyDeviceToHost, stream), "scan tail");
        check(cudaStreamSynchronize(stream), "scan sync");
        return tail[0] + tail[1];
    }
    void setItem(uint32_t *items, uint32_t value) { check(cudaMemcpyAsync(items, &value, 4, cudaMemcpyHostToDevice, stream), "root item"); check(cudaStreamSynchronize(stream), "root item"); }
    void setTop(const BuildArrays &a, uint4 rootSegment, uint32_t appended, uint32_t nextFree)
    {
        const uint32_t state[2] = {appended, nextFree};
        check(cudaMemcpyAsync(a.topSegments, &rootSegment, sizeof(uint4), cudaMemcpyHostToDevice, stream), "top root");
        check(cudaMemcpyAsync(a.topState, state, sizeof(state), cudaMemcpyHostToDevice, stream), "top state");
        check(cudaStreamSynchronize(stream), "top state"); // the sources are on this stack frame
    }
    uint32_t readWord(const uint32_t *p)
    {
        uint32_t v = 0;
        check(cudaMemcpyAsync(&v, p, 4, cudaMemcpyDeviceToHost, stream), "read back");
        check(cudaStreamSynchronize(stream), "read back");
        return v;
    }
    void sync() { check(cudaStreamSynchronize(stream), "BVH build sync"); }
};

struct HostExec {
    std::vector<void *> owned;
    template <class T> T *alloc(size_t n)
    {
        void *p = calloc(std::max<size_t>(n, 1), sizeof(T));
        if (!p) { throw std::runtime_error("out of memory (BVH build emulation)"); }
        owned.push_back(p);
        return (T *)p;
    }
    void releaseAll() { for (void *p : owned) { free(p); } owned.clear(); }
    template <class Op> void forEach(uint32_t n, const Op &op) { for (uint32_t i = 0; i < n; i++) { op(i); } }
    void centroidBounds(const BuildArrays &a)
    {
        float lo[3] = {kInf, kInf, kInf}, hi[3] = {-kInf, -kInf, -kInf};
        for (uint32_t p = 0; p < a.nPrims; p++) {
            float c[3];
            centroidOf(a.primLo[p], a.primHi[p], c);
            for (int k = 0; k < 3; k++) { lo[k] = fminf(lo[k], c[k]); hi[k] = fmaxf(hi[k], c[k]); }
        }
        for (int k = 0; k < 3; k++) { a.bounds[k] = orderedBits(lo[k]); a.bounds[3 + k] = orderedBits(hi[k]); }
    }
    int sortPairs(BuildArrays &a)
    {
        std::vector<uint32_t> perm(a.nPrims);
        for (uint32_t i = 0; i < a.nPrims; i++) { perm[i] = i; }
        std::stable_sort(perm.begin(), perm.end(), [&](uint32_t x, uint32_t y) { return a.keys[0][x] < a.keys[0][y]; }); // radix sort is stable
        for (uint32_t i = 0; i < a.nPrims; i++) { a.keys[1][i] = a.keys[0][perm[i]]; a.order[1][i] = a.order[0][perm[i]]; }
        return 1;
    }
    uint64_t scan(const BuildArrays &a, uint32_t n)
    {
        uint64_t sum = 0;
        for (uint32_t i = 0; i < n; i++) { a.scanOut[i] = sum; sum += a.scanIn[i]; }
        return sum;
    }
    void setItem(uint32_t *items, uint32_t value) { items[0] = value; }
    void setTop(const BuildArrays &a, uint4 rootSegment, uint32_t appended, uint32_t nextFree) { a.topSegments[0] = rootSegment; a.topState[0] = appended; a.topState[1] = nextFree; }
    uint32_t readWord(const uint32_t *p) { return *p; }
    void sync() {}
};

struct BuildResult {
    uint32_t nNodes = 0, nTriangles = 0, maxDepth = 0, plocIterations = 0;
    double ms[4] = {0, 0, 0, 0}; // boxes + sort, PLOC, emission, total
};

// The build, written once for both policies.  On return a.wideNodes / a.leafTriangles hold the result (owned by exec).
template <class Exec>
BuildResult runBuild(Exec &exec, BuildArrays &a)
{
    BuildResult result;
    const uint32_t n = a.nPrims;
    const auto t0 = std::chrono::steady_clock::now();
    a.costPrim = kCostPrim;
    if (const char *c = getenv("PTC_COST_PRIM")) { a.costPrim = (float)atof(c); } // tuning hook (tools/compare_builders.py)
    a.primLo = exec.template alloc<float4>(n); a.primHi = exec.template alloc<float4>(n);
    a.bounds = exec.template alloc<uint32_t>(6);
    for (int b = 0; b < 2; b++) {
        a.keys[b] = exec.template alloc<uint64_t>(n); a.order[b] = exec.template alloc<uint32_t>(n);
        a.clusterLo[b] = exec.template alloc<float4>(n); a.clusterHi[b] = exec.template alloc<float4>(n);
        a.items[b] = exec.template alloc<uint32_t>(n);
    }
    a.nodeLo = exec.template alloc<float4>(2 * (size_t)n); a.nodeHi = exec.template alloc<float4>(2 * (size_t)n);
    a.dp = exec.template alloc<NodeDP>(2 * (size_t)n);
    a.nearest = exec.template alloc<uint32_t>(n);
    a.scanIn = exec.template alloc<uint64_t>(n); a.scanOut = exec.template alloc<uint64_t>(n);
    a.itemChildren = exec.template alloc<uint32_t>(8 * (size_t)n);
    a.wideNodes = exec.template alloc<WideNode>((size_t)n + 1);
    a.leafTriangles = exec.template alloc<LeafTriangle>(n);

    exec.forEach(n, PrimBoxOp{a});
    exec.centroidBounds(a);
    exec.forEach(n, MortonOp{a});
    const int sortedIn = exec.sortPairs(a);
    exec.forEach(n, LeafOp{a, a.order[sortedIn]});
    exec.sync();
    const auto t1 = std::chrono::steady_clock::now();

    // PLOC: the host only learns the cluster count of the next iteration (8 bytes back per iteration)
    uint32_t nClusters = n, nextNode = n;
    int buffer = 0;
    uint32_t radius = PLOC_RADIUS;
    if (const char *r = getenv("PTC_PLOC_RADIUS")) { radius = (uint32_t)std::max(1, atoi(r)); } // tuning hook (tools/compare_builders.py)
    uint32_t topCount = PLOC_TOP_CLUSTERS;
    if (const char *r = getenv("PTC_PLOC_TOP")) { topCount = (uint32_t)std::max(0, atoi(r)); }
    while (nClusters > 1 && nClusters > topCount) {
        exec.forEach(nClusters, NearestOp{a, buffer, nClusters, radius});
        exec.forEach(nClusters, MergeFlagOp{a});
        const uint64_t total = exec.scan(a, nClusters);
        const uint32_t created = (uint32_t)(total >> 32), survivors = (uint32_t)(total & 0xFFFFFFFFu);
        if (created == 0 || survivors >= nClusters) { throw std::runtime_error("PLOC made no progress"); }
        exec.forEach(nClusters, MergeOp{a, buffer, nClusters, nextNode});
        nextNode += created; nClusters = survivors; buffer ^= 1;
        result.plocIterations++;
    }
    if (nClusters > 1) { // top of the tree: SAH over the remaining clusters, nClusters - 1 inner nodes = segments
        a.topSegments = exec.template alloc<uint4>(nClusters);
        a.topAxis = exec.template alloc<float4>(3 * (size_t)nClusters);
        a.topMid = exec.template alloc<uint32_t>(nClusters);
        a.topState = exec.template alloc<uint32_t>(2);
        const uint32_t rootNode = nextNode + nClusters - 2u;
        exec.setTop(a, make_uint4(0u, nClusters, rootNode, 0u), 1u, rootNode - 1u);
        std::vector<std::pair<uint32_t, uint32_t>> levels; // first segment, segment count
        uint32_t segBase = 0, segCount = 1;
        while (segCount) {
            levels.push_back({segBase, segCount});
            exec.forEach(3u * segCount, TopAxisOp{a, buffer, segBase});
            exec.forEach(segCount, TopSplitOp{a, buffer, segBase});
            exec.forEach(1u, TopEmitOp{a, buffer, segBase, segCount});
            const uint32_t appended = exec.readWord(a.topState);
            if (appended > nClusters - 1u || appended < segBase + segCount) { throw std::runtime_error("top-level SAH pass lost track of its segments"); }
            segBase += segCount; segCount = appended - segBase;
        }
        if (segBase != nClusters - 1u) { throw std::runtime_error("top-level SAH pass made the wrong number of nodes"); }
        for (size_t level = levels.size(); level-- > 0;) { exec.forEach(levels[level].second, TopFinishOp{a, levels[level].first}); }
        nextNode += nClusters - 1u;
    }
    exec.sync();
    const uint32_t root = nextNode - 1; // n == 1: the only leaf
    const auto t2 = std::chrono::steady_clock::now();

    // emission, one level of the wide tree per round
    uint32_t levelBase = 0, levelItems = 1, trisEmitted = 0;
    int itemBuffer = 0;
    exec.setItem(a.items[0], root);
    while (levelItems) {
        result.maxDepth++;
        exec.forEach(levelItems, EmitPlanOp{a, itemBuffer});
        const uint64_t total = exec.scan(a, levelItems);
        const uint32_t innerChildren = (uint32_t)(total >> 32), tris = (uint32_t)(total & 0xFFFFFFFFu);
        const uint32_t nextLevelBase = levelBase + levelItems;
        if ((uint64_t)nextLevelBase + innerChildren > (uint64_t)n + 1) { throw std::runtime_error("wide node overflow"); }
        exec.forEach(levelItems, EmitWriteOp{a, itemBuffer, levelBase, nextLevelBase, trisEmitted});
        trisEmitted += tris; levelBase = nextLevelBase; levelItems = innerChildren; itemBuffer ^= 1;
        if (result.maxDepth > PTC_STACK_SIZE) { throw std::runtime_error("BVH deeper than the traversal stack"); }
    }
    exec.sync();
    const auto t3 = std::chrono::steady_clock::now();
    result.nNodes = levelBase; result.nTriangles = trisEmitted;
    if (trisEmitted != n) { throw std::runtime_error("BVH build lost primitives"); }
    if (result.maxDepth + 2 > PTC_STACK_SIZE) { throw std::runtime_error("BVH deeper than the traversal stack"); }
    auto ms = [](auto x, auto y) { return std::chrono::duration<double, std::milli>(y - x).count(); };
    result.ms[0] = ms(t0, t1); result.ms[1] = ms(t1, t2); result.ms[2] = ms(t2, t3); result.ms[3] = ms(t0, t3);
    if (getenv("PTC_BUILD_TIMING")) {
        fprintf(stderr, "buildWideBVH(device algorithm): %u prims: boxes+sort %.2f ms, PLOC %.2f ms (%u iterations), emit %.2f ms (%u levels) -> %u wide nodes\n",
                n, result.ms[0], result.ms[1], result.plocIterations, result.ms[2], result.maxDepth, result.nNodes);
    }
    return result;
}

} // namespace

// ---- public entry points ---------------------------------------------------------------------------------------------
void buildWideBVHDevice(const float4 *dPositions, const uint4 *dPrims, uint32_t nPrims, cudaStream_t stream, DeviceWideBVH &out, void **workspaceOut)
{
    if (workspaceOut) { *workspaceOut = nullptr; }
    out = DeviceWideBVH();
    if (nPrims == 0) { return; }
    DeviceExec exec; exec.stream = stream;
    const bool timing = getenv("PTC_BUILD_TIMING") != nullptr;
    auto now = [] { return std::chrono::steady_clock::now(); };
    auto msBetween = [](auto x, auto y) { return std::chrono::duration<double, std::milli>(y - x).count(); };
    const auto c0 = now();
    exec.reserve((size_t)nPrims * 480u + (8u << 20)); // 436 B per primitive + radix-sort scratch (~24 B per primitive) + alignment
    const auto c1 = now();
    BuildArrays a;
    memset(&a, 0, sizeof(a));
    a.positions = dPositions; a.prims = dPrims; a.nPrims = nPrims;
    try {
        const BuildResult r = runBuild(exec, a);
        const auto c2 = now();
        // exact-size copies of the result; the build's working set (about 440 B per primitive) is released
        float4 *nodes = nullptr, *tris = nullptr;
        DeviceExec::check(cudaMalloc((void **)&nodes, (size_t)r.nNodes * sizeof(WideNode)), "cudaMalloc (BVH nodes)");
        if (cudaMalloc((void **)&tris, (size_t)r.nTriangles * sizeof(LeafTriangle)) != cudaSuccess) { cudaFree(nodes); throw std::runtime_error("cudaMalloc (BVH triangles)"); }
        const auto c2b = now();
        cudaMemcpyAsync(nodes, a.wideNodes, (size_t)r.nNodes * sizeof(WideNode), cudaMemcpyDeviceToDevice, stream);
        cudaMemcpyAsync(tris, a.leafTriangles, (size_t)r.nTriangles * sizeof(LeafTriangle), cudaMemcpyDeviceToDevice, stream);
        const cudaError_t e = cudaStreamSynchronize(stream);
        if (e != cudaSuccess) { cudaFree(nodes); cudaFree(tris); DeviceExec::check(e, "BVH copy"); }
        out.nodes = nodes; out.triangles = tris; out.nNodes = r.nNodes; out.nTriangles = r.nTriangles; out.maxDepth = r.maxDepth;
        out.plocIterations = r.plocIterations;
        for (int k = 0; k < 4; k++) { out.buildMs[k] = (float)r.ms[k]; }
        const auto c3 = now();
        if (workspaceOut && exec.arena) { *workspaceOut = exec.arena; exec.arena = nullptr; }
        exec.releaseAll();
        if (timing) {
            fprintf(stderr, "buildWideBVHDevice: reserve %.2f ms, build %.2f ms, exact-size allocations %.2f ms + copies %.2f ms, release %.2f ms\n", msBetween(c0, c1),
                    msBetween(c1, c2), msBetween(c2, c2b), msBetween(c2b, c3), msBetween(c3, now()));
        }
    } catch (...) {
        exec.releaseAll();
        throw;
    }
}

void buildWideBVHEmulated(const float *positions4, const uint32_t *indices4, uint32_t nPrims, WideBVH &out)
{
    out.nodes.clear(); out.triangles.clear(); out.maxDepth = 0;
    if (nPrims == 0) { return; }
    HostExec exec;
    BuildArrays a;
    memset(&a, 0, sizeof(a));
    a.positions = (const float4 *)positions4; a.prims = (const uint4 *)indices4; a.nPrims = nPrims;
    try {
        const BuildResult r = runBuild(exec, a);
        out.nodes.assign(a.wideNodes, a.wideNodes + r.nNodes);
        out.triangles.assign(a.leafTriangles, a.leafTriangles + r.nTriangles);
        out.maxDepth = r.maxDepth;
    } catch (...) {
        exec.releaseAll();
        throw;
    }
    exec.releaseAll();
}

} // namespace ptc
