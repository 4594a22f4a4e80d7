// Host BVH builder (see bvh.h): binned SAH binary tree -> greedy collapse to 8-wide -> compressed 80-byte nodes.
#include "bvh.h"
#include "traverse.cuh"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <cstring>
#include <future>
#include <queue>
#include <stdexcept>
#include <thread>

namespace ptc {

namespace {

struct Box {
    float lo[3], hi[3];
    void reset() { for (int a = 0; a < 3; a++) { lo[a] = 3.0e38f; hi[a] = -3.0e38f; } }
    void grow(const float *p) { for (int a = 0; a < 3; a++) { lo[a] = std::min(lo[a], p[a]); hi[a] = std::max(hi[a], p[a]); } }
    void grow(const Box &b) { for (int a = 0; a < 3; a++) { lo[a] = std::min(lo[a], b.lo[a]); hi[a] = std::max(hi[a], b.hi[a]); } }
    float halfArea() const
    {
        const float x = hi[0] - lo[0], y = hi[1] - lo[1], z = hi[2] - lo[2];
        return x < 0.f ? 0.f : x * y + y * z + z * x;
    }
};

struct Node2 {
    Box box;
    uint32_t left = 0, right = 0; // children when count == 0
    uint32_t first = 0, count = 0;
};

struct Builder {
    const float *pos;
    const uint32_t *idx;
    std::vector<Box> primBox;
    std::vector<float> centroid; // 3 per prim
    std::vector<uint32_t> order;
    std::vector<Node2> nodes;
    std::atomic<uint32_t> nodeCount{0};
    int maxThreads = 1;
    std::atomic<int> activeThreads{1};

    static constexpr int BINS = 16;
    static constexpr uint32_t MAX_LEAF = 3;

    uint32_t alloc() { return nodeCount.fetch_add(1); }

    void build(uint32_t nodeIndex, uint32_t first, uint32_t count, int depth)
    {
        Node2 &node = nodes[nodeIndex];
        node.box.reset();
        Box cbox; cbox.reset();
        for (uint32_t i = first; i < first + count; i++) {
            node.box.grow(primBox[order[i]]);
            cbox.grow(&centroid[3 * (size_t)order[i]]);
        }
        node.first = first; node.count = 0;
        if (count == 1) { node.count = 1; return; }

        // binned SAH over the three axes
        float bestCost = 3.0e38f; int bestAxis = -1, bestBin = -1;
        for (int axis = 0; axis < 3; axis++) {
            const float lo = cbox.lo[axis], extent = cbox.hi[axis] - cbox.lo[axis];
            if (!(extent > 0.f)) { continue; }
            Box binBox[BINS]; uint32_t binCount[BINS];
            for (int b = 0; b < BINS; b++) { binBox[b].reset(); binCount[b] = 0; }
            const float scale = (float)BINS / extent;
            for (uint32_t i = first; i < first + count; i++) {
                const uint32_t p = order[i];
                int b = (int)((centroid[3 * (size_t)p + axis] - lo) * scale);
                b = b < 0 ? 0 : (b >= BINS ? BINS - 1 : b);
                binBox[b].grow(primBox[p]); binCount[b]++;
            }
            float rightArea[BINS]; uint32_t rightCount[BINS];
            Box acc; acc.reset(); uint32_t n = 0;
            for (int b = BINS - 1; b > 0; b--) { acc.grow(binBox[b]); n += binCount[b]; rightArea[b] = acc.halfArea(); rightCount[b] = n; }
            acc.reset(); n = 0;
            for (int b = 0; b < BINS - 1; b++) {
                acc.grow(binBox[b]); n += binCount[b];
                if (n == 0 || rightCount[b + 1] == 0) { continue; }
                const float cost = acc.halfArea() * n + rightArea[b + 1] * rightCount[b + 1];
                if (cost < bestCost) { bestCost = cost; bestAxis = axis; bestBin = b; }
            }
        }
        // leaf when it is small enough and splitting does not pay (unit triangle cost, 1.0 per inner step)
        if (count <= MAX_LEAF) {
            const float leafCost = (float)count * node.box.halfArea();
            if (bestAxis < 0 || bestCost + 1.0f * node.box.halfArea() >= leafCost) { node.count = count; return; }
        }
        uint32_t mid;
        if (bestAxis < 0) {
            mid = first + count / 2; // identical centroids: split by index
        } else {
            const float lo = cbox.lo[bestAxis], scale = (float)BINS / (cbox.hi[bestAxis] - cbox.lo[bestAxis]);
            auto it = std::partition(order.begin() + first, order.begin() + first + count, [&](uint32_t p) {
                int b = (int)((centroid[3 * (size_t)p + bestAxis] - lo) * scale);
                b = b < 0 ? 0 : (b >= BINS ? BINS - 1 : b);
                return b <= bestBin;
            });
            mid = (uint32_t)(it - order.begin());
            if (mid == first || mid == first + count) { mid = first + count / 2; }
        }
        const uint32_t l = alloc(), r = alloc();
        nodes[nodeIndex].left = l; nodes[nodeIndex].right = r;
        const uint32_t leftCount = mid - first, rightCount = first + count - mid;
        if (count > 16384 && activeThreads.load() < maxThreads) {
            activeThreads.fetch_add(1);
            std::thread worker([=]() { build(l, first, leftCount, depth + 1); activeThreads.fetch_sub(1); });
            build(r, mid, rightCount, depth + 1);
            worker.join();
        } else {
            build(l, first, leftCount, depth + 1);
            build(r, mid, rightCount, depth + 1);
        }
    }
};

uint8_t exponentFor(float extent)
{
    // smallest power of two 2^e with 255 * 2^e >= extent
    if (!(extent > 0.f)) { return 1; }
    int e;
    std::frexp(extent / 255.f, &e); // extent/255 = m * 2^e, m in [0.5, 1)  ->  2^e >= extent/255
    int biased = e + 127;
    if (biased < 1) { biased = 1; }
    if (biased > 254) { biased = 254; }
    return (uint8_t)biased;
}

} // namespace

void buildWideBVH(const float *positions4, const uint32_t *indices4, uint32_t nPrims, WideBVH &out)
{
    out.nodes.clear(); out.triangles.clear(); out.maxDepth = 0;
    if (nPrims == 0) { return; }

    const auto t0 = std::chrono::steady_clock::now();
    Builder b;
    b.pos = positions4; b.idx = indices4;
    b.primBox.resize(nPrims); b.centroid.resize(3 * (size_t)nPrims); b.order.resize(nPrims);
    for (uint32_t p = 0; p < nPrims; p++) {
        Box box; box.reset();
        for (int k = 0; k < 3; k++) { box.grow(positions4 + 4 * (size_t)indices4[4 * (size_t)p + k]); }
        b.primBox[p] = box;
        for (int a = 0; a < 3; a++) { b.centroid[3 * (size_t)p + a] = 0.5f * (box.lo[a] + box.hi[a]); }
        b.order[p] = p;
    }
    b.nodes.resize(2 * (size_t)nPrims);
    b.maxThreads = (int)std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
    const uint32_t root = b.alloc();
    b.build(root, 0, nPrims, 0);

    const auto t1 = std::chrono::steady_clock::now();
    // ---- SAH-optimal collapse to 8-wide (Ylitie, Karras, Laine 2017, section 3.1): C(n, i) = cheapest way to represent the
    // binary subtree n as a forest of at most i wide-BVH roots, bottom-up; a subtree of at most 3 triangles may become one leaf.
    const float cNode = 1.0f, cPrim = 0.4f;
    const size_t nBinary = b.nodeCount.load();
    std::vector<float> cost(nBinary * 7);          // cost[n*7 + i-1] = C(n, i), i = 1..7
    std::vector<uint8_t> splitAt(nBinary * 8, 0);  // splitAt[n*8 + j-1]: best k of C_distribute(n, j), j = 2..8
    std::vector<uint8_t> rootIsLeaf(nBinary, 0);
    std::vector<uint32_t> primCount(nBinary, 0);
    {
        std::vector<std::pair<uint32_t, bool>> todo;
        todo.emplace_back(root, false);
        while (!todo.empty()) {
            const uint32_t n = todo.back().first;
            const bool expanded = todo.back().second;
            const Node2 &node = b.nodes[n];
            float *c = &cost[(size_t)n * 7];
            if (node.count) { // binary leaf
                todo.pop_back();
                primCount[n] = node.count;
                for (int i = 0; i < 7; i++) { c[i] = node.box.halfArea() * (float)node.count * cPrim; }
                rootIsLeaf[n] = 1;
                continue;
            }
            if (!expanded) { todo.back().second = true; todo.emplace_back(node.left, false); todo.emplace_back(node.right, false); continue; }
            todo.pop_back();
            primCount[n] = primCount[node.left] + primCount[node.right];
            const float *cl = &cost[(size_t)node.left * 7], *cr = &cost[(size_t)node.right * 7];
            float distribute[9];
            for (int j = 2; j <= 8; j++) {
                float best = 3.0e38f; int bestK = 1;
                for (int k = 1; k < j; k++) {
                    if (k > 7 || j - k > 7) { continue; }
                    const float v = cl[k - 1] + cr[j - k - 1];
                    if (v < best) { best = v; bestK = k; }
                }
                distribute[j] = best; splitAt[(size_t)n * 8 + j - 1] = (uint8_t)bestK;
            }
            const float area = node.box.halfArea();
            const float internal = distribute[8] + area * cNode;
            const float leaf = primCount[n] <= Builder::MAX_LEAF ? area * (float)primCount[n] * cPrim : 3.0e38f;
            rootIsLeaf[n] = leaf <= internal ? 1 : 0;
            c[0] = std::min(leaf, internal);
            for (int i = 2; i <= 7; i++) { c[i - 1] = std::min(distribute[i], c[i - 2]); }
        }
    }
    // children of the wide node made from binary node n: follow the recorded decisions
    struct Collector {
        const Builder &b; const std::vector<float> &cost; const std::vector<uint8_t> &splitAt;
        void distribute(uint32_t n, int j, uint32_t *out, int &count) const
        {
            const int k = splitAt[(size_t)n * 8 + j - 1];
            place(b.nodes[n].left, k, out, count);
            place(b.nodes[n].right, j - k, out, count);
        }
        void place(uint32_t m, int i, uint32_t *out, int &count) const
        {
            if (b.nodes[m].count) { out[count++] = m; return; }
            const float *c = &cost[(size_t)m * 7];
            while (i > 1 && c[i - 1] == c[i - 2]) { i--; } // C(m, i) took the C(m, i-1) branch
            if (i == 1) { out[count++] = m; return; }
            distribute(m, i, out, count);
        }
    };
    const Collector collector = {b, cost, splitAt};

    const auto t2 = std::chrono::steady_clock::now();
    // ---- emit wide nodes breadth first so that the inner children of a node are contiguous
    struct Work { uint32_t wide, node2, depth; };
    std::queue<Work> work;
    out.nodes.emplace_back();
    work.push({0u, root, 1u});
    while (!work.empty()) {
        const Work w = work.front(); work.pop();
        out.maxDepth = std::max(out.maxDepth, w.depth);
        uint32_t child[8]; int n = 0;
        const Node2 &self = b.nodes[w.node2];
        if (self.count || rootIsLeaf[w.node2]) { child[n++] = w.node2; } // a single-leaf scene still needs an inner root
        else { collector.distribute(w.node2, 8, child, n); }
        // slot assignment: child -> slot minimising (centroid - node centroid) . octant direction, greedily,
        // so that visiting slots in (slot ^ ray octant) order approximates front-to-back
        float center[3];
        for (int a = 0; a < 3; a++) { center[a] = 0.5f * (self.box.lo[a] + self.box.hi[a]); }
        float slotCost[8][8];
        for (int c = 0; c < n; c++) {
            const Box &cb = b.nodes[child[c]].box;
            for (int s = 0; s < 8; s++) {
                const float ds[3] = {(s & 4) ? -1.f : 1.f, (s & 2) ? -1.f : 1.f, (s & 1) ? -1.f : 1.f};
                slotCost[c][s] = 0.f;
                for (int a = 0; a < 3; a++) { slotCost[c][s] += (0.5f * (cb.lo[a] + cb.hi[a]) - center[a]) * ds[a]; }
            }
        }
        int slotOf[8]; bool slotUsed[8] = {false, false, false, false, false, false, false, false};
        for (int c = 0; c < 8; c++) { slotOf[c] = -1; }
        for (int round = 0; round < n; round++) {
            float bestCost = 3.0e38f; int bc = -1, bs = -1;
            for (int c = 0; c < n; c++) {
                if (slotOf[c] >= 0) { continue; }
                for (int s = 0; s < 8; s++) { if (!slotUsed[s] && slotCost[c][s] < bestCost) { bestCost = slotCost[c][s]; bc = c; bs = s; } }
            }
            slotOf[bc] = bs; slotUsed[bs] = true;
        }
        int childInSlot[8];
        for (int s = 0; s < 8; s++) { childInSlot[s] = -1; }
        for (int c = 0; c < n; c++) { childInSlot[slotOf[c]] = c; }

        WideNode node;
        memset(&node, 0, sizeof(node));
        for (int a = 0; a < 3; a++) {
            node.origin[a] = self.box.lo[a];
            node.exponent[a] = exponentFor(self.box.hi[a] - self.box.lo[a]);
        }
        node.childBase = (uint32_t)out.nodes.size();
        node.triBase = (uint32_t)out.triangles.size();
        for (int s = 0; s < 8; s++) {
            if (childInSlot[s] < 0) { continue; }
            const uint32_t c2 = child[childInSlot[s]];
            const Node2 &c = b.nodes[c2];
            // quantise outwards and verify against the fp32 decode the kernels use
            for (int a = 0; a < 3; a++) {
                const float scale = u2f((uint32_t)node.exponent[a] << 23);
                int qlo = (int)std::floor((c.box.lo[a] - node.origin[a]) / scale);
                int qhi = (int)std::ceil((c.box.hi[a] - node.origin[a]) / scale);
                qlo = std::max(0, std::min(255, qlo)); qhi = std::max(0, std::min(255, qhi));
                while (qlo > 0 && node.origin[a] + (float)qlo * scale > c.box.lo[a]) { qlo--; }
                while (qhi < 255 && node.origin[a] + (float)qhi * scale < c.box.hi[a]) { qhi++; }
                uint8_t *lo = a == 0 ? node.qlox : (a == 1 ? node.qloy : node.qloz);
                uint8_t *hi = a == 0 ? node.qhix : (a == 1 ? node.qhiy : node.qhiz);
                lo[s] = (uint8_t)qlo; hi[s] = (uint8_t)qhi;
            }
            const uint32_t leafPrims = c.count ? c.count : (rootIsLeaf[c2] ? primCount[c2] : 0u);
            if (leafPrims == 0) {
                node.imask |= (uint8_t)(1u << s);
                node.meta[s] = (uint8_t)((1u << 5) | (24u + (uint32_t)s));
                const uint32_t wideIndex = (uint32_t)out.nodes.size();
                out.nodes.emplace_back();
                work.push({wideIndex, c2, w.depth + 1});
            } else {
                const uint32_t offset = (uint32_t)out.triangles.size() - node.triBase;
                const uint32_t unary = leafPrims == 1 ? 1u : (leafPrims == 2 ? 3u : 7u);
                node.meta[s] = (uint8_t)((unary << 5) | offset);
                for (uint32_t i = 0; i < leafPrims; i++) {
                    const uint32_t p = b.order[c.first + i];
                    const float *v0 = positions4 + 4 * (size_t)indices4[4 * (size_t)p];
                    const float *v1 = positions4 + 4 * (size_t)indices4[4 * (size_t)p + 1];
                    const float *v2 = positions4 + 4 * (size_t)indices4[4 * (size_t)p + 2];
                    LeafTriangle t;
                    memset(&t, 0, sizeof(t));
                    for (int a = 0; a < 3; a++) { t.v0[a] = v0[a]; t.e1[a] = v0[a] - v1[a]; t.e2[a] = v2[a] - v0[a]; }
                    t.prim = p;
                    out.triangles.push_back(t);
                }
            }
        }
        out.nodes[w.wide] = node;
    }
    if (getenv("PTC_BUILD_TIMING")) {
        const auto t3 = std::chrono::steady_clock::now();
        auto ms = [](auto a, auto b) { return std::chrono::duration<double, std::milli>(b - a).count(); };
        fprintf(stderr, "buildWideBVH: %u prims: binary SAH %.1f ms, collapse DP %.1f ms, emit %.1f ms -> %zu wide nodes\n", nPrims,
                ms(t0, t1), ms(t1, t2), ms(t2, t3), out.nodes.size());
    }
    if (out.maxDepth + 2 > PTC_STACK_SIZE) { throw std::runtime_error("BVH deeper than the traversal stack"); }
}

double wideBVHCost(const WideBVH &bvh)
{
    if (bvh.nodes.empty()) { return 0.0; }
    struct Entry { uint32_t node; double area; };
    std::vector<Entry> todo;
    auto slotArea = [](const WideNode &n, int s) {
        double e[3];
        const uint8_t *lo[3] = {n.qlox, n.qloy, n.qloz}, *hi[3] = {n.qhix, n.qhiy, n.qhiz};
        for (int a = 0; a < 3; a++) { e[a] = (double)u2f((uint32_t)n.exponent[a] << 23) * (double)((int)hi[a][s] - (int)lo[a][s]); }
        return e[0] * e[1] + e[1] * e[2] + e[2] * e[0];
    };
    double rootArea = 0.0;
    {
        const WideNode &r = bvh.nodes[0];
        double lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300};
        const uint8_t *ql[3] = {r.qlox, r.qloy, r.qloz}, *qh[3] = {r.qhix, r.qhiy, r.qhiz};
        for (int s = 0; s < 8; s++) {
            if (!r.meta[s]) { continue; }
            for (int a = 0; a < 3; a++) { lo[a] = std::min(lo[a], (double)ql[a][s]); hi[a] = std::max(hi[a], (double)qh[a][s]); }
        }
        double e[3];
        for (int a = 0; a < 3; a++) { e[a] = (double)u2f((uint32_t)r.exponent[a] << 23) * std::max(0.0, hi[a] - lo[a]); }
        rootArea = e[0] * e[1] + e[1] * e[2] + e[2] * e[0];
    }
    double cost = 0.0;
    todo.push_back({0u, rootArea});
    while (!todo.empty()) {
        const Entry en = todo.back(); todo.pop_back();
        const WideNode &n = bvh.nodes[en.node];
        cost += en.area * 1.0;
        uint32_t inner = 0;
        for (int s = 0; s < 8; s++) {
            if (!n.meta[s]) { continue; }
            if (n.imask & (1u << s)) { todo.push_back({n.childBase + inner, slotArea(n, s)}); inner++; }
            else { cost += slotArea(n, s) * 0.4 * (double)popCount((uint32_t)n.meta[s] >> 5); }
        }
    }
    return rootArea > 0.0 ? cost / rootArea : 0.0;
}

bool traverseReference(const WideBVH &bvh, const float o[3], const float d[3], float tnear, float tfar, bool anyHit,
                       float *tOut, uint32_t *primOut, TraversalCounts *counts)
{
    BvhView view;
    view.nodes = (const float4 *)bvh.nodes.data();
    view.triangles = (const float4 *)bvh.triangles.data();
    view.spheres = nullptr; view.nSpheres = 0; view.nNodes = (uint32_t)bvh.nodes.size();
    view.primEvent = nullptr; view.sphereEvent = nullptr;
    view.placements = bvh.placements.empty() ? nullptr : (const float4 *)bvh.placements.data();
    RayHit hit; TraverseCounters c = {0, 0};
    const bool found = anyHit ? traverseBVH<true, true>(view, o[0], o[1], o[2], d[0], d[1], d[2], tnear, tfar, hit, &c)
                              : traverseBVH<false, true>(view, o[0], o[1], o[2], d[0], d[1], d[2], tnear, tfar, hit, &c);
    if (tOut) { *tOut = hit.t; }
    if (primOut) { *primOut = hit.prim; }
    if (counts) { counts->innerVisits += c.inner; counts->triangleTests += c.tris; }
    return found;
}

} // namespace ptc
