// Host-side BLAS builder: C++ mirror of the reference's C# builder, which stays
// on the host in production (north_star: "the C# host keeps glTF load, SweepSAH
// BVH build and camera"). It exists here because this image has no .NET; it
// produces exactly the arrays the engine uploads to SSBO 20-23.
//
// Mirrors (file:line relative to /root/reference/IDKEngine/Source):
//   Bvh/PreSplitting.cs:26-160   PreSplit (early split clipping)
//   Bvh/BLAS.cs:128-157          GetBuildData (3 radix sorts by centroid key)
//   Bvh/BLAS.cs:159-274          Build / ProcessBuildTask / RemoveEmptySubtrees
//   Bvh/BLAS.cs:730-873          TrySplit (SweepSAH with early-outs)
//   Bvh/BLAS.cs:875-937          OptimizeStackSize
//   Bvh/BLAS.cs:441-466          GetUnindexedTriangles (refittable path)
//   Bvh/PreSplitting.cs:169-273  GetUnindexedTriangles (dedup + straddling)
//   Utils/Algorithms.cs:15-112,276-297  FloatToKey, RadixSort, StablePartition
//   Shapes/Box.cs, Shapes/Triangle.cs:47-92, Utils/MyMath.cs:222-230
//
// Float semantics: C# does not contract a*b+c; only MyMath.HalfArea uses an
// explicit fused multiply-add (float.MultiplyAddEstimate). Compile with
// -ffp-contract=off; fmaf() is used where the reference fuses.

#include <cstdint>
#include <cstring>
#include <cmath>
#include <cfloat>
#include <climits>
#include <vector>
#include <algorithm>
#include <thread>
#include <chrono>
#include <atomic>
#include <mutex>
#include <condition_variable>
#include <string>

#include "../../include/idk_gpu_types.h"
#include "../../include/idk_cbrtf.h"

namespace {

struct V3 {
    float x, y, z;
    float operator[](int i) const { return i == 0 ? x : (i == 1 ? y : z); }
};
static inline V3 operator-(V3 a, V3 b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
static inline V3 operator+(V3 a, V3 b) { return {a.x + b.x, a.y + b.y, a.z + b.z}; }
static inline V3 operator*(float s, V3 a) { return {s * a.x, s * a.y, s * a.z}; }
static inline V3 cross(V3 l, V3 r) {
    // OpenTK Vector3.Cross
    return {l.y * r.z - l.z * r.y, l.z * r.x - l.x * r.z, l.x * r.y - l.y * r.x};
}

// Vector128.MinNative/MaxNative on x86 = minps/maxps: (a < b) ? a : b.
static inline float minN(float a, float b) { return a < b ? a : b; }
static inline float maxN(float a, float b) { return a > b ? a : b; }

struct Box {
    float mn[3], mx[3];
    static Box empty() { return {{FLT_MAX, FLT_MAX, FLT_MAX}, {-FLT_MAX, -FLT_MAX, -FLT_MAX}}; }
    void grow(V3 p) {
        mn[0] = minN(mn[0], p.x); mn[1] = minN(mn[1], p.y); mn[2] = minN(mn[2], p.z);
        mx[0] = maxN(mx[0], p.x); mx[1] = maxN(mx[1], p.y); mx[2] = maxN(mx[2], p.z);
    }
    void grow(const Box& b) {
        for (int i = 0; i < 3; i++) { mn[i] = minN(mn[i], b.mn[i]); mx[i] = maxN(mx[i], b.mx[i]); }
    }
    void clip(const Box& b) {
        for (int i = 0; i < 3; i++) { mn[i] = maxN(mn[i], b.mn[i]); mx[i] = minN(mx[i], b.mx[i]); }
    }
    float size(int i) const { return mx[i] - mn[i]; }
    int largestAxis() const {
        int axis = 0;
        if (size(0) < size(1)) axis = 1;
        if (size(axis) < size(2)) axis = 2;
        return axis;
    }
    float largestExtent() const { return maxN(size(0), maxN(size(1), size(2))); }
    // MyMath.HalfArea: fma(x + y, z, x * y)
    float halfArea() const {
        float sx = size(0), sy = size(1), sz = size(2);
        return fmaf(sx + sy, sz, sx * sy);
    }
    float area() const { return halfArea() * 2.0f; }
};

static inline float nodeHalfArea(const GpuBlasNode& n) {
    float sx = n.Max[0] - n.Min[0], sy = n.Max[1] - n.Min[1], sz = n.Max[2] - n.Min[2];
    return fmaf(sx + sy, sz, sx * sy);
}

struct Tri { V3 p0, p1, p2; };

static Box boxFromTri(const Tri& t) {
    Box b = {{t.p0.x, t.p0.y, t.p0.z}, {t.p0.x, t.p0.y, t.p0.z}};
    b.grow(t.p1);
    b.grow(t.p2);
    return b;
}

// Triangle.Split, Shapes/Triangle.cs:47-92
static void triSplit(const Tri& t, int axis, float position, Box& lBox, Box& rBox) {
    lBox = Box::empty();
    rBox = Box::empty();
    bool q0 = t.p0[axis] <= position;
    bool q1 = t.p1[axis] <= position;
    bool q2 = t.p2[axis] <= position;
    if (q0) lBox.grow(t.p0); else rBox.grow(t.p0);
    if (q1) lBox.grow(t.p1); else rBox.grow(t.p1);
    if (q2) lBox.grow(t.p2); else rBox.grow(t.p2);
    auto splitEdge = [&](V3 a, V3 b) {
        float tt = (position - a[axis]) / (b[axis] - a[axis]);
        return a + tt * (b - a);
    };
    if (q0 ^ q1) { V3 m = splitEdge(t.p0, t.p1); lBox.grow(m); rBox.grow(m); }
    if (q1 ^ q2) { V3 m = splitEdge(t.p1, t.p2); lBox.grow(m); rBox.grow(m); }
    if (q2 ^ q0) { V3 m = splitEdge(t.p2, t.p0); lBox.grow(m); rBox.grow(m); }
}

static inline uint32_t floatToKey(float v) {
    uint32_t f;
    memcpy(&f, &v, 4);
    uint32_t mask = (uint32_t)(((int32_t)f >> 31) | (1 << 31));
    return f ^ mask;
}

// C# (int)float on x86-64 (cvttss2si): NaN / out of range -> INT_MIN.
static inline int csFloatToInt(float f) {
    if (!(f > -2147483904.0f && f < 2147483648.0f)) return INT_MIN;
    return (int)f;
}

struct Settings {
    int   stopSplittingThreshold = 1;
    int   maxLeafTriangleCount = 2;
    float triangleCost = 1.1f;
    int   stackOptThreshold = 16;
    float stackOptSahIncreaseAcceptance = 0.0009745f;
    float stackOptMaxLeafTriangleCount = (float)INT_MAX;
    float splitFactor = 0.3f;
    int   doPreSplit = 1;
    int   threads = 1;
};

struct Geometry {
    const PackedVec3* pos;
    const GpuBlasTriangle* tris;
    int triCount;
    Tri tri(int i) const {
        const GpuBlasTriangle& t = tris[i];
        return {{pos[t.X].x, pos[t.X].y, pos[t.X].z}, {pos[t.Y].x, pos[t.Y].y, pos[t.Y].z}, {pos[t.Z].x, pos[t.Z].y, pos[t.Z].z}};
    }
};

struct Fragments {
    std::vector<Box> bounds;
    std::vector<int> originalTriIds; // empty when not presplit
};

// ---------------------------------------------------------------- PreSplitting.PreSplit
static float priority(const Tri& t) {
    Box b = boxFromTri(t);
    float le = b.largestExtent();
    float extentPrio = le * le;
    V3 c = cross(t.p1 - t.p0, t.p2 - t.p0);
    float triArea = sqrtf(c.x * c.x + c.y * c.y + c.z * c.z) * 0.5f;
    float emptyAreaPrio = b.area() - triArea;
    return idk_cbrtf(extentPrio * emptyAreaPrio);   // glibc's cbrtf, restated: include/idk_cbrtf.h
}

static int getSplitCount(float prio, float totalPrio, int triCount, float splitFactor) {
    float shareOfTris = prio / totalPrio * (float)triCount;
    int c = csFloatToInt(shareOfTris * splitFactor);
    if (c == INT_MIN || c < 0) c = 0; // robustness guard (degenerate input); reference would overflow
    return 1 + c;
}

static float getNodeSize(float extent, float globalSize) {
    float alpha = extent / globalSize;
    uint32_t bits;
    memcpy(&bits, &alpha, 4);
    bits &= (255u << 23);
    float p2;
    memcpy(&p2, &bits, 4);
    return p2 * globalSize;
}

static void preSplit(const Geometry& g, const Settings& s, Fragments& out) {
    // Priorities once (the reference evaluates GetPriority three times per triangle); the total is summed in triangle order
    // on one thread, exactly as PreSplitting.cs:33-37 does, because float addition order matters.
    std::vector<float> prio((size_t)g.triCount);
    auto chunked = [&](auto&& f) {
        const int workers = std::max(1, std::min(s.threads, g.triCount / 4096 + 1));
        if (workers == 1) { f(0, g.triCount); return; }
        std::vector<std::thread> pool;
        const int per = (g.triCount + workers - 1) / workers;
        for (int w = 0; w < workers; w++) pool.emplace_back([&, w]() { f(std::min(g.triCount, w * per), std::min(g.triCount, (w + 1) * per)); });
        for (auto& t : pool) t.join();
    };
    chunked([&](int b0, int e0) { for (int i = b0; i < e0; i++) prio[i] = priority(g.tri(i)); });
    float totalPriority = 0.0f;
    for (int i = 0; i < g.triCount; i++) totalPriority += prio[i];

    // every triangle emits exactly its split count (left + right counts always add up), so the output offsets are a prefix sum
    std::vector<size_t> offset((size_t)g.triCount + 1, 0);
    for (int i = 0; i < g.triCount; i++) offset[i + 1] = offset[i] + (size_t)getSplitCount(prio[i], totalPriority, g.triCount, s.splitFactor);
    out.bounds.resize(offset[g.triCount]);
    out.originalTriIds.resize(offset[g.triCount]);

    Box globalBox = Box::empty();
    for (int i = 0; i < g.triCount; i++) {
        Tri t = g.tri(i);
        globalBox.grow(t.p0); globalBox.grow(t.p1); globalBox.grow(t.p2);
    }
    float globalSize[3] = {globalBox.size(0), globalBox.size(1), globalBox.size(2)};

    struct Item { Box box; int splits; };
    chunked([&](int b0, int e0) {
    std::vector<Item> stack(64 + 4096);
    for (int i = b0; i < e0; i++) {
        Tri tri = g.tri(i);
        size_t counter = offset[i];
        int splitCount = (int)(offset[i + 1] - offset[i]);
        int sp = 0;
        stack[sp++] = {boxFromTri(tri), splitCount};
        while (sp > 0) {
            Item it = stack[--sp];
            if (it.splits == 1) {
                out.bounds[counter] = it.box;
                out.originalTriIds[counter] = i;
                counter++;
                continue;
            }
            int axis = it.box.largestAxis();
            float largestExtent = it.box.largestExtent();
            float nodeSize = getNodeSize(largestExtent, globalSize[axis]);
            if (nodeSize >= largestExtent - 0.0001f) nodeSize *= 0.5f;

            float midPos = (it.box.mn[axis] + it.box.mx[axis]) * 0.5f;
            float index = nearbyintf((midPos - globalBox.mn[axis]) / nodeSize); // MathF.Round: half to even
            float splitPos = globalBox.mn[axis] + index * nodeSize;

            Box lBox, rBox;
            triSplit(tri, axis, splitPos, lBox, rBox);
            lBox.clip(it.box);
            rBox.clip(it.box);

            float leftExtent = lBox.largestExtent();
            float rightExtent = rBox.largestExtent();
            int leftCount = csFloatToInt((float)it.splits * (leftExtent / (leftExtent + rightExtent)));
            leftCount = std::min(std::max(leftCount, 1), it.splits - 1);
            int rightCount = it.splits - leftCount;

            if (sp + 2 > (int)stack.size()) stack.resize(stack.size() * 2);
            stack[sp++] = {rBox, rightCount};
            stack[sp++] = {lBox, leftCount};
        }
    }
    });
}

// ---------------------------------------------------------------- BLAS.GetBuildData
struct BuildData {
    Fragments frags;
    std::vector<float> rightCostsAccum;
    std::vector<int> partitionAux;
    std::vector<uint8_t> fragLeftTable;
    std::vector<int> sorted[3];
    int n() const { return (int)frags.bounds.size(); }
};

// Algorithms.RadixSort: 3 x 11-bit LSD passes (stable).
static void radixSortFragments(const Fragments& f, int axis, std::vector<int>& output) {
    const int n = (int)f.bounds.size();
    const int radixSize = 11, binSize = 1 << radixSize, mask = binSize - 1;
    std::vector<uint32_t> keys(n);
    for (int i = 0; i < n; i++) keys[i] = floatToKey(f.bounds[i].mn[axis] + f.bounds[i].mx[axis]);
    std::vector<int> prefix(binSize * 3, 0);
    for (int i = 0; i < n; i++) {
        uint32_t k = keys[i];
        prefix[(k & mask)]++;
        prefix[((k >> 11) & mask) + binSize]++;
        prefix[((k >> 22) & mask) + 2 * binSize]++;
    }
    for (int p = 0; p < 3; p++) {
        int sum = 0;
        for (int i = 0; i < binSize; i++) { int t = prefix[i + p * binSize]; prefix[i + p * binSize] = sum; sum += t; }
    }
    std::vector<int> a(n), b(n);
    for (int i = 0; i < n; i++) a[i] = i;
    std::vector<int>* in = &a; std::vector<int>* outp = &b;
    for (int p = 0; p < 3; p++) {
        for (int j = 0; j < n; j++) {
            int el = (*in)[j];
            uint32_t r = (keys[el] >> (p * radixSize)) & mask;
            (*outp)[prefix[r + p * binSize]++] = el;
        }
        std::swap(in, outp);
    }
    output = *in; // after 3 passes the result lives in the buffer 'in' points to
}

static Box computeBoundingBox(int start, int count, const BuildData& bd, int axis) {
    Box box = Box::empty();
    const int* ids = bd.sorted[axis].data() + start;
    for (int i = 0; i < count; i++) box.grow(bd.frags.bounds[ids[i]]);
    return box;
}

// Algorithms.StablePartition(source, auxiliary, bitArray)
static int stablePartition(int* source, int count, int* aux, const uint8_t* table) {
    int l = 0, r = 0;
    for (int i = 0; i < count; i++) {
        int id = source[i];
        if (table[id]) source[l++] = id; else aux[r++] = id;
    }
    memcpy(source + l, aux, sizeof(int) * (size_t)r);
    return l;
}

struct ObjectSplit { int axis; int splitIndex; float newCost; bool valid; };

// BLAS.TrySplit, Bvh/BLAS.cs:730-873
static ObjectSplit trySplit(const GpuBlasNode& parent, BuildData& bd, const Settings& s) {
    ObjectSplit none = {0, 0, 0.0f, false};
    Box parentBox = {{parent.Min[0], parent.Min[1], parent.Min[2]}, {parent.Max[0], parent.Max[1], parent.Max[2]}};
    if (parent.TriCount <= s.stopSplittingThreshold) return none;

    const int start = parent.TriStartOrChild;
    const int end = parent.TriStartOrChild + parent.TriCount;

    ObjectSplit best = {0, 0, FLT_MAX, true};
    float* rightCostsAccum = bd.rightCostsAccum.data();
    const Box* fragBounds = bd.frags.bounds.data();

    for (int axis = 0; axis < 3; axis++) {
        const int* ids = bd.sorted[axis].data();
        int firstRight = start + 1;

        Box rightBoxAccum = Box::empty();
        float rightCounter = 0.0f;
        for (int i = end - 1; i >= firstRight; i--) {
            rightCounter++;
            rightBoxAccum.grow(fragBounds[ids[i]]);
            float rightCost = rightBoxAccum.halfArea() * rightCounter;
            rightCostsAccum[i] = rightCost;
            if (rightCost >= best.newCost) { firstRight = i + 1; break; }
        }

        Box leftBoxAccum = Box::empty();
        float leftCounter = (float)(firstRight - start) - 1.0f;
        for (int i = start; i < firstRight - 1; i++) leftBoxAccum.grow(fragBounds[ids[i]]);
        for (int i = firstRight - 1; i < end - 1; i++) {
            int splitIndex = i + 1;
            leftCounter++;
            leftBoxAccum.grow(fragBounds[ids[i]]);
            float leftCost = leftBoxAccum.halfArea() * leftCounter;
            float rightCost = rightCostsAccum[splitIndex];
            float cost = leftCost + rightCost;
            if (cost < best.newCost) {
                best.splitIndex = splitIndex;
                best.axis = axis;
                best.newCost = cost;
            } else if (leftCost >= best.newCost) {
                break;
            }
        }
    }

    if (best.newCost == FLT_MAX) {
        // Degenerate input (non-finite costs): the reference would index out of range.
        // Robustness guard: median split on axis 0.
        best.axis = 0;
        best.splitIndex = start + parent.TriCount / 2;
    }

    if (parent.TriCount <= s.maxLeafTriangleCount) {
        float notSplitCost = s.triangleCost * (float)parent.TriCount;
        best.newCost = 1.0f /*TRAVERSAL_COST*/ + (s.triangleCost * best.newCost / parentBox.halfArea());
        if (best.newCost >= notSplitCost) return none;
    }

    Box leftBox = computeBoundingBox(start, best.splitIndex - start, bd, best.axis);
    Box rightBox = computeBoundingBox(best.splitIndex, end - best.splitIndex, bd, best.axis);
    bool leftSmaller = leftBox.halfArea() < rightBox.halfArea();
    bool swapSides = leftSmaller; // larger child goes left

    uint8_t* table = bd.fragLeftTable.data();
    int* ids = bd.sorted[best.axis].data();
    for (int i = start; i < best.splitIndex; i++) table[ids[i]] = !swapSides;
    for (int i = best.splitIndex; i < end; i++) table[ids[i]] = swapSides;

    int* aux = bd.partitionAux.data() + start;
    if (swapSides) best.splitIndex = start + stablePartition(ids + start, parent.TriCount, aux, table);
    stablePartition(bd.sorted[(best.axis + 1) % 3].data() + start, parent.TriCount, aux, table);
    stablePartition(bd.sorted[(best.axis + 2) % 3].data() + start, parent.TriCount, aux, table);
    return best;
}


// ---- wide variant of TrySplit for the few huge nodes at the top of the tree --------------------------------------------------
// Same decisions as trySplit, bit for bit: the six box scans (prefix = left cost, suffix = right cost, per axis) are
// computed in full by up to six threads (min/max accumulation is exact, so a scan computed in full equals the
// reference's early-terminated one wherever the reference looks at it); the reference's sweep loop with its early-outs
// then runs over the precomputed costs. The two child boxes and the three stable partitions run concurrently as well.
struct WideScratch {
    std::vector<float> L[3], R[3];   // indexed by absolute fragment position
    void ensure(int n) { for (int a = 0; a < 3; a++) { if ((int)L[a].size() < n) { L[a].resize(n); R[a].resize(n); } } }
};

template <class F>
static void runTasks(int taskCount, int threads, F&& f) {
    const int workers = std::max(1, std::min(threads, taskCount));
    if (workers == 1) { for (int t = 0; t < taskCount; t++) f(t); return; }
    std::atomic<int> next(0);
    std::vector<std::thread> pool;
    for (int w = 0; w < workers - 1; w++) pool.emplace_back([&]() { for (;;) { int t = next.fetch_add(1); if (t >= taskCount) break; f(t); } });
    for (;;) { int t = next.fetch_add(1); if (t >= taskCount) break; f(t); }
    for (auto& th : pool) th.join();
}

static ObjectSplit trySplitWide(const GpuBlasNode& parent, BuildData& bd, const Settings& s, WideScratch& ws) {
    ObjectSplit none = {0, 0, 0.0f, false};
    Box parentBox = {{parent.Min[0], parent.Min[1], parent.Min[2]}, {parent.Max[0], parent.Max[1], parent.Max[2]}};
    if (parent.TriCount <= s.stopSplittingThreshold) return none;
    const int start = parent.TriStartOrChild;
    const int end = parent.TriStartOrChild + parent.TriCount;
    const Box* fragBounds = bd.frags.bounds.data();
    ws.ensure(bd.n());

    runTasks(6, s.threads, [&](int task) {
        const int axis = task >> 1;
        const int* ids = bd.sorted[axis].data();
        if (task & 1) {           // suffix: R[i] = halfArea(box of [i, end)) * (end - i)
            Box acc = Box::empty();
            float counter = 0.0f;
            float* R = ws.R[axis].data();
            for (int i = end - 1; i >= start + 1; i--) { counter++; acc.grow(fragBounds[ids[i]]); R[i] = acc.halfArea() * counter; }
        } else {                  // prefix: L[i] = halfArea(box of [start, i]) * (i - start + 1)
            Box acc = Box::empty();
            float counter = 0.0f;
            float* L = ws.L[axis].data();
            for (int i = start; i < end - 1; i++) { counter++; acc.grow(fragBounds[ids[i]]); L[i] = acc.halfArea() * counter; }
        }
    });

    ObjectSplit best = {0, 0, FLT_MAX, true};
    for (int axis = 0; axis < 3; axis++) {   // BLAS.TrySplit's sweep, reading the precomputed costs
        const float* L = ws.L[axis].data();
        const float* R = ws.R[axis].data();
        int firstRight = start + 1;
        for (int i = end - 1; i >= firstRight; i--)
            if (R[i] >= best.newCost) { firstRight = i + 1; break; }
        for (int i = firstRight - 1; i < end - 1; i++) {
            const int splitIndex = i + 1;
            const float leftCost = L[i];
            const float cost = leftCost + R[splitIndex];
            if (cost < best.newCost) {
                best.splitIndex = splitIndex;
                best.axis = axis;
                best.newCost = cost;
            } else if (leftCost >= best.newCost) {
                break;
            }
        }
    }
    if (best.newCost == FLT_MAX) {
        best.axis = 0;
        best.splitIndex = start + parent.TriCount / 2;
    }
    if (parent.TriCount <= s.maxLeafTriangleCount) {
        float notSplitCost = s.triangleCost * (float)parent.TriCount;
        best.newCost = 1.0f + (s.triangleCost * best.newCost / parentBox.halfArea());
        if (best.newCost >= notSplitCost) return none;
    }

    Box childBox[2];
    runTasks(2, s.threads, [&](int t) {
        childBox[t] = t == 0 ? computeBoundingBox(start, best.splitIndex - start, bd, best.axis)
                             : computeBoundingBox(best.splitIndex, end - best.splitIndex, bd, best.axis);
    });
    const bool swapSides = childBox[0].halfArea() < childBox[1].halfArea();   // larger child goes left

    uint8_t* table = bd.fragLeftTable.data();
    int* ids = bd.sorted[best.axis].data();
    const int split0 = best.splitIndex;
    runTasks(2, s.threads, [&](int t) {
        if (t == 0) for (int i = start; i < split0; i++) table[ids[i]] = !swapSides;
        else for (int i = split0; i < end; i++) table[ids[i]] = swapSides;
    });

    // three independent id arrays: each needs its own auxiliary range
    std::vector<int> auxB(parent.TriCount), auxC(parent.TriCount);
    int newSplit = best.splitIndex;
    runTasks(3, s.threads, [&](int t) {
        if (t == 0) { if (swapSides) newSplit = start + stablePartition(ids + start, parent.TriCount, bd.partitionAux.data() + start, table); }
        else if (t == 1) stablePartition(bd.sorted[(best.axis + 1) % 3].data() + start, parent.TriCount, auxB.data(), table);
        else stablePartition(bd.sorted[(best.axis + 2) % 3].data() + start, parent.TriCount, auxC.data(), table);
    });
    best.splitIndex = newSplit;
    return best;
}

// ---------------------------------------------------------------- BLAS.Build
struct BuildResult {
    std::vector<GpuBlasNode> nodes;
    int requiredStackSize = 0;
};

static void setBounds(GpuBlasNode& n, const Box& b) {
    for (int i = 0; i < 3; i++) { n.Min[i] = b.mn[i]; n.Max[i] = b.mx[i]; }
}

struct BuildTask { int parentNodeId; int newNodesId; };

static void processSubtree(BuildResult& blas, BuildData& bd, const Settings& s, BuildTask root,
                           std::vector<BuildTask>* spill, int spillThreshold) {
    std::vector<BuildTask> stack;
    stack.push_back(root);
    while (!stack.empty()) {
        BuildTask t = stack.back();
        stack.pop_back();
        GpuBlasNode& parent = blas.nodes[t.parentNodeId];
        setBounds(parent, computeBoundingBox(parent.TriStartOrChild, parent.TriCount, bd, 0));
        ObjectSplit split = trySplit(parent, bd, s);
        if (!split.valid) continue;

        GpuBlasNode left = {};
        left.TriStartOrChild = parent.TriStartOrChild;
        left.TriCount = split.splitIndex - left.TriStartOrChild;
        GpuBlasNode right = {};
        right.TriStartOrChild = split.splitIndex;
        right.TriCount = parent.TriCount - left.TriCount;

        int leftId = t.newNodesId, rightId = leftId + 1;
        blas.nodes[leftId] = left;
        blas.nodes[rightId] = right;
        parent.TriStartOrChild = leftId;
        parent.TriCount = 0;

        BuildTask lt = {leftId, rightId + 1};
        BuildTask rt = {rightId, rightId + (2 * left.TriCount - 1)};
        // Sub-tasks touch disjoint ranges of every array, so any execution order
        // yields the same tree (BLAS.cs:221-231 runs them on separate threads).
        if (spill && std::min(left.TriCount, right.TriCount) >= spillThreshold) {
            spill->push_back(lt);
            spill->push_back(rt);
        } else {
            stack.push_back(rt);
            stack.push_back(lt);
        }
    }
}

static int computeRequiredStackSize(const BuildResult& blas, int nodeId) {
    const GpuBlasNode& l = blas.nodes[nodeId];
    const GpuBlasNode& r = blas.nodes[nodeId + 1];
    bool tl = !(l.TriCount > 0), tr = !(r.TriCount > 0);
    if (tl || tr) {
        if (tl && tr) {
            int a = computeRequiredStackSize(blas, l.TriStartOrChild);
            int b = computeRequiredStackSize(blas, r.TriStartOrChild);
            return std::max(a, b) + 1;
        }
        return computeRequiredStackSize(blas, tl ? l.TriStartOrChild : r.TriStartOrChild);
    }
    return 0;
}

static double computeGlobalSAH(const BuildResult& blas, const Settings& s) {
    double cost = 0.0;
    double rootArea = 1.0 / (double)nodeHalfArea(blas.nodes[1]);
    std::vector<int> stack;
    stack.push_back(1);
    while (!stack.empty()) {
        const GpuBlasNode& n = blas.nodes[stack.back()];
        stack.pop_back();
        double prob = (double)nodeHalfArea(n) * rootArea;
        if (n.TriCount > 0) {
            cost += (double)(s.triangleCost * (float)n.TriCount) * prob; // float*int in C# = float, then * double
        } else {
            cost += 1.0 * prob;
            stack.push_back(n.TriStartOrChild + 1);
            stack.push_back(n.TriStartOrChild);
        }
    }
    return cost;
}

static void collapseDeepestLevel(BuildResult& blas, const Settings& s, int newStackSize, bool firstPass,
                                 double& nextCollapseCost, int parentId, int stackSize) {
    GpuBlasNode& parent = blas.nodes[parentId];
    const int childId = parent.TriStartOrChild;
    GpuBlasNode& l = blas.nodes[childId];
    GpuBlasNode& r = blas.nodes[childId + 1];

    if (!(l.TriCount > 0)) collapseDeepestLevel(blas, s, newStackSize, firstPass, nextCollapseCost, childId, stackSize + 1);
    if (!(r.TriCount > 0)) collapseDeepestLevel(blas, s, newStackSize, firstPass, nextCollapseCost, childId + 1, stackSize + 1);

    if (l.TriCount > 0 && r.TriCount > 0) {
        if (stackSize > newStackSize && !firstPass) {
            parent.TriStartOrChild = l.TriStartOrChild;
            parent.TriCount = l.TriCount + r.TriCount;
        }
        if ((stackSize == newStackSize && !firstPass) || (stackSize > newStackSize && firstPass)) {
            if ((float)(l.TriCount + r.TriCount) > s.stackOptMaxLeafTriangleCount) {
                nextCollapseCost = (double)FLT_MAX;
                return;
            }
            double leavesCost = (double)s.triangleCost * ((double)l.TriCount * (double)nodeHalfArea(l) + (double)r.TriCount * (double)nodeHalfArea(r));
            double newParentLeafCost = (double)s.triangleCost * (double)(l.TriCount + r.TriCount);
            nextCollapseCost += ((double)nodeHalfArea(parent) * (newParentLeafCost - 1.0) - leavesCost) / (double)nodeHalfArea(blas.nodes[1]);
        }
    }
}

static void optimizeStackSize(BuildResult& blas, const Settings& s) {
    blas.requiredStackSize = computeRequiredStackSize(blas, 2);
    if (blas.requiredStackSize < s.stackOptThreshold) return;
    double currentCost = computeGlobalSAH(blas, s);
    double addedCost = 0.0;
    collapseDeepestLevel(blas, s, blas.requiredStackSize - 1, true, addedCost, 1, 0);
    double increasePercent = addedCost / currentCost;
    while (increasePercent <= (double)s.stackOptSahIncreaseAcceptance && blas.requiredStackSize > 0) {
        collapseDeepestLevel(blas, s, --blas.requiredStackSize, false, addedCost, 1, 0);
        increasePercent = addedCost / currentCost;
    }
}

static int removeEmptySubtrees(BuildResult& blas) {
    int nodeCounter = 2;
    std::vector<int> stack;
    stack.push_back(1);
    while (!stack.empty()) {
        int pid = stack.back();
        stack.pop_back();
        GpuBlasNode& parent = blas.nodes[pid];
        GpuBlasNode l = blas.nodes[parent.TriStartOrChild];
        GpuBlasNode r = blas.nodes[parent.TriStartOrChild + 1];
        int lid = nodeCounter, rid = nodeCounter + 1;
        blas.nodes[lid] = l;
        blas.nodes[rid] = r;
        parent.TriStartOrChild = lid;
        nodeCounter += 2;
        if (!(r.TriCount > 0)) stack.push_back(rid);
        if (!(l.TriCount > 0)) stack.push_back(lid);
    }
    return nodeCounter;
}

static int buildBlas(BuildResult& blas, BuildData& bd, const Settings& s) {
    const bool timing = getenv("IDKHOST_TIMING") != nullptr;
    auto now = []() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    double t0 = now(), t1;
    auto lap = [&](const char* what) { if (timing) { t1 = now(); fprintf(stderr, "[idkhost]   %-14s %8.1f ms\n", what, (t1 - t0) * 1e3); t0 = t1; } };
    blas.nodes[0] = GpuBlasNode{};
    GpuBlasNode& root = blas.nodes[1];
    root = GpuBlasNode{};
    root.TriStartOrChild = 0;
    root.TriCount = bd.n();

    if (s.threads > 1 && bd.n() >= (1 << 14)) {
        // Task pool over the tree (BLAS.cs:221-231 runs sub-tasks on separate threads): a worker takes a node; a node
        // above the threshold is split once and its two children become tasks, a smaller one is finished serially.
        // Sub-tasks touch disjoint ranges of every array, so any execution order yields the same tree. The one or two
        // levels where there are fewer nodes than workers use the wide split (all threads on one node).
        const int threshold = std::max(1 << 13, bd.n() / (s.threads * 8)); // BLAS.THREADED_RECURSION_THRESHOLD
        const int wideThreshold = std::max(2 * threshold, bd.n() / 3);
        std::mutex mu;
        std::condition_variable cv;
        std::vector<BuildTask> queue;
        int active = 0;
        queue.push_back({1, 2});
        auto splitOnce = [&](BuildTask t, WideScratch* wide) {
            GpuBlasNode& parent = blas.nodes[t.parentNodeId];
            setBounds(parent, computeBoundingBox(parent.TriStartOrChild, parent.TriCount, bd, 0));
            ObjectSplit split = wide ? trySplitWide(parent, bd, s, *wide) : trySplit(parent, bd, s);
            if (!split.valid) return;
            GpuBlasNode left = {}; left.TriStartOrChild = parent.TriStartOrChild; left.TriCount = split.splitIndex - left.TriStartOrChild;
            GpuBlasNode right = {}; right.TriStartOrChild = split.splitIndex; right.TriCount = parent.TriCount - left.TriCount;
            int leftId = t.newNodesId, rightId = leftId + 1;
            blas.nodes[leftId] = left; blas.nodes[rightId] = right;
            parent.TriStartOrChild = leftId; parent.TriCount = 0;
            std::lock_guard<std::mutex> lk(mu);
            queue.push_back({leftId, rightId + 1});
            queue.push_back({rightId, rightId + (2 * left.TriCount - 1)});
        };
        {   // top of the tree: all threads on one node at a time
            WideScratch wide;
            for (;;) {
                size_t pick = queue.size();
                for (size_t i = 0; i < queue.size(); i++)
                    if (blas.nodes[queue[i].parentNodeId].TriCount >= wideThreshold) { pick = i; break; }
                if (pick == queue.size()) break;
                BuildTask t = queue[pick];
                queue.erase(queue.begin() + pick);
                splitOnce(t, &wide);
            }
        }
        lap("breadth");
        std::vector<std::thread> pool;
        for (int i = 0; i < s.threads; i++) {
            pool.emplace_back([&]() {
                std::unique_lock<std::mutex> lk(mu);
                for (;;) {
                    while (queue.empty() && active > 0) cv.wait(lk);
                    if (queue.empty()) break;                       // nothing queued and nobody working: done
                    BuildTask t = queue.back();
                    queue.pop_back();
                    active++;
                    lk.unlock();
                    if (blas.nodes[t.parentNodeId].TriCount >= 2 * threshold) splitOnce(t, nullptr);
                    else processSubtree(blas, bd, s, t, nullptr, 0);
                    lk.lock();
                    active--;
                    cv.notify_all();
                }
                cv.notify_all();
            });
        }
        for (auto& th : pool) th.join();
    } else {
        processSubtree(blas, bd, s, {1, 2}, nullptr, 0);
    }

    lap("subtrees");
    if (root.TriCount > 0) {
        blas.nodes[2] = root;
        blas.nodes[3] = root;
        root.TriStartOrChild = 2;
        root.TriCount = 0;
    }
    optimizeStackSize(blas, s);
    lap("stack opt");
    const int used = removeEmptySubtrees(blas);
    lap("compact");
    return used;
}

// ---------------------------------------------------------------- GetUnindexedTriangles
static std::vector<int> uniqueTriIds(const GpuBlasNode& leaf, const BuildData& bd) {
    std::vector<int> ids(leaf.TriCount);
    for (int i = 0; i < leaf.TriCount; i++) ids[i] = bd.frags.originalTriIds[bd.sorted[0][leaf.TriStartOrChild + i]];
    std::sort(ids.begin(), ids.end());
    ids.erase(std::unique(ids.begin(), ids.end()), ids.end());
    return ids;
}

static bool contains(const std::vector<int>& v, int x) { return std::find(v.begin(), v.end(), x) != v.end(); }

// PreSplitting.GetUnindexedTriangles, Bvh/PreSplitting.cs:169-273
static void unindexPreSplit(BuildResult& blas, const BuildData& bd, const Geometry& g, std::vector<GpuBlasTriangle>& tris) {
    tris.assign(bd.n(), GpuBlasTriangle{});
    int counter = 0;
    std::vector<int> stack;
    stack.push_back(2);
    while (!stack.empty()) {
        int top = stack.back();
        stack.pop_back();
        GpuBlasNode& l = blas.nodes[top];
        GpuBlasNode& r = blas.nodes[top + 1];
        bool ll = l.TriCount > 0, rl = r.TriCount > 0;
        if (ll && rl) {
            std::vector<int> lu = uniqueTriIds(l, bd), ru = uniqueTriIds(r, bd);
            int onlyLeft = 0, backwards = 0;
            for (size_t i = 0; i < lu.size(); i++) {
                int id = lu[i];
                if (contains(ru, id)) tris[counter + (int)lu.size() - backwards++ - 1] = g.tris[id];
                else tris[counter + onlyLeft++] = g.tris[id];
            }
            int onlyRight = 0;
            for (size_t i = 0; i < ru.size(); i++) {
                int id = ru[i];
                if (!contains(lu, id)) tris[counter + (int)lu.size() + onlyRight++] = g.tris[id];
            }
            l.TriStartOrChild = counter;
            l.TriCount = (int)lu.size();
            r.TriStartOrChild = counter + onlyLeft;
            r.TriCount = (int)ru.size();
            counter += (r.TriStartOrChild + r.TriCount) - l.TriStartOrChild;
        } else if (ll || rl) {
            GpuBlasNode& leaf = ll ? l : r;
            std::vector<int> u = uniqueTriIds(leaf, bd);
            for (size_t i = 0; i < u.size(); i++) tris[counter + (int)i] = g.tris[u[i]];
            leaf.TriStartOrChild = counter;
            leaf.TriCount = (int)u.size();
            counter += (int)u.size();
        }
        if (!rl) stack.push_back(r.TriStartOrChild);
        if (!ll) stack.push_back(l.TriStartOrChild);
    }
    tris.resize(counter);
}

// BLAS.GetUnindexedTriangles, Bvh/BLAS.cs:441-466
static void unindexPlain(BuildResult& blas, const BuildData& bd, const Geometry& g, std::vector<GpuBlasTriangle>& tris) {
    tris.assign(bd.n(), GpuBlasTriangle{});
    int counter = 0;
    for (size_t i = 2; i < blas.nodes.size(); i++) {
        GpuBlasNode& n = blas.nodes[i];
        if (n.TriCount > 0) {
            // A root that did not split is listed twice (nodes 2 and 3); the second copy's triangles fall past the
            // array's end and are dropped rather than written out of bounds.
            for (int j = 0; j < n.TriCount && counter + j < (int)tris.size(); j++) tris[counter + j] = g.tris[bd.sorted[0][n.TriStartOrChild + j]];
            n.TriStartOrChild = counter;
            counter += n.TriCount;
        }
    }
}

} // namespace

struct IdkBlasBuild {
    std::vector<GpuBlasNode> nodes;
    std::vector<GpuBlasTriangle> tris;
    int requiredStackSize = 0;
    int fragmentCount = 0;
    double sah = 0.0;
};

extern "C" {

// Settings blob mirrors BLAS.BuildSettings (BLAS.cs:31-48) + PreSplitting.Settings (PreSplitting.cs:17-24).
struct IdkBlasBuildSettings {
    int32_t StopSplittingThreshold;
    int32_t MaxLeafTriangleCount;
    float   TriangleCost;
    int32_t StackOptThreshold;
    float   StackOptSahIncreaseAcceptance;
    float   SplitFactor;
    int32_t DoPreSplit;   // !IsRefittable (BVH.cs:324-333)
    int32_t Threads;
};

__attribute__((visibility("default")))
void idkhost_default_build_settings(IdkBlasBuildSettings* s) {
    s->StopSplittingThreshold = 1;
    s->MaxLeafTriangleCount = 2;
    s->TriangleCost = 1.1f;
    s->StackOptThreshold = 16;
    s->StackOptSahIncreaseAcceptance = 0.0009745f;
    s->SplitFactor = 0.3f;
    s->DoPreSplit = 1;
    s->Threads = 1;
}

// One BLAS: BVH.BlasesBuild loop body, Bvh/BVH.cs:315-377.
__attribute__((visibility("default")))
IdkBlasBuild* idkhost_blas_build(const PackedVec3* positions, uint64_t vertexCount,
                                 const GpuBlasTriangle* triangles, uint64_t triangleCount,
                                 const IdkBlasBuildSettings* settings) {
    (void)vertexCount;
    Settings s;
    s.stopSplittingThreshold = settings->StopSplittingThreshold;
    s.maxLeafTriangleCount = settings->MaxLeafTriangleCount;
    s.triangleCost = settings->TriangleCost;
    s.stackOptThreshold = settings->StackOptThreshold;
    s.stackOptSahIncreaseAcceptance = settings->StackOptSahIncreaseAcceptance;
    s.splitFactor = settings->SplitFactor;
    s.doPreSplit = settings->DoPreSplit;
    s.threads = std::max(1, settings->Threads);

    const bool timing = getenv("IDKHOST_TIMING") != nullptr;
    auto now = []() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    double t0 = now(), t1;
    auto lap = [&](const char* what) { if (timing) { t1 = now(); fprintf(stderr, "[idkhost] %-14s %8.1f ms\n", what, (t1 - t0) * 1e3); t0 = t1; } };
    Geometry g = {positions, triangles, (int)triangleCount};
    BuildData bd;
    if (s.doPreSplit) {
        preSplit(g, s, bd.frags);
    } else {
        bd.frags.bounds.resize(g.triCount);
        for (int i = 0; i < g.triCount; i++) bd.frags.bounds[i] = boxFromTri(g.tri(i));
    }
    lap("presplit");
    const int n = bd.n();
    bd.fragLeftTable.assign(n, 0);
    bd.rightCostsAccum.assign(n, 0.0f);
    bd.partitionAux.assign(n, 0);
    if (s.threads > 1 && n >= (1 << 16)) {
        std::thread t0([&]() { radixSortFragments(bd.frags, 0, bd.sorted[0]); });
        std::thread t1([&]() { radixSortFragments(bd.frags, 1, bd.sorted[1]); });
        radixSortFragments(bd.frags, 2, bd.sorted[2]);
        t0.join(); t1.join();
    } else {
        for (int a = 0; a < 3; a++) radixSortFragments(bd.frags, a, bd.sorted[a]);
    }

    lap("radix sort");
    BuildResult blas;
    blas.nodes.assign(std::max(2 * n, 4), GpuBlasNode{});
    int used = buildBlas(blas, bd, s);
    blas.nodes.resize(used);
    lap("build+stackopt");

    IdkBlasBuild* out = new IdkBlasBuild();
    if (s.doPreSplit) unindexPreSplit(blas, bd, g, out->tris);
    else unindexPlain(blas, bd, g, out->tris);
    lap("unindex");
    out->sah = computeGlobalSAH(blas, s);
    lap("sah");
    out->nodes = std::move(blas.nodes);
    out->requiredStackSize = blas.requiredStackSize;
    out->fragmentCount = n;
    return out;
}

__attribute__((visibility("default"))) uint64_t idkhost_blas_node_count(const IdkBlasBuild* b) { return b->nodes.size(); }
__attribute__((visibility("default"))) uint64_t idkhost_blas_triangle_count(const IdkBlasBuild* b) { return b->tris.size(); }
__attribute__((visibility("default"))) int32_t idkhost_blas_required_stack_size(const IdkBlasBuild* b) { return b->requiredStackSize; }
__attribute__((visibility("default"))) int32_t idkhost_blas_fragment_count(const IdkBlasBuild* b) { return b->fragmentCount; }
__attribute__((visibility("default"))) double idkhost_blas_sah(const IdkBlasBuild* b) { return b->sah; }
__attribute__((visibility("default")))
void idkhost_blas_copy(const IdkBlasBuild* b, GpuBlasNode* nodes, GpuBlasTriangle* tris) {
    memcpy(nodes, b->nodes.data(), b->nodes.size() * sizeof(GpuBlasNode));
    memcpy(tris, b->tris.data(), b->tris.size() * sizeof(GpuBlasTriangle));
}
__attribute__((visibility("default"))) void idkhost_blas_free(IdkBlasBuild* b) { delete b; }

// The builder's cube root (include/idk_cbrtf.h) over an array, for tests that compare it with the C library.
__attribute__((visibility("default")))
void idkhost_cbrtf(const float* x, float* out, uint64_t count) {
    for (uint64_t i = 0; i < count; i++) out[i] = idk_cbrtf(x[i]);
}

} // extern "C"

// ---------------------------------------------------------------- TLAS (Bvh/TLAS.cs:28-141, serial PLOC)
namespace {

static inline uint32_t insertTwoZeros(uint32_t v) {   // MyMath.InsertTwoZerosAfterEachBit
    v = (v * 0x00010001u) & 0xFF0000FFu;
    v = (v * 0x00000101u) & 0x0F00F00Fu;
    v = (v * 0x00000011u) & 0xC30C30C3u;
    v = (v * 0x00000005u) & 0x49249249u;
    return v;
}
static inline uint32_t morton30(float x, float y, float z) {   // MyMath.GetMortonCode30
    auto q = [](float f) { float s = f * 1024.0f; uint32_t u = s <= 0.0f ? 0u : (s >= 4294967040.0f ? 0xFFFFFFFFu : (uint32_t)s); return std::min(u, 1023u); };
    return (insertTwoZeros(q(x)) << 2) | (insertTwoZeros(q(y)) << 1) | insertTwoZeros(q(z));
}
static inline Box tlasBox(const GpuTlasNode& n) { return {{n.Min[0], n.Min[1], n.Min[2]}, {n.Max[0], n.Max[1], n.Max[2]}}; }
static inline void tlasSetBounds(GpuTlasNode& n, const Box& b) { for (int i = 0; i < 3; i++) { n.Min[i] = b.mn[i]; n.Max[i] = b.mx[i]; } }

static int findBestMatch(const GpuTlasNode* nodes, int start, int end, int nodeIndex) {
    float smallestArea = FLT_MAX;
    int best = -1;
    Box nodeBox = tlasBox(nodes[nodeIndex]);
    for (int i = start; i < end; i++) {
        if (i == nodeIndex) continue;
        Box merged = nodeBox;
        merged.grow(tlasBox(nodes[i]));
        float area = merged.halfArea();
        if (area < smallestArea) { smallestArea = area; best = i; }
    }
    return best;
}

} // namespace

extern "C" {

// Box.Transformed(localBounds, modelMatrix) (Shapes/Box.cs:166-175): 8 corners through the (column-vector) 3x4 model matrix.
__attribute__((visibility("default")))
void idkhost_transform_box(const float mn[3], const float mx[3], const float model3x4[12], float outMin[3], float outMax[3]) {
    Box b = Box::empty();
    for (int i = 0; i < 8; i++) {
        float x = (i & 1) ? mx[0] : mn[0], y = (i & 2) ? mx[1] : mn[1], z = (i & 4) ? mx[2] : mn[2];
        // OpenTK Vector4 * Matrix4 (row vector): x*Row0 + y*Row1 + z*Row2 + w*Row3; Row_k.c = model3x4[c][k]
        V3 p;
        p.x = x * model3x4[0] + y * model3x4[1] + z * model3x4[2] + 1.0f * model3x4[3];
        p.y = x * model3x4[4] + y * model3x4[5] + z * model3x4[6] + 1.0f * model3x4[7];
        p.z = x * model3x4[8] + y * model3x4[9] + z * model3x4[10] + 1.0f * model3x4[11];
        b.grow(p);
    }
    for (int i = 0; i < 3; i++) { outMin[i] = b.mn[i]; outMax[i] = b.mx[i]; }
}

// TLAS.Build: boxes = primitiveCount x {min[3], max[3]} (world space), nodes = 2*primitiveCount-1 GpuTlasNode, root at 0.
__attribute__((visibility("default")))
void idkhost_tlas_build(const float* boxes, int32_t primitiveCount, GpuTlasNode* nodes, int32_t searchRadius) {
    const int nodeCount = std::max(2 * primitiveCount - 1, 0);
    if (nodeCount == 0) return;
    std::vector<GpuTlasNode> temp(nodeCount);
    memset(nodes, 0, sizeof(GpuTlasNode) * (size_t)nodeCount);
    {
        GpuTlasNode* leaves = temp.data() + (nodeCount - primitiveCount);
        Box global = Box::empty();
        for (int i = 0; i < primitiveCount; i++) {
            Box b = {{boxes[6 * i], boxes[6 * i + 1], boxes[6 * i + 2]}, {boxes[6 * i + 3], boxes[6 * i + 4], boxes[6 * i + 5]}};
            global.grow(b);
            GpuTlasNode n = {};
            tlasSetBounds(n, b);
            n.IsLeafAndChildOrInstanceId = (1u << 31) | (uint32_t)i;
            leaves[i] = n;
        }
        std::vector<std::pair<uint32_t, int>> keyed(primitiveCount);
        for (int i = 0; i < primitiveCount; i++) {
            const GpuTlasNode& n = leaves[i];
            float c[3], m[3];
            for (int a = 0; a < 3; a++) {
                c[a] = (n.Max[a] + n.Min[a]) * 0.5f;
                float t = global.mx[a] - global.mn[a];
                m[a] = (c[a] - global.mn[a]) / t * (1.0f - 0.0f) + 0.0f;   // MyMath.MapToZeroOne / Remap
                if (t == 0.0f) m[a] = 0.0f;
            }
            keyed[i] = {morton30(m[0], m[1], m[2]), i};
        }
        std::stable_sort(keyed.begin(), keyed.end(), [](const std::pair<uint32_t, int>& a, const std::pair<uint32_t, int>& b) { return a.first < b.first; });
        for (int i = 0; i < primitiveCount; i++) nodes[nodeCount - primitiveCount + i] = leaves[keyed[i].second];
    }
    int activeRangeCount = primitiveCount, activeRangeEnd = nodeCount;
    std::vector<int> pref(primitiveCount);
    while (activeRangeCount > 1) {
        const int activeRangeStart = activeRangeEnd - activeRangeCount;
        for (int i = 0; i < activeRangeCount; i++) {
            int a = activeRangeStart + i;
            int s = std::max(a - searchRadius, activeRangeStart), e = std::min(a + searchRadius + 1, activeRangeEnd);
            pref[i] = findBestMatch(nodes, s, e, a) - activeRangeStart;
        }
        int merged = 0;
        for (int i = 0; i < activeRangeCount; i++) { int b = pref[i], c = pref[b]; if (i == c && i < b) merged += 2; }
        const int unmerged = activeRangeCount - merged, newNodes = merged / 2;
        int mergedHead = activeRangeEnd - merged;
        const int newBegin = mergedHead - unmerged - newNodes;
        int unmergedHead = newBegin;
        for (int i = 0; i < activeRangeCount; i++) {
            int b = pref[i], c = pref[b];
            int aId = i + activeRangeStart;
            if (i == c) {
                if (i < b) {
                    int bId = b + activeRangeStart;
                    temp[mergedHead] = nodes[aId];
                    temp[mergedHead + 1] = nodes[bId];
                    Box mb = tlasBox(temp[mergedHead]);
                    mb.grow(tlasBox(temp[mergedHead + 1]));
                    GpuTlasNode nn = {};
                    tlasSetBounds(nn, mb);
                    nn.IsLeafAndChildOrInstanceId = (uint32_t)mergedHead;
                    temp[unmergedHead++] = nn;
                    mergedHead += 2;
                }
            } else {
                temp[unmergedHead++] = nodes[aId];
            }
        }
        memcpy(nodes + newBegin, temp.data() + newBegin, sizeof(GpuTlasNode) * (size_t)(activeRangeEnd - newBegin));
        activeRangeCount -= merged / 2;
        activeRangeEnd -= merged;
    }
}

} // extern "C"
