// Device BLAS builder: BVH.BlasesBuild (Bvh/BVH.cs:300-377) for a batch of BLASes, node for node equal to the host
// mirror (host_mirror/bvh_build.cpp). Same decisions, same floats: the library builds with -fmad=false, and __fmaf_rn
// stands exactly where the host calls fmaf.
//
// Why a parallel build can give the host's bytes:
//  - Min/max accumulation is exact, and Box::grow keeps the later operand when two values compare equal (only +0 / -0
//    do), so a box fold is associative as long as every combine keeps the earlier part of the sequence on the left.
//    Every scan and reduction below does; the suffix scans run in the host's (descending) order.
//  - The split search evaluates every candidate (full prefix and suffix scans on all three axes) and takes the first
//    strict minimum in (axis, split index) order. The host's early-outs skip only candidates that cannot be strictly
//    better: suffix and prefix costs grow monotonically (half-areas of growing boxes times growing counts, both
//    rounded monotonically), so a skipped candidate costs at least the best found earlier in that order. Costs are
//    never NaN: inputs are finite and every BLAS box has a finite half-area (checked before the build).
//  - Node ids need no scheduling: the host pre-assigns them (children at newNodesId, subtrees at rightId + 1 and
//    rightId + 2 * leftCount - 1), so nodes split level by level, and subtrees finished by one thread each, land
//    where the host's depth-first build puts them. Sibling tasks touch disjoint ranges of every array.
//  - The reserved id ranges nest, and a subtree covers a contiguous fragment range, so pre-order is the order of
//    (range start, depth); stack optimisation, compaction and the SAH sums follow from sorted orders, subtree sizes
//    and prefix sums. Only the double sums (SAH, collapse costs) stay serial: one warp per BLAS streams the terms and
//    adds them one at a time in the host's order.
#pragma once
#include <cub/cub.cuh>
#include <cfloat>
#include <climits>
#include "../../include/idk_cbrtf.h"

namespace idkbb {

constexpr int NT = 512;                 // threads of the level-by-level split kernel
constexpr int ITEMS = 4;                // consecutive elements per thread in its scans
constexpr int CHUNK = NT * ITEMS;
constexpr int SMALL = 128;              // nodes of at most this many fragments are finished by one thread (k_split_small)
constexpr int MAX_FRAGMENTS = 1 << 24;  // the host counts fragments in floats; exact below this

struct Box { float mn[3], mx[3]; };

struct Settings {
    int   stopSplittingThreshold;
    int   maxLeafTriangleCount;
    float triangleCost;
    int   stackOptThreshold;
    float stackOptSahIncreaseAcceptance;
    float splitFactor;
};

struct Task { int blas, node, newNodes, depth; };

__device__ __forceinline__ float minN(float a, float b) { return a < b ? a : b; }
__device__ __forceinline__ float maxN(float a, float b) { return a > b ? a : b; }
__device__ __forceinline__ Box emptyBox() { return {{FLT_MAX, FLT_MAX, FLT_MAX}, {-FLT_MAX, -FLT_MAX, -FLT_MAX}}; }
// a comes first in the host's accumulation order
__device__ __forceinline__ Box comb(const Box& a, const Box& b) {
    Box r;
    #pragma unroll
    for (int i = 0; i < 3; i++) { r.mn[i] = minN(a.mn[i], b.mn[i]); r.mx[i] = maxN(a.mx[i], b.mx[i]); }
    return r;
}
__device__ __forceinline__ float halfArea(const Box& b) {
    const float sx = b.mx[0] - b.mn[0], sy = b.mx[1] - b.mn[1], sz = b.mx[2] - b.mn[2];
    return __fmaf_rn(sx + sy, sz, sx * sy);
}
__device__ __forceinline__ float nodeHalfArea(const GpuBlasNode& n) {
    const float sx = n.Max[0] - n.Min[0], sy = n.Max[1] - n.Min[1], sz = n.Max[2] - n.Min[2];
    return __fmaf_rn(sx + sy, sz, sx * sy);
}
__device__ __forceinline__ Box loadBox(const Box* b, int i) {
    const float2* p = (const float2*)(b + i);
    const float2 a = p[0], c = p[1], d = p[2];
    return {{a.x, a.y, c.x}, {c.y, d.x, d.y}};
}
__device__ __forceinline__ void setBounds(GpuBlasNode& n, const Box& b) {
    for (int i = 0; i < 3; i++) { n.Min[i] = b.mn[i]; n.Max[i] = b.mx[i]; }
}
__device__ __forceinline__ uint32_t floatToKey(float v) {
    const uint32_t f = __float_as_uint(v);
    return f ^ (uint32_t)(((int32_t)f >> 31) | (1 << 31));
}
// C# (int)float on x86-64 (cvttss2si): NaN / out of range -> INT_MIN
__device__ __forceinline__ int csFloatToInt(float f) {
    if (!(f > -2147483904.0f && f < 2147483648.0f)) return INT_MIN;
    return (int)f;
}

struct Tri { float p[3][3]; };
__device__ __forceinline__ Tri loadTri(const float* pos, int4 t) {
    Tri r;
    const int id[3] = {t.x, t.y, t.z};
    for (int v = 0; v < 3; v++) for (int a = 0; a < 3; a++) r.p[v][a] = pos[3 * (size_t)id[v] + a];
    return r;
}
__device__ __forceinline__ void growP(Box& b, const float* p) {
    for (int i = 0; i < 3; i++) { b.mn[i] = minN(b.mn[i], p[i]); b.mx[i] = maxN(b.mx[i], p[i]); }
}
__device__ __forceinline__ Box boxFromTri(const Tri& t) {
    Box b = {{t.p[0][0], t.p[0][1], t.p[0][2]}, {t.p[0][0], t.p[0][1], t.p[0][2]}};
    growP(b, t.p[1]);
    growP(b, t.p[2]);
    return b;
}
__device__ __forceinline__ float boxSize(const Box& b, int i) { return b.mx[i] - b.mn[i]; }
__device__ __forceinline__ int largestAxis(const Box& b) {
    int axis = 0;
    if (boxSize(b, 0) < boxSize(b, 1)) axis = 1;
    if (boxSize(b, axis) < boxSize(b, 2)) axis = 2;
    return axis;
}
__device__ __forceinline__ float largestExtent(const Box& b) { return maxN(boxSize(b, 0), maxN(boxSize(b, 1), boxSize(b, 2))); }

// ------------------------------------------------------------------------------------------------ pre-splitting
// PreSplitting.GetPriority with the shared cube root
__device__ float priority(const Tri& t) {
    const Box b = boxFromTri(t);
    const float le = largestExtent(b);
    const float extentPrio = le * le;
    const float e1[3] = {t.p[1][0] - t.p[0][0], t.p[1][1] - t.p[0][1], t.p[1][2] - t.p[0][2]};
    const float e2[3] = {t.p[2][0] - t.p[0][0], t.p[2][1] - t.p[0][1], t.p[2][2] - t.p[0][2]};
    const float cx = e1[1] * e2[2] - e1[2] * e2[1], cy = e1[2] * e2[0] - e1[0] * e2[2], cz = e1[0] * e2[1] - e1[1] * e2[0];
    const float triArea = sqrtf(cx * cx + cy * cy + cz * cz) * 0.5f;
    const float emptyAreaPrio = halfArea(b) * 2.0f - triArea;
    return idk_cbrtf(extentPrio * emptyAreaPrio);
}

// Triangle.Split (Shapes/Triangle.cs:47-92)
__device__ void triSplit(const Tri& t, int axis, float position, Box& lBox, Box& rBox) {
    lBox = emptyBox();
    rBox = emptyBox();
    const bool q[3] = {t.p[0][axis] <= position, t.p[1][axis] <= position, t.p[2][axis] <= position};
    for (int v = 0; v < 3; v++) { if (q[v]) growP(lBox, t.p[v]); else growP(rBox, t.p[v]); }
    for (int e = 0; e < 3; e++) {
        const int a = e, b = (e + 1) % 3;
        if (q[a] ^ q[b]) {
            const float tt = (position - t.p[a][axis]) / (t.p[b][axis] - t.p[a][axis]);
            float m[3];
            for (int i = 0; i < 3; i++) m[i] = t.p[a][i] + tt * (t.p[b][i] - t.p[a][i]);
            growP(lBox, m);
            growP(rBox, m);
        }
    }
}

struct PreArgs {
    const float* pos;            // PackedVec3[]
    const int4* tris;            // GpuBlasTriangle[] of the call
    const int* blasItemStart;    // [B + 1]: first work item (triangle of a BLAS) of every BLAS
    const int* blasTriOffset;
    const int* blasPresplit;
    int itemCount, blasCount;
    float* prio;                 // [items]
    float* totalPrio;            // [B]
    Box* globalBox;              // [B]
    long long* splitCount;       // [items + 1] -> exclusive scan -> fragment offsets
    int* itemBlas;               // [items]
    float splitFactor;
};

__device__ __forceinline__ int upperBound(const int* a, int n, int v) {   // first index with a[i] > v
    int lo = 0, hi = n;
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (a[mid] <= v) lo = mid + 1; else hi = mid; }
    return lo;
}

__global__ void k_item_prepare(PreArgs a) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= a.itemCount) return;
    const int b = upperBound(a.blasItemStart, a.blasCount + 1, k) - 1;
    a.itemBlas[k] = b;
    a.prio[k] = a.blasPresplit[b] ? priority(loadTri(a.pos, a.tris[a.blasTriOffset[b] + (k - a.blasItemStart[b])])) : 0.0f;
}

// The total is summed in triangle order, as PreSplitting.cs:33-37 does: float addition order matters.
__global__ void k_total_priority(PreArgs a) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= a.blasCount || !a.blasPresplit[b]) return;
    float total = 0.0f;
    for (int k = a.blasItemStart[b]; k < a.blasItemStart[b + 1]; k++) total += a.prio[k];
    a.totalPrio[b] = total;
}

// ---- block primitives (NT threads) ----
struct Smem {
    Box w[32], w2[32];
    int iw[32];
    float cost[32];
    int axis[32], idx[32];
};

__device__ __forceinline__ Box shflUpBox(const Box& v, int o) {
    Box u;
    for (int i = 0; i < 3; i++) { u.mn[i] = __shfl_up_sync(0xffffffffu, v.mn[i], o); u.mx[i] = __shfl_up_sync(0xffffffffu, v.mx[i], o); }
    return u;
}
__device__ __forceinline__ Box warpInclScan(Box v, int lane) {
    #pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const Box u = shflUpBox(v, o);
        if (lane >= o) v = comb(u, v);
    }
    return v;
}
// exclusive scan of one Box per thread in thread order; `total` = fold of all of them
__device__ Box blockExclScan(const Box& v, Box& total, Smem& sm) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const Box incl = warpInclScan(v, lane);
    if (lane == 31) sm.w[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        Box w = lane < nw ? sm.w[lane] : emptyBox();
        w = warpInclScan(w, lane);
        sm.w2[lane] = w;
    }
    __syncthreads();
    Box ex = shflUpBox(incl, 1);
    if (lane == 0) ex = emptyBox();
    if (warp > 0) ex = comb(sm.w2[warp - 1], ex);
    total = sm.w2[nw - 1];
    __syncthreads();
    return ex;
}
__device__ int blockExclScanInt(int v, int& total, Smem& sm) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    int incl = v;
    #pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int u = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += u; }
    if (lane == 31) sm.iw[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        int w = lane < nw ? sm.iw[lane] : 0;
        #pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int u = __shfl_up_sync(0xffffffffu, w, o); if (lane >= o) w += u; }
        sm.iw[lane] = w;
    }
    __syncthreads();
    const int ex = incl - v + (warp > 0 ? sm.iw[warp - 1] : 0);
    total = sm.iw[nw - 1];
    __syncthreads();
    return ex;
}

// Box of the elements boxes[ids[p]] for p in [begin, end), accumulated in ascending p (Box.GrowToFit order)
__device__ Box blockFold(const int* ids, int begin, int end, const Box* boxes, Smem& sm) {
    Box carry = emptyBox();
    for (int base = begin; base < end; base += CHUNK) {
        Box v = emptyBox();
        const int p0 = base + threadIdx.x * ITEMS;
        for (int k = 0; k < ITEMS; k++) if (p0 + k < end) v = comb(v, loadBox(boxes, ids ? ids[p0 + k] : p0 + k));
        Box tot;
        blockExclScan(v, tot, sm);
        carry = comb(carry, tot);
    }
    return carry;
}

// global box of a pre-split BLAS: every vertex in triangle order (PreSplitting.cs:41-46); one block per BLAS
__global__ void __launch_bounds__(NT) k_global_box(PreArgs a) {
    __shared__ Smem sm;
    const int b = blockIdx.x;
    if (!a.blasPresplit[b]) return;
    const int first = a.blasItemStart[b], end = a.blasItemStart[b + 1];
    Box carry = emptyBox();
    for (int base = first; base < end; base += CHUNK) {
        Box v = emptyBox();
        const int p0 = base + threadIdx.x * ITEMS;
        for (int k = 0; k < ITEMS; k++)
            if (p0 + k < end) v = comb(v, boxFromTri(loadTri(a.pos, a.tris[a.blasTriOffset[b] + (p0 + k - first)])));
        Box tot;
        blockExclScan(v, tot, sm);
        carry = comb(carry, tot);
    }
    if (threadIdx.x == 0) a.globalBox[b] = carry;
}

__global__ void k_split_counts(PreArgs a) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k > a.itemCount) return;
    if (k == a.itemCount) { a.splitCount[k] = 0; return; }
    const int b = a.itemBlas[k];
    long long c = 1;
    if (a.blasPresplit[b]) {      // PreSplitting.GetSplitCount
        const int triCount = a.blasItemStart[b + 1] - a.blasItemStart[b];
        const float shareOfTris = a.prio[k] / a.totalPrio[b] * (float)triCount;
        int s = csFloatToInt(shareOfTris * a.splitFactor);
        if (s == INT_MIN || s < 0) s = 0;      // the host mirror's guard for degenerate input
        c = 1 + (long long)s;
    }
    a.splitCount[k] = c;
}

__device__ __forceinline__ float getNodeSize(float extent, float globalSize) {
    const float alpha = extent / globalSize;
    return __uint_as_float(__float_as_uint(alpha) & (255u << 23)) * globalSize;
}

struct FragArgs {
    const float* pos;
    const int4* tris;
    const int* blasItemStart;
    const int* blasTriOffset;
    const int* blasPresplit;
    const int* itemBlas;
    const long long* offset;      // [items + 1]
    const Box* globalBox;
    int itemCount;
    long long fragCount;
    Box* bounds;                  // [F]
    int* fragTri;                 // [F] triangle index in the call's array
    int* fragBlas;                // [F]
};

// One thread per fragment. The host splits each triangle depth-first with a stack (left child first); each split
// depends only on the item's own box, so a fragment descends from the triangle to its own leaf: left children keep
// the offset, right children start at offset + leftCount.
__global__ void k_fragments(FragArgs a) {
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= a.fragCount) return;
    int lo = 0, hi = a.itemCount;          // item k with offset[k] <= j < offset[k + 1]
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (a.offset[mid] <= j) lo = mid; else hi = mid; }
    const int k = lo, b = a.itemBlas[k];
    const int tri = a.blasTriOffset[b] + (k - a.blasItemStart[b]);
    const Tri t = loadTri(a.pos, a.tris[tri]);
    Box box = boxFromTri(t);
    if (a.blasPresplit[b]) {
        int splits = (int)(a.offset[k + 1] - a.offset[k]);
        int local = (int)(j - a.offset[k]);
        const Box g = a.globalBox[b];
        while (splits > 1) {
            const int axis = largestAxis(box);
            const float le = largestExtent(box);
            float nodeSize = getNodeSize(le, g.mx[axis] - g.mn[axis]);
            if (nodeSize >= le - 0.0001f) nodeSize *= 0.5f;
            const float midPos = (box.mn[axis] + box.mx[axis]) * 0.5f;
            const float index = nearbyintf((midPos - g.mn[axis]) / nodeSize);   // MathF.Round: half to even
            const float splitPos = g.mn[axis] + index * nodeSize;
            Box l, r;
            triSplit(t, axis, splitPos, l, r);
            for (int i = 0; i < 3; i++) {    // Box.ShrinkToFit
                l.mn[i] = maxN(l.mn[i], box.mn[i]); l.mx[i] = minN(l.mx[i], box.mx[i]);
                r.mn[i] = maxN(r.mn[i], box.mn[i]); r.mx[i] = minN(r.mx[i], box.mx[i]);
            }
            const float leftExtent = largestExtent(l), rightExtent = largestExtent(r);
            int leftCount = csFloatToInt((float)splits * (leftExtent / (leftExtent + rightExtent)));
            leftCount = min(max(leftCount, 1), splits - 1);
            if (local < leftCount) { box = l; splits = leftCount; }
            else { box = r; local -= leftCount; splits -= leftCount; }
        }
    }
    a.bounds[j] = box;
    a.fragTri[j] = tri;
    a.fragBlas[j] = b;
}

__global__ void k_sort_keys(const Box* bounds, const int* fragBlas, long long n, int axis, unsigned long long* keys, int* vals) {
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const Box b = loadBox(bounds, (int)j);
    keys[j] = ((unsigned long long)fragBlas[j] << 32) | floatToKey(b.mn[axis] + b.mx[axis]);
    vals[j] = (int)j;
}

// ------------------------------------------------------------------------------------------------ splits
struct SplitArgs {
    const Box* bounds;
    int* sorted[3];               // fragment ids by position (global positions)
    uint8_t* table;               // by fragment id
    int* aux;                     // by position
    float* R[3];                  // suffix costs by position
    int* stack;                   // by position: 3 ints per entry (k_split_small)
    GpuBlasNode* nodes;           // node slots (BLAS b at nodeBase[b])
    int* depth; int* parent; int* rangeStart; int* rangeCount;
    const int* fragOffset; const int* nodeBase;
    Settings s;
    const Task* in; int inCount;
    Task* outBig; int* outBigCount;
    Task* small; int* smallCount;
};

__device__ __forceinline__ void createChild(const SplitArgs& a, int nb, int id, int parentId, int start, int count, int depth) {
    GpuBlasNode n = {};
    n.TriStartOrChild = start;
    n.TriCount = count;
    a.nodes[nb + id] = n;
    a.depth[nb + id] = depth;
    a.parent[nb + id] = parentId;
    a.rangeStart[nb + id] = start;
    a.rangeCount[nb + id] = count;
}

__device__ __forceinline__ void pushTask(const SplitArgs& a, Task t, int count) {
    if (count > SMALL) a.outBig[atomicAdd(a.outBigCount, 1)] = t;
    else a.small[atomicAdd(a.smallCount, 1)] = t;
}

// One block per node of the current level: BLAS.ProcessBuildTask + TrySplit for one node, every scan block-parallel.
__global__ void __launch_bounds__(NT) k_split_big(SplitArgs a) {
    __shared__ Smem sm;
    __shared__ int sAxis, sSplit;
    __shared__ float sCost;
    const Task t = a.in[blockIdx.x];
    const int nb = a.nodeBase[t.blas], fo = a.fragOffset[t.blas];
    GpuBlasNode node = a.nodes[nb + t.node];
    const int start = fo + node.TriStartOrChild, count = node.TriCount, end = start + count;

    const Box parentBox = blockFold(a.sorted[0], start, end, a.bounds, sm);
    setBounds(node, parentBox);
    bool split = count > a.s.stopSplittingThreshold;

    if (split) {
        float bestCost = FLT_MAX;
        int bestAxis = 0, bestSplit = INT_MAX;
        for (int axis = 0; axis < 3; axis++) {
            const int* ids = a.sorted[axis];
            float* R = a.R[axis];
            // suffix: R[i] = halfArea(box of [i, end)) * (end - i), accumulated from end - 1 down to start + 1
            Box carry = emptyBox();
            for (int qb = 0; qb < count - 1; qb += CHUNK) {
                Box item[ITEMS];
                Box v = emptyBox();
                const int q0 = qb + threadIdx.x * ITEMS;
                for (int k = 0; k < ITEMS; k++) {
                    item[k] = q0 + k < count - 1 ? loadBox(a.bounds, ids[end - 1 - (q0 + k)]) : emptyBox();
                    v = comb(v, item[k]);
                }
                Box tot;
                Box run = comb(carry, blockExclScan(v, tot, sm));
                for (int k = 0; k < ITEMS; k++) {
                    if (q0 + k >= count - 1) break;
                    run = comb(run, item[k]);
                    R[end - 1 - (q0 + k)] = halfArea(run) * (float)(q0 + k + 1);
                }
                carry = comb(carry, tot);
            }
            __syncthreads();
            // prefix: L[i] = halfArea(box of [start, i]) * (i - start + 1); candidate split i + 1 costs L[i] + R[i + 1]
            carry = emptyBox();
            for (int qb = 0; qb < count - 1; qb += CHUNK) {
                Box item[ITEMS];
                Box v = emptyBox();
                const int q0 = qb + threadIdx.x * ITEMS;
                for (int k = 0; k < ITEMS; k++) {
                    item[k] = q0 + k < count - 1 ? loadBox(a.bounds, ids[start + q0 + k]) : emptyBox();
                    v = comb(v, item[k]);
                }
                Box tot;
                Box run = comb(carry, blockExclScan(v, tot, sm));
                for (int k = 0; k < ITEMS; k++) {
                    if (q0 + k >= count - 1) break;
                    run = comb(run, item[k]);
                    const int i = start + q0 + k;
                    const float cost = halfArea(run) * (float)(q0 + k + 1) + R[i + 1];
                    // first strict minimum in (axis, split index) order, among costs below FLT_MAX
                    if (cost < FLT_MAX && (cost < bestCost || (cost == bestCost && (axis < bestAxis || (axis == bestAxis && i + 1 < bestSplit))))) {
                        bestCost = cost; bestAxis = axis; bestSplit = i + 1;
                    }
                }
                carry = comb(carry, tot);
            }
            __syncthreads();
        }
        // block argmin of (cost, axis, split)
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        auto better = [](float c, int ax, int sp, float c2, int ax2, int sp2) {
            return c < c2 || (c == c2 && (ax < ax2 || (ax == ax2 && sp < sp2)));
        };
        for (int o = 16; o > 0; o >>= 1) {
            const float c = __shfl_down_sync(0xffffffffu, bestCost, o);
            const int ax = __shfl_down_sync(0xffffffffu, bestAxis, o), sp = __shfl_down_sync(0xffffffffu, bestSplit, o);
            if (better(c, ax, sp, bestCost, bestAxis, bestSplit)) { bestCost = c; bestAxis = ax; bestSplit = sp; }
        }
        if (lane == 0) { sm.cost[warp] = bestCost; sm.axis[warp] = bestAxis; sm.idx[warp] = bestSplit; }
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < (int)(blockDim.x >> 5); w++)
                if (better(sm.cost[w], sm.axis[w], sm.idx[w], bestCost, bestAxis, bestSplit)) { bestCost = sm.cost[w]; bestAxis = sm.axis[w]; bestSplit = sm.idx[w]; }
            if (bestCost == FLT_MAX) { bestAxis = 0; bestSplit = start + count / 2; }   // the host mirror's guard (no finite cost)
            bool ok = true;
            if (count <= a.s.maxLeafTriangleCount) {
                const float notSplitCost = a.s.triangleCost * (float)count;
                const float newCost = 1.0f + (a.s.triangleCost * bestCost / halfArea(parentBox));
                if (newCost >= notSplitCost) ok = false;
            }
            sAxis = bestAxis; sSplit = ok ? bestSplit : -1;
        }
        __syncthreads();
        split = sSplit >= 0;
    }

    if (!split) {
        if (threadIdx.x == 0) a.nodes[nb + t.node] = node;
        return;
    }
    const int axis = sAxis, splitIndex = sSplit;
    int* ids = a.sorted[axis];
    const Box lb = blockFold(ids, start, splitIndex, a.bounds, sm);
    const Box rb = blockFold(ids, splitIndex, end, a.bounds, sm);
    const bool swapSides = halfArea(lb) < halfArea(rb);   // the larger child goes left
    for (int p = start + threadIdx.x; p < end; p += blockDim.x) a.table[ids[p]] = (p < splitIndex) != swapSides;
    __syncthreads();
    const int leftCount = swapSides ? end - splitIndex : splitIndex - start;
    for (int arr = 0; arr < 3; arr++) {       // Algorithms.StablePartition on the three id arrays
        if (arr == axis && !swapSides) continue;
        int* src = a.sorted[arr];
        int carryL = 0;
        for (int base = start; base < end; base += CHUNK) {
            const int p0 = base + threadIdx.x * ITEMS;
            int id[ITEMS];
            int f = 0;
            for (int k = 0; k < ITEMS; k++) { id[k] = p0 + k < end ? src[p0 + k] : -1; f += (id[k] >= 0 && a.table[id[k]]) ? 1 : 0; }
            int tot;
            int before = carryL + blockExclScanInt(f, tot, sm);
            for (int k = 0; k < ITEMS; k++) {
                if (id[k] < 0) break;
                const int p = p0 + k;
                if (a.table[id[k]]) a.aux[start + before++] = id[k];
                else a.aux[start + leftCount + (p - start) - before] = id[k];
            }
            carryL += tot;
        }
        __syncthreads();
        for (int p = start + threadIdx.x; p < end; p += blockDim.x) src[p] = a.aux[p];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const int leftId = t.newNodes, rightId = leftId + 1;
        const int lStart = start - fo, rCount = count - leftCount;
        createChild(a, nb, leftId, t.node, lStart, leftCount, t.depth + 1);
        createChild(a, nb, rightId, t.node, lStart + leftCount, rCount, t.depth + 1);
        node.TriStartOrChild = leftId;
        node.TriCount = 0;
        a.nodes[nb + t.node] = node;
        pushTask(a, {t.blas, leftId, rightId + 1, t.depth + 1}, leftCount);
        pushTask(a, {t.blas, rightId, rightId + (2 * leftCount - 1), t.depth + 1}, rCount);
    }
}

// BLAS.TrySplit (Bvh/BLAS.cs:730-873) as the host mirror runs it, on one thread over one subtree's ranges
__device__ bool trySplitSerial(const SplitArgs& a, const GpuBlasNode& parent, int fo, int& outSplit) {
    const Settings& s = a.s;
    if (parent.TriCount <= s.stopSplittingThreshold) return false;
    const int start = fo + parent.TriStartOrChild, end = start + parent.TriCount;
    float bestCost = FLT_MAX;
    int bestAxis = 0, bestSplit = 0;
    float* rightCostsAccum = a.R[0];
    for (int axis = 0; axis < 3; axis++) {
        const int* ids = a.sorted[axis];
        int firstRight = start + 1;
        Box acc = emptyBox();
        float rightCounter = 0.0f;
        for (int i = end - 1; i >= firstRight; i--) {
            rightCounter++;
            acc = comb(acc, loadBox(a.bounds, ids[i]));
            const float rightCost = halfArea(acc) * rightCounter;
            rightCostsAccum[i] = rightCost;
            if (rightCost >= bestCost) { firstRight = i + 1; break; }
        }
        Box lacc = emptyBox();
        float leftCounter = (float)(firstRight - start) - 1.0f;
        for (int i = start; i < firstRight - 1; i++) lacc = comb(lacc, loadBox(a.bounds, ids[i]));
        for (int i = firstRight - 1; i < end - 1; i++) {
            leftCounter++;
            lacc = comb(lacc, loadBox(a.bounds, ids[i]));
            const float leftCost = halfArea(lacc) * leftCounter;
            const float cost = leftCost + rightCostsAccum[i + 1];
            if (cost < bestCost) { bestSplit = i + 1; bestAxis = axis; bestCost = cost; }
            else if (leftCost >= bestCost) break;
        }
    }
    if (bestCost == FLT_MAX) { bestAxis = 0; bestSplit = start + parent.TriCount / 2; }
    if (parent.TriCount <= s.maxLeafTriangleCount) {
        const float notSplitCost = s.triangleCost * (float)parent.TriCount;
        const float newCost = 1.0f + (s.triangleCost * bestCost / nodeHalfArea(parent));
        if (newCost >= notSplitCost) return false;
    }
    int* ids = a.sorted[bestAxis];
    Box lb = emptyBox(), rb = emptyBox();
    for (int i = start; i < bestSplit; i++) lb = comb(lb, loadBox(a.bounds, ids[i]));
    for (int i = bestSplit; i < end; i++) rb = comb(rb, loadBox(a.bounds, ids[i]));
    const bool swapSides = halfArea(lb) < halfArea(rb);
    for (int i = start; i < bestSplit; i++) a.table[ids[i]] = !swapSides;
    for (int i = bestSplit; i < end; i++) a.table[ids[i]] = swapSides;
    int leftCount = bestSplit - start;
    for (int arr = 0; arr < 3; arr++) {
        if (arr == bestAxis && !swapSides) continue;
        int* src = a.sorted[arr];
        int l = 0, r = 0;
        for (int i = start; i < end; i++) {
            const int id = src[i];
            if (a.table[id]) src[start + l++] = id; else a.aux[start + r++] = id;
        }
        for (int i = 0; i < r; i++) src[start + l + i] = a.aux[start + i];
        if (arr == bestAxis) leftCount = l;
    }
    outSplit = start + leftCount;
    return true;
}

// BLAS.ProcessBuildTask for a whole subtree of at most SMALL fragments on one thread; its stack lives in the
// subtree's own range of `stack` (depth < fragment count).
__global__ void k_split_small(SplitArgs a, int count) {
    const int ti = blockIdx.x * blockDim.x + threadIdx.x;
    if (ti >= count) return;
    const Task root = a.small[ti];
    const int nb = a.nodeBase[root.blas], fo = a.fragOffset[root.blas];
    int* stk = a.stack + 3 * (size_t)(fo + a.nodes[nb + root.node].TriStartOrChild);
    int sp = 0;
    stk[0] = root.node; stk[1] = root.newNodes; stk[2] = root.depth; sp = 1;
    while (sp > 0) {
        sp--;
        const int nodeId = stk[3 * sp], newNodes = stk[3 * sp + 1], depth = stk[3 * sp + 2];
        GpuBlasNode parent = a.nodes[nb + nodeId];
        Box box = emptyBox();
        const int start = fo + parent.TriStartOrChild;
        for (int i = start; i < start + parent.TriCount; i++) box = comb(box, loadBox(a.bounds, a.sorted[0][i]));
        setBounds(parent, box);
        int splitIndex;
        if (!trySplitSerial(a, parent, fo, splitIndex)) { a.nodes[nb + nodeId] = parent; continue; }
        const int leftCount = splitIndex - start, rightCount = parent.TriCount - leftCount;
        const int leftId = newNodes, rightId = leftId + 1;
        createChild(a, nb, leftId, nodeId, parent.TriStartOrChild, leftCount, depth + 1);
        createChild(a, nb, rightId, nodeId, parent.TriStartOrChild + leftCount, rightCount, depth + 1);
        parent.TriStartOrChild = leftId;
        parent.TriCount = 0;
        a.nodes[nb + nodeId] = parent;
        stk[3 * sp] = rightId; stk[3 * sp + 1] = rightId + (2 * leftCount - 1); stk[3 * sp + 2] = depth + 1; sp++;
        stk[3 * sp] = leftId; stk[3 * sp + 1] = rightId + 1; stk[3 * sp + 2] = depth + 1; sp++;
    }
}

// ------------------------------------------------------------------------------------------------ after the splits
struct PostArgs {
    GpuBlasNode* nodes;           // built tree (node slots)
    GpuBlasNode* out;             // compacted result (same slots)
    int* depth; int* parent; int* rangeStart; int* rangeCount;
    const int* nodeBase;          // [B + 1]
    const int* fragOffset; const int* fragCount;
    int blasCount; int nodeSlots;
    Settings s;
    int* rootWasLeaf;             // [B]
    int* created;                 // [B]
    unsigned long long* keys; int* vals;
    int* pre;                     // pre-order: node slot at each position
    int* byDepth;                 // (depth, range start) order
    int* prePos;                  // node slot -> pre-order position
    int* cflag;                   // [slots + 1] created flags -> exclusive scan
    int* size;                    // subtree node count
    int* diff;                    // [slots + 1] -> inclusive scan
    int* rs0;                     // [B]
    double* sahPre;               // by pre-order position
    double* collPre;              // by pre-order position: collapse cost term (internal nodes)
    int* qualPre;                 // by pre-order position: internal with two leaf children; depth
    int* depthPre;
    double* collDep;              // by depth-order position
    int* internalDep; int* depthDep;
    int* finalK; int* rsOut;      // [B]
    int* flag;                    // [slots + 1]
    int* newId;                   // node slot -> compacted id (-1: removed)
    int* pairCount;               // [slots + 1]
    int* uniq;                    // by position: sorted unique triangle ids of every leaf
    int* uniqCount;               // node slot (of `out`) -> unique triangle count
    int* newCount;                // [B]
    int* triOutCount;             // [B]
    double* sah;                  // [B]
    const int* sorted0; const int* fragTri;
    const int4* tris; int4* triOut;
    const int* presplit;
};

__device__ __forceinline__ int slotBlas(const PostArgs& a, int g) { return upperBound(a.nodeBase, a.blasCount + 1, g) - 1; }

// BLAS.Build (BLAS.cs:185-193): a root that did not split becomes the parent of two copies of itself
__global__ void k_root_fix(PostArgs a) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= a.blasCount) return;
    const int nb = a.nodeBase[b];
    GpuBlasNode root = a.nodes[nb + 1];
    a.rootWasLeaf[b] = root.TriCount > 0;
    if (root.TriCount > 0) {
        for (int c = 2; c < 4; c++) {
            a.nodes[nb + c] = root;
            a.depth[nb + c] = 1; a.parent[nb + c] = 1; a.rangeStart[nb + c] = 0; a.rangeCount[nb + c] = root.TriCount;
        }
        root.TriStartOrChild = 2;
        root.TriCount = 0;
        a.nodes[nb + 1] = root;
    }
}

__global__ void k_node_keys(PostArgs a, int depthMajor) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= a.nodeSlots) return;
    const int b = slotBlas(a, g);
    const unsigned long long hi = (unsigned long long)b << 48;
    const int d = a.depth[g];
    unsigned long long lo = 0xFFFFFFFFFFFFull;
    if (d >= 0) {
        const unsigned long long s = (unsigned)a.rangeStart[g], dd = (unsigned)d;
        lo = depthMajor ? (dd << 24) | s : (s << 24) | dd;
        if (!depthMajor) atomicAdd(&a.created[b], 1);
    }
    a.keys[g] = hi | lo;
    a.vals[g] = g;
    if (!depthMajor) a.cflag[g] = d >= 0;
    if (!depthMajor && g == 0) a.cflag[a.nodeSlots] = 0;
}

__global__ void k_pre_pos(PostArgs a) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= a.nodeSlots) return;
    a.prePos[a.pre[q]] = q;
    a.diff[q] = 0;
    if (q == 0) a.diff[a.nodeSlots] = 0;
}

// subtree node counts: the descendants of a node with child pair c and n fragments are the created nodes in [c, c + 2n - 2)
__global__ void k_sizes_both(PostArgs a) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= a.nodeSlots || a.depth[g] < 0) return;
    const GpuBlasNode n = a.nodes[g];
    if (n.TriCount > 0) { a.size[g] = 1; return; }
    const int b = slotBlas(a, g), nb = a.nodeBase[b];
    int sz;
    if (g - nb == 1 && a.rootWasLeaf[b]) sz = 3;
    else sz = 1 + a.cflag[nb + n.TriStartOrChild + 2 * a.rangeCount[g] - 2] - a.cflag[nb + n.TriStartOrChild];
    a.size[g] = sz;
    const GpuBlasNode l = a.nodes[nb + n.TriStartOrChild], r = a.nodes[nb + n.TriStartOrChild + 1];
    if (l.TriCount == 0 && r.TriCount == 0) {      // a pair of internal nodes: one more stack entry below here
        atomicAdd(&a.diff[a.prePos[g]], 1);
        atomicAdd(&a.diff[a.prePos[g] + sz], -1);
    }
}

// computeRequiredStackSize(2) = the most "both children internal" nodes on any root path; per-node terms of the SAH
// and of the collapse costs
__global__ void k_terms(PostArgs a) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= a.nodeSlots || a.depth[g] < 0) return;
    const int b = slotBlas(a, g), nb = a.nodeBase[b];
    const int q = a.prePos[g];
    atomicMax(&a.rs0[b], a.diff[q]);
    const GpuBlasNode n = a.nodes[g];
    const double rootHA = (double)nodeHalfArea(a.nodes[nb + 1]);
    const double prob = (double)nodeHalfArea(n) * (1.0 / rootHA);
    a.sahPre[q] = n.TriCount > 0 ? (double)(a.s.triangleCost * (float)n.TriCount) * prob : 1.0 * prob;
    a.depthPre[q] = a.depth[g];
    int qual = 0;
    double term = 0.0;
    if (n.TriCount == 0) {
        const int lg = nb + n.TriStartOrChild;
        const GpuBlasNode l = a.nodes[lg], r = a.nodes[lg + 1];
        const int lc = a.rangeCount[lg], rc = a.rangeCount[lg + 1];   // counts once the children are leaves
        const double leavesCost = (double)a.s.triangleCost * ((double)lc * (double)nodeHalfArea(l) + (double)rc * (double)nodeHalfArea(r));
        const double newParentLeafCost = (double)a.s.triangleCost * (double)(lc + rc);
        term = ((double)nodeHalfArea(n) * (newParentLeafCost - 1.0) - leavesCost) / rootHA;
        qual = l.TriCount > 0 && r.TriCount > 0;
    }
    a.collPre[q] = term;
    a.qualPre[q] = qual;
}

__global__ void k_dep_arrays(PostArgs a) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= a.nodeSlots) return;
    const int g = a.byDepth[q];
    if (a.depth[g] < 0) return;
    a.depthDep[q] = a.depth[g];
    a.internalDep[q] = a.nodes[g].TriCount == 0;
    a.collDep[q] = a.collPre[a.prePos[g]];
}

// Ordered double sum over q in [begin, end) by one warp: each lane loads one of 32 consecutive terms (the next 32 are in
// flight meanwhile), then the terms are added one at a time in q order, so the result is the serial loop's bit for bit.
// Skipped nodes contribute +0.0, which leaves a sum that starts at +0.0 unchanged.
template <class F>
__device__ double warpOrderedSum(double acc, int begin, int end, F term) {
    const int lane = threadIdx.x & 31;
    double next = begin + lane < end ? term(begin + lane) : 0.0;
    for (int base = begin; base < end; base += 32) {
        const double v = next;
        next = base + 32 + lane < end ? term(base + 32 + lane) : 0.0;
        const int n = min(32, end - base);
        for (int j = 0; j < n; j++) acc += __shfl_sync(0xffffffffu, v, j);
    }
    return acc;
}

// BLAS.OptimizeStackSize (BLAS.cs:875-937): the double sums in the host's visiting order, one warp per BLAS.
// collapseDeepestLevel's first pass adds the nodes deeper than rs - 1 with two leaf children, in post-order (= pre-order
// for such nodes); every later pass at level K collapses everything below K and adds every internal node at depth K,
// left to right. (Its FLT_MAX branch needs more than 2^31 triangles in a leaf; the build refuses 2^24.)
__global__ void __launch_bounds__(32) k_stack_opt(PostArgs a) {
    const int b = blockIdx.x;
    const int base = a.nodeBase[b], n = a.created[b];
    int rs = a.rs0[b], fk = -1;
    if (rs >= a.s.stackOptThreshold) {
        const int k0 = rs - 1;
        const double cur = warpOrderedSum(0.0, base, base + n, [&](int q) { return a.sahPre[q]; });
        double added = warpOrderedSum(0.0, base, base + n, [&](int q) { return a.qualPre[q] && a.depthPre[q] > k0 ? a.collPre[q] : 0.0; });
        double inc = added / cur;
        while (inc <= (double)a.s.stackOptSahIncreaseAcceptance && rs > 0) {
            rs--;
            int lo = base, hi = base + n;     // the nodes of depth rs in (depth, range start) order
            while (lo < hi) { const int mid = (lo + hi) >> 1; if (a.depthDep[mid] < rs) lo = mid + 1; else hi = mid; }
            int end = lo;
            hi = base + n;
            while (end < hi) { const int mid = (end + hi) >> 1; if (a.depthDep[mid] <= rs) end = mid + 1; else hi = mid; }
            added = warpOrderedSum(added, lo, end, [&](int q) { return a.internalDep[q] ? a.collDep[q] : 0.0; });
            inc = added / cur;
            fk = rs;
        }
    }
    if (threadIdx.x == 0) { a.finalK[b] = fk; a.rsOut[b] = rs; }
}

// BLAS.RemoveEmptySubtrees: the children of the k-th internal node in pre-order get ids 2 + 2k, 3 + 2k
__global__ void k_survivors(PostArgs a) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q > a.nodeSlots) return;
    if (q == a.nodeSlots) { a.flag[q] = 0; return; }
    const int g = a.pre[q];
    int f = 0;
    if (a.depth[g] >= 0) {
        const int fk = a.finalK[slotBlas(a, g)];
        const int d = a.depth[g];
        f = (fk < 0 || d <= fk) && a.nodes[g].TriCount == 0;
    }
    a.flag[q] = f;
}

__global__ void k_emit(PostArgs a) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= a.nodeSlots) return;
    const int d = a.depth[g];
    a.newId[g] = -1;
    if (d < 0) return;
    const int b = slotBlas(a, g), nb = a.nodeBase[b], fk = a.finalK[b];
    if (fk >= 0 && d > fk + 1) return;
    const int base = a.flag[nb];       // exclusive scan of the flags, by pre-order position
    const int v = g - nb;
    int id = 1;
    if (v != 1) {
        const int p = a.parent[g];
        id = 2 + 2 * (a.flag[a.prePos[nb + p]] - base) + (v == a.nodes[nb + p].TriStartOrChild + 1 ? 1 : 0);
    }
    GpuBlasNode n = a.nodes[g];
    if (n.TriCount == 0 && (fk < 0 || d <= fk)) n.TriStartOrChild = 2 + 2 * (a.flag[a.prePos[g]] - base);
    else { n.TriStartOrChild = a.rangeStart[g]; n.TriCount = a.rangeCount[g]; }
    a.out[nb + id] = n;
    a.newId[g] = id;
    if (v == 1) a.newCount[b] = 2 + 2 * (a.flag[nb + a.nodeBase[b + 1] - a.nodeBase[b]] - base);
}

// ---- unindexing
// BLAS.GetUnindexedTriangles (BLAS.cs:441-466): leaves in id order, triangle offsets = prefix sum of their counts
__global__ void k_leaf_counts(PostArgs a) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g > a.nodeSlots) return;
    int c = 0;
    if (g < a.nodeSlots) {
        const int b = slotBlas(a, g), v = g - a.nodeBase[b];
        if (!a.presplit[b]) {
            if (v >= 2 && v < a.newCount[b] && a.out[g].TriCount > 0) c = a.out[g].TriCount;
        } else if (v >= 2 && v < a.newCount[b] && !(v & 1)) {
            c = a.pairCount[g];
        }
    }
    a.flag[g] = c;
}

__global__ void k_unindex_plain(PostArgs a) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= a.nodeSlots) return;
    const int b = slotBlas(a, g), nb = a.nodeBase[b], v = g - nb;
    if (a.presplit[b] || v < 2 || v >= a.newCount[b]) return;
    GpuBlasNode n = a.out[g];
    if (n.TriCount <= 0) return;
    const int counter = a.flag[g] - a.flag[nb], fo = a.fragOffset[b], nf = a.fragCount[b];
    // (a root that did not split is listed twice; the host writes the second copy past the array's end and drops it)
    for (int j = 0; j < n.TriCount && counter + j < nf; j++) a.triOut[fo + counter + j] = a.tris[a.fragTri[a.sorted0[fo + n.TriStartOrChild + j]]];
    n.TriStartOrChild = counter;
    a.out[g] = n;
    if (v == 2) a.triOutCount[b] = nf;
}

__device__ void heapSort(int* x, int n) {
    auto sift = [&](int i, int m) {
        for (;;) {
            int c = 2 * i + 1;
            if (c >= m) break;
            if (c + 1 < m && x[c + 1] > x[c]) c++;
            if (x[i] >= x[c]) break;
            const int t = x[i]; x[i] = x[c]; x[c] = t;
            i = c;
        }
    };
    for (int i = n / 2 - 1; i >= 0; i--) sift(i, n);
    for (int m = n - 1; m > 0; m--) { const int t = x[0]; x[0] = x[m]; x[m] = t; sift(0, m); }
}

// sorted unique original triangles of a leaf, written over its own range of `uniq`
__device__ int leafUnique(const PostArgs& a, int fo, const GpuBlasNode& leaf) {
    int* u = a.uniq + fo + leaf.TriStartOrChild;
    for (int i = 0; i < leaf.TriCount; i++) u[i] = a.fragTri[a.sorted0[fo + leaf.TriStartOrChild + i]];
    heapSort(u, leaf.TriCount);
    int m = 0;
    for (int i = 0; i < leaf.TriCount; i++) if (i == 0 || u[i] != u[m - 1]) u[m++] = u[i];
    return m;
}
__device__ __forceinline__ bool sortedContains(const int* u, int n, int x) {
    int lo = 0, hi = n;
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (u[mid] < x) lo = mid + 1; else hi = mid; }
    return lo < n && u[lo] == x;
}

// PreSplitting.GetUnindexedTriangles (PreSplitting.cs:169-273): pairs in id order (its depth-first walk visits them so)
__global__ void k_pair_counts(PostArgs a) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= a.nodeSlots) return;
    const int b = slotBlas(a, g), nb = a.nodeBase[b], v = g - nb;
    a.pairCount[g] = 0;
    if (!a.presplit[b] || v < 2 || v >= a.newCount[b] || (v & 1)) return;
    const int fo = a.fragOffset[b];
    const GpuBlasNode l = a.out[g], r = a.out[g + 1];
    const bool ll = l.TriCount > 0, rl = r.TriCount > 0;
    int c = 0;
    if (ll && rl) {
        const int lu = leafUnique(a, fo, l);
        const int ru = (r.TriStartOrChild == l.TriStartOrChild) ? lu : leafUnique(a, fo, r);
        const int* L = a.uniq + fo + l.TriStartOrChild;
        const int* Rr = a.uniq + fo + r.TriStartOrChild;
        int shared = 0;
        for (int i = 0; i < lu; i++) shared += sortedContains(Rr, ru, L[i]);
        c = lu + ru - shared;
        a.uniqCount[g] = lu; a.uniqCount[g + 1] = ru;
    } else if (ll || rl) {
        const GpuBlasNode& leaf = ll ? l : r;
        c = leafUnique(a, fo, leaf);
        a.uniqCount[ll ? g : g + 1] = c;
    }
    a.pairCount[g] = c;
}

__global__ void k_unindex_pairs(PostArgs a) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= a.nodeSlots) return;
    const int b = slotBlas(a, g), nb = a.nodeBase[b], v = g - nb;
    if (!a.presplit[b] || v < 2 || v >= a.newCount[b] || (v & 1)) return;
    const int fo = a.fragOffset[b];
    const int counter = a.flag[g] - a.flag[nb];
    GpuBlasNode l = a.out[g], r = a.out[g + 1];
    const bool ll = l.TriCount > 0, rl = r.TriCount > 0;
    int4* out = a.triOut + fo;
    if (ll && rl) {
        const int lu = a.uniqCount[g], ru = a.uniqCount[g + 1];
        const int* L = a.uniq + fo + l.TriStartOrChild;
        const int* Rr = a.uniq + fo + r.TriStartOrChild;
        int onlyLeft = 0, backwards = 0;
        for (int i = 0; i < lu; i++) {
            if (sortedContains(Rr, ru, L[i])) out[counter + lu - backwards++ - 1] = a.tris[L[i]];
            else out[counter + onlyLeft++] = a.tris[L[i]];
        }
        int onlyRight = 0;
        for (int i = 0; i < ru; i++)
            if (!sortedContains(L, lu, Rr[i])) out[counter + lu + onlyRight++] = a.tris[Rr[i]];
        l.TriStartOrChild = counter; l.TriCount = lu;
        r.TriStartOrChild = counter + onlyLeft; r.TriCount = ru;
        a.out[g] = l; a.out[g + 1] = r;
    } else if (ll || rl) {
        GpuBlasNode leaf = ll ? l : r;
        const int u = a.uniqCount[ll ? g : g + 1];
        const int* U = a.uniq + fo + leaf.TriStartOrChild;
        for (int i = 0; i < u; i++) out[counter + i] = a.tris[U[i]];
        leaf.TriStartOrChild = counter; leaf.TriCount = u;
        a.out[ll ? g : g + 1] = leaf;
    }
    if (v == 2) a.triOutCount[b] = a.flag[nb + a.nodeBase[b + 1] - a.nodeBase[b]] - a.flag[nb];
}

// computeGlobalSAH on the result: terms at the surviving nodes' pre-order positions, summed in that order per BLAS
__global__ void k_final_terms(PostArgs a) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= a.nodeSlots || a.depth[g] < 0) return;
    const int q = a.prePos[g];
    const int id = a.newId[g];
    a.qualPre[q] = id >= 0;
    if (id < 0) return;
    const int nb = a.nodeBase[slotBlas(a, g)];
    const GpuBlasNode n = a.out[nb + id];
    const double prob = (double)nodeHalfArea(n) * (1.0 / (double)nodeHalfArea(a.out[nb + 1]));
    a.sahPre[q] = n.TriCount > 0 ? (double)(a.s.triangleCost * (float)n.TriCount) * prob : 1.0 * prob;
}

__global__ void __launch_bounds__(32) k_final_sah(PostArgs a) {
    const int b = blockIdx.x;
    const double cost = warpOrderedSum(0.0, a.nodeBase[b], a.nodeBase[b] + a.created[b], [&](int q) { return a.qualPre[q] ? a.sahPre[q] : 0.0; });
    if (threadIdx.x == 0) a.sah[b] = cost;
}

} // namespace idkbb
