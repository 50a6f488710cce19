// libidkpt: C ABI (include/idkpt.h) over the sm_100a wavefront kernels (idk_kernels.cuh).
// Host sequencing mirrors PathTracer.Compute(), IDKEngine/Source/Render/PathTracer.cs:214-297, with
// every GL dispatch replaced by a CUDA launch on one stream and no CPU read-back inside the loop
// (alive counts stay on the device, like the reference's indirect dispatch).
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <string>
#include <vector>
#include <algorithm>

#include "../../include/idkpt.h"
#include "idk_kernels.cuh"
#include "idk_sort.cuh"
#include "idk_shadows.cuh"
#include "idk_dynamic.cuh"
#include "idk_post.cuh"
#include "idk_blas_build.cuh"
#include "idk_textures_host.h"

#define IDKPT_ABI_VERSION 4u   // 2: IdkPtSceneDesc gained Textures / TextureCount; 3: IdkPtStats gained CompactMs / AccumulateMs, host-buffer registration;
                               // 4: gather handle blob is 5 IPC handles (320 bytes), IDKPT_CREATE_GLOBAL_SLOTS, idkpt_gather_connect

static thread_local std::string g_createError;

struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
};

#define IDK_MAX_LANES 16

struct Lane {
    cudaStream_t stream = nullptr;
    cudaEvent_t radianceReady = nullptr;   // recorded on the lane stream after the last shade of a sample
    cudaEvent_t accDone = nullptr;         // recorded on the main stream after that sample's FinalDraw consumed `radiance`
    bool accPending = false;
    bool allocated = false;
    DevBuf state, aov, alive[2], survivors, keysTmp, sortedAlive, hits, hitXform, debugCost, radiance, aovAlbedoFinal, aovNormalFinal;
    DevBuf countsDev;              // uint32 counts[IDKPT_MAX_RAY_DEPTH + 1]
    DevBuf tickets;                // uint32 tickets[2 * (IDKPT_MAX_RAY_DEPTH + 1)] (traverse, compact)
    DevBuf tileStatus;             // u64 per tile
    uint32_t epoch = 0;            // compaction epoch of this lane's status words: 1 .. IDK_EPOCH_MASK, cleared on wrap
    DevBuf keys;                   // ray sorting: key per slot of the compacted alive list
    IdkSortScratch sortScratch;
    DevBuf slotDelta;              // global slots: per local stripe, global - local slot of the current bounce (k_slot_exchange)
    uint32_t slotEpoch = 0;        // exchanges issued on this lane since the peers were connected (identical on every rank)
};

struct IdkPtCtx {
    int device = 0;
    int smCount = 148;
    cudaStream_t stream = nullptr;
    std::string lastError;

    // image / tile geometry
    int width = 0, height = 0;
    int stripeH = 8, tileIndex = 0, tileCount = 1;
    std::vector<int> rows;         // owned rows, ascending
    uint32_t nLocal = 0;           // rows.size() * width
    uint32_t accumulatedSamples = 0;

    // scene
    bool haveScene = false;
    DeviceScene sc = {};
    IdkPtSceneDesc counts = {};    // element counts only (pointers unused)
    DevBuf nodes, triRec, blasTris, positions, descs, instances, xforms, meshes, materials, vertices, lights, tlas, vtxFrame, surfRec;
    float sky[3] = {0.0f, 0.0f, 0.0f};
    DevBuf skyFaces;
    int skyFaceSize = 0;
    DevBuf texPixels, texRecs, srgbLut;   // material textures (RGBA8 base levels), their records, sRGB decode table
    std::vector<uint64_t> hostMaterialMaxHandle;   // per material: largest texture handle it uses (validation of later edits)

    // host-array entry points (trace_rays, shadows): device staging buffers, kept between calls
    DevBuf scratch[3];

    // present chain: bloom mip chains (rgba16f), AgX constants, RGBA8 frame
    DevBuf bloomDown, bloomUp, postConsts, ldr;
    // denoise hand-off: OIDN-layout packed RGB buffers (beauty, albedo, normal, output), a-trous ping-pong, denoised rgba32f image
    DevBuf oidn[4], denoiseWork[2], denoised;
    bool haveDenoised = false;

    // dynamic geometry: unskinned vertices, joint matrices, refit scratch (parents + locks of the largest BLAS)
    DevBuf unskinned, joints, refitParents, refitLocks, tlasScratch;
    uint64_t unskinnedCount = 0;
    std::vector<uint32_t> unskinnedMaxJoint;   // per vertex max(JointIndices), host copy for range validation
    std::vector<GpuBlasDesc> hostDescs;
    size_t nodeBytes = 0;

    // wavefront buffers: one set per lane. A lane is one sample in flight (ray-gen .. last shade) on its own stream; with
    // several lanes the latency-bound tail bounces of one sample overlap the throughput-bound head of the next
    // (profiles/r01h_overlap_probe.json). Lane 0 also serves the synchronous path (stats, export, debug).
    Lane lanes[IDK_MAX_LANES];
    int laneCount = 8;             // lanes used by asynchronous idkpt_compute (stats == NULL); IDKPT_LANES / CreateInfo.Flags
    int nextLane = 0;
    bool asyncPending = false;     // work issued on lane streams / main stream that no host call has waited for yet
    DevBuf images[3];
    DevBuf counters;               // TraceCounters
    DevBuf countLog;               // per-sample copies of the alive counts (stats only)
    uint32_t epochStart = 0;       // IDKPT_DEBUG_EPOCH_START: first compaction epoch of a fresh lane (wrap-around test hook)
    uint32_t slotEpochStart = 0;   // IDKPT_DEBUG_SLOT_EPOCH_START: slot-exchange epoch right after the peers are connected (wrap-around test hook)
    bool exportEnabled = false;

    // launch configuration
    int traverseBlocks = 0, traverseBlocksStats = 0, shadeBlocks = 0, traceRaysBlocks = 0, compactBlocks = 0;
    int traverse1Blocks = 0, traverse1BlocksStats = 0;
    int traverseBlocksLane = 0, traverse1BlocksLane = 0;   // grids of the asynchronous path: the resident-block budget split between the lanes
    int traverseVariant = 3;       // 1 = k_traverse (one ray per lane, reference loop), 2 = k_traverse2 (phase-scheduled warps),
                                   // 3 = k_traverse for the coherent primary rays, k_traverse2 for every bounce (default)
    TraverseTuning tune = {12, 4, 0, 6, 0};   // swept on B200 (profiles/r01b_tuning.txt); packRays is set per launch
    int packCta = 0;                 // IDKPT_PACK_CTA: pipelined launches let only ceil(rays / (256 * k)) CTAs take part (0 = all; measured neutral at k = 1, slower at 2 / 4: profiles/r02_traverse_experiments.txt)
    int packAsync = 1;               // IDKPT_PACK_ASYNC: asynchronous (pipelined) launches pack 32 rays per warp instead of spreading few rays over all warps
    size_t stackBytes = 0;
    size_t traverse2Smem = 0;      // treelet + stacks
    int treeletNodes = 0;

    std::vector<cudaEvent_t> events;
    cudaStreamAttrValue l2Window = {};   // persisting-L2 window over [nodes | triRec]; applied to the main stream and every lane stream

    // multi-GPU gather over NVLink peer memory (CUDA IPC): full-size images (double-buffered) + arrival flags per rank
    int gatherWorld = 0, gatherRank = 0;
    DevBuf gatherImage[2], gatherFlags[2], gatherRows, gatherScratch;     // own buffers (exported)
    void* peerImage[2][IDK_MAX_PEERS] = {};                               // mapped peers (own entries = own buffers)
    void* peerFlags[2][IDK_MAX_PEERS] = {};
    bool peerMapped[IDK_MAX_PEERS] = {};
    uint32_t gatherEpoch = 0;
    double gatherTimeoutMs = 30000.0;                                     // arrival wait bound (IDKPT_GATHER_TIMEOUT_MS); a dead peer becomes an error, not a hung GPU
    int clockKHz = 1965000;
    int gatherCurrent = -1;                                               // buffer holding the last completed frame
    bool peerIsIpc = false;                                               // peers mapped with cudaIpcOpenMemHandle (else: same-process pointers)
    // global slots (IDKPT_CREATE_GLOBAL_SLOTS): per-stripe alive counts exchanged every bounce; table = [lane][parity][stripe] u64
    bool globalSlots = false;
    int nStripes = 0, nLocalStripes = 0;
    DevBuf slotTable;                                                     // own table (exported)
    void* peerSlotTable[IDK_MAX_PEERS] = {};

    // asynchronous presentation (device snapshot + D2H on a second stream, overlapping the next Compute)
    cudaStream_t copyStream = nullptr;
    cudaEvent_t snapDone = nullptr, copyDone = nullptr;
    DevBuf presentSnap;
    bool copyPending = false;

    // device BLAS build (idkpt_blas_build): its own stream and buffers, the results of the last build
    struct BlasBuild {
        cudaStream_t stream = nullptr;
        DevBuf buf[48];
        std::vector<IdkPtBlasBuildInfo> infos;
        std::vector<int> nodeBase, fragOffset;
        float phaseMs[6] = {};
    } bb;
};

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            char buf_[512];                                                                        \
            snprintf(buf_, sizeof(buf_), "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
            ctx->lastError = buf_;                                                                 \
            return IDKPT_ERR_CUDA;                                                                 \
        }                                                                                          \
    } while (0)

static int fail(IdkPtCtx* ctx, int code, const char* msg) {
    if (ctx) ctx->lastError = msg; else g_createError = msg;
    return code;
}

static cudaError_t ensure(DevBuf& b, size_t bytes) {
    if (bytes <= b.bytes && b.p) return cudaSuccess;
    if (b.p) cudaFree(b.p);
    b.p = nullptr;
    b.bytes = 0;
    if (bytes == 0) return cudaSuccess;
    cudaError_t e = cudaMalloc(&b.p, bytes);
    if (e == cudaSuccess) b.bytes = bytes;
    return e;
}

static void release(DevBuf& b) {
    if (b.p) cudaFree(b.p);
    b.p = nullptr;
    b.bytes = 0;
}

static int upload(IdkPtCtx* ctx, DevBuf& b, const void* src, size_t bytes) {
    CK(ensure(b, std::max<size_t>(bytes, 16)));
    if (bytes) CK(cudaMemcpyAsync(b.p, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return IDKPT_OK;
}

static void compute_tile_rows(IdkPtCtx* ctx) {
    ctx->rows.clear();
    for (int y = 0; y < ctx->height; y++)
        if (ctx->tileCount <= 1 || ((y / ctx->stripeH) % ctx->tileCount) == ctx->tileIndex) ctx->rows.push_back(y);
    ctx->nLocal = (uint32_t)(ctx->rows.size() * (size_t)ctx->width);
    ctx->nStripes = (ctx->height + ctx->stripeH - 1) / ctx->stripeH;
    ctx->nLocalStripes = 0;
    for (int s = 0; s < ctx->nStripes; s++)
        if (ctx->tileCount <= 1 || (s % ctx->tileCount) == ctx->tileIndex) ctx->nLocalStripes++;
}

static int configure_launches(IdkPtCtx* ctx) {
    const int stackSize = std::max(1, ctx->sc.stackSize);
    ctx->stackBytes = (size_t)stackSize * IDK_BLOCK * sizeof(uint32_t);
    if (ctx->stackBytes > 200 * 1024) return fail(ctx, IDKPT_ERR_UNSUPPORTED, "BlasStackSize too large for the shared-memory traversal stack");
    CK(cudaFuncSetAttribute(k_traverse<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ctx->stackBytes));
    CK(cudaFuncSetAttribute(k_traverse<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ctx->stackBytes));
    CK(cudaFuncSetAttribute(k_trace_rays, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ctx->stackBytes));
    CK(cudaFuncSetAttribute(k_trace_rays_any, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ctx->stackBytes));
    CK(cudaFuncSetAttribute(k_shadows_ray_traced, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ctx->stackBytes));
    ctx->traverse2Smem = (size_t)stackSize * IDK_T2_BLOCK * sizeof(uint32_t) + (size_t)ctx->treeletNodes * 32 + (IDK_STAGED_FETCH ? IDK_STAGE_BYTES : 0);
    if (const char* v = getenv("IDKPT_EXTRA_SMEM")) ctx->traverse2Smem += (size_t)std::max(0, atoi(v));   // experiment: L1 capacity sensitivity
    CK(cudaFuncSetAttribute(k_traverse2<false, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ctx->traverse2Smem));
    CK(cudaFuncSetAttribute(k_traverse2<true, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ctx->traverse2Smem));
    CK(cudaFuncSetAttribute(k_traverse2<false, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ctx->traverse2Smem));
    CK(cudaFuncSetAttribute(k_traverse2<true, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ctx->traverse2Smem));
    CK(cudaFuncSetAttribute(k_traverse2<false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ctx->traverse2Smem));
    CK(cudaFuncSetAttribute(k_traverse2<true, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ctx->traverse2Smem));
    int n = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k_traverse<false>, IDK_BLOCK, ctx->stackBytes));
    ctx->traverse1Blocks = std::max(1, n) * ctx->smCount;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k_traverse<true>, IDK_BLOCK, ctx->stackBytes));
    ctx->traverse1BlocksStats = std::max(1, n) * ctx->smCount;
    if (ctx->traverseVariant == 1) {
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k_traverse<false>, IDK_BLOCK, ctx->stackBytes));
        ctx->traverseBlocks = std::max(1, n) * ctx->smCount;
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k_traverse<true>, IDK_BLOCK, ctx->stackBytes));
        ctx->traverseBlocksStats = std::max(1, n) * ctx->smCount;
    } else if (ctx->sc.useTlas) {
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k_traverse2<false, false, true>, IDK_T2_BLOCK, ctx->traverse2Smem));
        ctx->traverseBlocks = std::max(1, n) * ctx->smCount;
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k_traverse2<true, false, true>, IDK_T2_BLOCK, ctx->traverse2Smem));
        ctx->traverseBlocksStats = std::max(1, n) * ctx->smCount;
    } else {
        if (ctx->treeletNodes) CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k_traverse2<false, true, false>, IDK_T2_BLOCK, ctx->traverse2Smem));
        else CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k_traverse2<false, false, false>, IDK_T2_BLOCK, ctx->traverse2Smem));
        ctx->traverseBlocks = std::max(1, n) * ctx->smCount;
        if (ctx->treeletNodes) CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k_traverse2<true, true, false>, IDK_T2_BLOCK, ctx->traverse2Smem));
        else CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k_traverse2<true, false, false>, IDK_T2_BLOCK, ctx->traverse2Smem));
        ctx->traverseBlocksStats = std::max(1, n) * ctx->smCount;
    }
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k_trace_rays, IDK_BLOCK, ctx->stackBytes));
    ctx->traceRaysBlocks = std::max(1, n) * ctx->smCount;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k_shade<false>, IDK_BLOCK, 0));
    ctx->shadeBlocks = std::max(1, n) * ctx->smCount;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k_compact, IDK_BLOCK, 0));
    ctx->compactBlocks = std::max(1, std::min(n, 4)) * ctx->smCount;
    // asynchronous path: `laneCount` samples in flight share the SMs; each lane's persistent traversal grid takes its share of
    // the resident-block budget (profiles/r01h_overlap_probe.json: 4 x 1 block/SM beats 4 x full grid by 24 % on a 1/8 tile)
    {
        const int lanes = std::max(1, ctx->laneCount);
        const int perSm2 = (ctx->traverseBlocks / ctx->smCount + lanes - 1) / lanes, perSm1 = (ctx->traverse1Blocks / ctx->smCount + lanes - 1) / lanes;
        ctx->traverseBlocksLane = std::max(1, perSm2) * ctx->smCount;      // profiles/r01h_lanes_probe.json: 3 lanes x 2 blocks/SM, 4+ lanes x 1
        ctx->traverse1BlocksLane = std::max(1, perSm1) * ctx->smCount;
    }
    if (const char* v = getenv("IDKPT_LANE_BLOCKS_PER_SM")) {        // developer knob
        const int b = std::max(1, atoi(v));
        ctx->traverseBlocksLane = std::min(ctx->traverseBlocks, b * ctx->smCount);
        ctx->traverse1BlocksLane = std::min(ctx->traverse1Blocks, b * ctx->smCount);
    }
    if (const char* v = getenv("IDKPT_TRAVERSE_BLOCKS_PER_SM")) {   // developer knob
        const int b = std::max(1, atoi(v));
        ctx->traverseBlocks = std::min(ctx->traverseBlocks, b * ctx->smCount);
        ctx->traverseBlocksStats = std::min(ctx->traverseBlocksStats, b * ctx->smCount);
    }
    if (const char* v = getenv("IDKPT_CARVEOUT")) {                 // developer knob: same shared-memory carve-out for every kernel
        const int pct = atoi(v);
        if (pct >= 0) {
            cudaFuncSetAttribute(k_traverse<false>, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
            cudaFuncSetAttribute(k_traverse<true>, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
            cudaFuncSetAttribute(k_traverse2<false, false, false>, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
            cudaFuncSetAttribute(k_traverse2<true, false, false>, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
            cudaFuncSetAttribute(k_shade<false>, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
            cudaFuncSetAttribute(k_shade<true>, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
            cudaFuncSetAttribute(k_compact, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
            cudaFuncSetAttribute(k_raygen, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
            cudaFuncSetAttribute(k_accumulate, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
            cudaFuncSetAttribute(k_init_sample, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
        }
    }
    return IDKPT_OK;
}

static int allocate_lane(IdkPtCtx* ctx, Lane& ln) {
    const size_t n = std::max<uint32_t>(ctx->nLocal, 1);
    CK(ensure(ln.state, n * sizeof(PathState)));
    CK(ensure(ln.aov, n * 32));
    for (int i = 0; i < 2; i++) CK(ensure(ln.alive[i], n * 4));
    CK(ensure(ln.survivors, n * 4));
    CK(ensure(ln.hits, n * 16));
    CK(ensure(ln.hitXform, n * 4));
    CK(ensure(ln.debugCost, n * 4));
    CK(ensure(ln.radiance, n * 16));
    CK(ensure(ln.aovAlbedoFinal, n * 16));
    CK(ensure(ln.aovNormalFinal, n * 16));
    CK(ensure(ln.countsDev, (IDKPT_MAX_RAY_DEPTH + 1) * sizeof(uint32_t)));
    CK(ensure(ln.tickets, 2 * (IDKPT_MAX_RAY_DEPTH + 1) * sizeof(uint32_t)));
    CK(ensure(ln.tileStatus, ((n + IDK_BLOCK * IDK_COMPACT_ITEMS - 1) / (IDK_BLOCK * IDK_COMPACT_ITEMS) + 1) * sizeof(unsigned long long)));
    if (ctx->globalSlots && ctx->tileCount > 1) CK(ensure(ln.slotDelta, (size_t)std::max(1, ctx->nLocalStripes) * sizeof(uint32_t)));
    CK(cudaMemsetAsync(ln.tileStatus.p, 0, ln.tileStatus.bytes, ctx->stream));
    if (!ln.stream) CK(cudaStreamCreateWithFlags(&ln.stream, cudaStreamNonBlocking));
    if (!ln.radianceReady) CK(cudaEventCreateWithFlags(&ln.radianceReady, cudaEventDisableTiming));
    if (!ln.accDone) CK(cudaEventCreateWithFlags(&ln.accDone, cudaEventDisableTiming));
    CK(cudaStreamSynchronize(ctx->stream));   // the status words are cleared before any lane stream touches them
    ln.epoch = ctx->epochStart;
    CK(cudaStreamSetAttribute(ln.stream, cudaStreamAttributeAccessPolicyWindow, &ctx->l2Window));   // BVH persistence on the lane streams too
    ln.accPending = false;
    ln.allocated = true;
    return IDKPT_OK;
}

static void release_lane(Lane& ln, bool keepStream) {
    DevBuf* all[] = {&ln.state, &ln.aov, &ln.alive[0], &ln.alive[1], &ln.survivors, &ln.keysTmp, &ln.sortedAlive, &ln.hits, &ln.hitXform, &ln.debugCost,
                     &ln.radiance, &ln.aovAlbedoFinal, &ln.aovNormalFinal, &ln.countsDev, &ln.tickets, &ln.tileStatus, &ln.keys, &ln.slotDelta};
    for (DevBuf* b : all) release(*b);
    idk_sort_release(ln.sortScratch);
    ln.allocated = false;
    ln.accPending = false;
    if (!keepStream) {
        if (ln.stream) { cudaStreamDestroy(ln.stream); ln.stream = nullptr; }
        if (ln.radianceReady) { cudaEventDestroy(ln.radianceReady); ln.radianceReady = nullptr; }
        if (ln.accDone) { cudaEventDestroy(ln.accDone); ln.accDone = nullptr; }
    }
}

// Wait for everything issued so far: every lane stream and the main (image) stream. Every entry point that reads or
// changes device data other than idkpt_compute / idkpt_present_async starts with this.
static cudaError_t drain(IdkPtCtx* ctx) {
    cudaError_t first = cudaSuccess;
    for (int i = 0; i < IDK_MAX_LANES; i++)
        if (ctx->lanes[i].stream) { cudaError_t e = cudaStreamSynchronize(ctx->lanes[i].stream); if (first == cudaSuccess) first = e; }
    if (ctx->stream) { cudaError_t e = cudaStreamSynchronize(ctx->stream); if (first == cudaSuccess) first = e; }
    for (int i = 0; i < IDK_MAX_LANES; i++) ctx->lanes[i].accPending = false;
    ctx->asyncPending = false;
    return first;
}

// Errors that only the device knows about (a kernel fault, a peer rank that never delivered its tile) surface at the
// next host-synchronising call.
static int check_device_errors(IdkPtCtx* ctx, cudaError_t se, const char* who) {
    if (se != cudaSuccess) {
        ctx->lastError = std::string(who) + ": kernel execution failed: " + cudaGetErrorString(se);
        return IDKPT_ERR_CUDA;
    }
    if (ctx->gatherWorld > 1) {
        uint32_t timedOut = 0;
        CK(cudaMemcpy(&timedOut, (uint32_t*)ctx->gatherScratch.p + 1, 4, cudaMemcpyDeviceToHost));
        if (timedOut) {
            cudaMemset((uint32_t*)ctx->gatherScratch.p + 1, 0, 4);
            return fail(ctx, IDKPT_ERR_CUDA, timedOut == 2u ? "idkpt_compute: timed out waiting for a peer rank's per-stripe alive counts (multi-GPU global slots)"
                                                            : "idkpt_compute: timed out waiting for a peer rank's tile (multi-GPU gather)");
        }
    }
    return IDKPT_OK;
}

// Entry points that change or expose device data wait for the samples in flight first.
#define DRAIN_PENDING(who)                                                         \
    do {                                                                           \
        if (ctx->asyncPending) {                                                   \
            cudaSetDevice(ctx->device);                                            \
            int rc_ = check_device_errors(ctx, drain(ctx), who);                   \
            if (rc_) return rc_;                                                   \
        }                                                                          \
    } while (0)

static int allocate_wavefront(IdkPtCtx* ctx) {
    const size_t n = std::max<uint32_t>(ctx->nLocal, 1);
    for (int i = 1; i < IDK_MAX_LANES; i++) if (ctx->lanes[i].allocated) release_lane(ctx->lanes[i], true);   // re-created on demand at the new size
    int rc = allocate_lane(ctx, ctx->lanes[0]);
    if (rc) return rc;
    for (int i = 0; i < 3; i++) {
        CK(ensure(ctx->images[i], n * 16));
        CK(cudaMemsetAsync(ctx->images[i].p, 0, n * 16, ctx->stream));   // Result.Fill(0), PathTracer.cs:305
    }
    CK(ensure(ctx->counters, sizeof(TraceCounters)));
    return IDKPT_OK;
}

// Device-private node layout for single-BLAS scenes: the first `pairs` sibling pairs in breadth-first order are moved to
// the front of the array (node indices 2 .. 2*pairs+1) so that the hot top of the tree is one contiguous block that a
// single bulk copy (TMA) can stage into shared memory; all remaining pairs keep their relative order. Child pointers are
// rewritten; leaves (triangle ranges) are untouched, so traversal order and results are unchanged.
static int relayout_treelet(const GpuBlasNode* src, uint32_t nodeCount, uint32_t wantPairs, std::vector<GpuBlasNode>& out) {
    const uint32_t pairCount = nodeCount / 2;            // pair p = nodes 2p, 2p+1 (pair 0 = pad + root)
    if (pairCount < 2) return 0;
    std::vector<uint32_t> newOf(pairCount, 0xFFFFFFFFu), order;
    order.reserve(pairCount);
    std::vector<uint32_t> queue;
    queue.push_back(1);                                  // children of the root
    size_t head = 0;
    const uint32_t treeletPairs = std::min(wantPairs, pairCount - 1);
    while (head < queue.size() && order.size() < treeletPairs) {
        const uint32_t p = queue[head++];
        newOf[p] = (uint32_t)order.size() + 1;
        order.push_back(p);
        for (int c = 0; c < 2; c++) {
            const GpuBlasNode& n = src[2 * p + c];
            if (n.TriCount == 0) {
                if (n.TriStartOrChild < 2 || (uint32_t)n.TriStartOrChild + 1 >= nodeCount || (n.TriStartOrChild & 1)) return -1;
                queue.push_back((uint32_t)n.TriStartOrChild / 2);
            }
        }
    }
    const uint32_t inTreelet = (uint32_t)order.size();
    for (uint32_t p = 1; p < pairCount; p++)
        if (newOf[p] == 0xFFFFFFFFu) { newOf[p] = (uint32_t)order.size() + 1; order.push_back(p); }
    out.assign(nodeCount, GpuBlasNode{});
    out[0] = src[0];
    out[1] = src[1];
    if (src[1].TriCount == 0) out[1].TriStartOrChild = 2;
    for (uint32_t i = 0; i < order.size(); i++) {
        const uint32_t p = order[i], np = i + 1;
        for (int c = 0; c < 2; c++) {
            GpuBlasNode n = src[2 * p + c];
            if (n.TriCount == 0) {
                if (n.TriStartOrChild < 2 || (uint32_t)n.TriStartOrChild + 1 >= nodeCount || (n.TriStartOrChild & 1)) return -1;
                n.TriStartOrChild = (int32_t)(2 * newOf[(uint32_t)n.TriStartOrChild / 2]);
            }
            out[2 * np + c] = n;
        }
    }
    return (int)inTreelet;
}

// Structural validation of one BLAS before its arrays reach the kernels (a malformed host array must become an error
// code, never a device fault): child pairs in range, even, and behind their parent (the builder emits DFS order, which
// also rules out cycles); leaf ranges inside the BLAS's triangle range; and the traversal stack the kernels will need
// (BLAS.ComputeRequiredStackSize, Bvh/BLAS.cs:672-702) must fit BlasStackSize. Returns nullptr or an error text.
static const char* validate_material_textures(const GpuMaterial& m, uint64_t textureCount, const char* msg) {
    const uint64_t h[5] = {m.BaseColorTexture, m.MetallicRoughnessTexture, m.NormalTexture, m.EmissiveTexture, m.TransmissionTexture};
    for (int i = 0; i < 5; i++) if (h[i] > textureCount) return msg;
    return nullptr;
}

static uint64_t material_max_handle(const GpuMaterial& m) {
    return std::max(std::max(std::max(m.BaseColorTexture, m.MetallicRoughnessTexture), std::max(m.NormalTexture, m.EmissiveTexture)), m.TransmissionTexture);
}

// Material textures: all base levels in one allocation, 256-byte aligned; 32-byte records point into it.
static int upload_textures(IdkPtCtx* ctx, const IdkPtTextureDesc* textures, uint64_t count) {
    IdkPtSceneDesc tmp = {};
    tmp.Textures = textures; tmp.TextureCount = count;
    const std::vector<size_t> off = idk_texture_offsets(&tmp);
    CK(ensure(ctx->texPixels, std::max<size_t>(off[count], 16)));
    std::vector<TexRec> recs;
    CK(idk_upload_texture_table(textures, count, off, ctx->texPixels.p, ctx->stream, recs));
    int rc;
    if ((rc = upload(ctx, ctx->texRecs, recs.data(), recs.size() * sizeof(TexRec)))) return rc;
    float lut[256];
    idk_srgb_lut(lut);
    if ((rc = upload(ctx, ctx->srgbLut, lut, sizeof(lut)))) return rc;
    CK(cudaStreamSynchronize(ctx->stream));   // recs / lut are locals
    ctx->sc.textures = (const TexRec*)ctx->texRecs.p;
    ctx->sc.textureCount = (uint32_t)count;
    ctx->sc.srgbLut = (const float*)ctx->srgbLut.p;
    return IDKPT_OK;
}

static const char* validate_blas(const GpuBlasNode* nodes, const GpuBlasDesc& d, int blasStackSize) {
    const int n = d.NodeCount;
    if (n < 4 || (n & 1)) return "idkpt_set_scene: BLAS node count must be even and >= 4";
    if (nodes[1].TriCount != 0 || nodes[1].TriStartOrChild != 2) return "idkpt_set_scene: BLAS root must be interior with children at 2 (BLAS.cs:16-22)";
    std::vector<int> req((size_t)n / 2, 0);
    for (int p = n / 2 - 1; p >= 1; p--) {
        int need[2] = {-1, -1};
        for (int c = 0; c < 2; c++) {
            const GpuBlasNode& nd = nodes[2 * p + c];
            if (nd.TriCount > 0) {
                if (nd.TriStartOrChild < 0 || (int64_t)nd.TriStartOrChild + nd.TriCount > d.TriangleCount) return "idkpt_set_scene: BLAS leaf triangle range outside the BLAS";
            } else if (nd.TriCount == 0) {
                const int ch = nd.TriStartOrChild;
                if (ch <= 2 * p || (ch & 1) || ch + 1 >= n) return "idkpt_set_scene: BLAS child index out of range / not in DFS order";
                need[c] = req[(size_t)ch / 2];
            } else {
                return "idkpt_set_scene: negative TriCount in a BLAS node";
            }
        }
        req[p] = (need[0] >= 0 && need[1] >= 0) ? std::max(need[0], need[1]) + 1 : std::max(need[0], std::max(need[1], 0));
    }
    if (req[1] > blasStackSize) return "idkpt_set_scene: BlasStackSize smaller than the traversal stack this BLAS needs";
    return nullptr;
}

// Height of a host-provided TLAS (= stack entries the walk needs); children follow their parent (validated before).
static int tlas_height(const GpuTlasNode* t, uint64_t count) {
    std::vector<int> need(count, 0);
    for (int64_t i = (int64_t)count - 1; i >= 0; i--) {
        const uint32_t w = t[i].IsLeafAndChildOrInstanceId, c = w & 0x7FFFFFFFu;
        need[i] = (w >> 31) ? 0 : 1 + std::max(need[c], need[c + 1]);
    }
    return count ? need[0] : 0;
}

static void gather_teardown(IdkPtCtx* ctx) {
    for (int b = 0; b < 2; b++)
        for (int p = 0; p < IDK_MAX_PEERS; p++) {
            if (ctx->peerMapped[p] && p != ctx->gatherRank && ctx->peerIsIpc) {
                if (ctx->peerImage[b][p]) cudaIpcCloseMemHandle(ctx->peerImage[b][p]);
                if (ctx->peerFlags[b][p]) cudaIpcCloseMemHandle(ctx->peerFlags[b][p]);
            }
            ctx->peerImage[b][p] = nullptr;
            ctx->peerFlags[b][p] = nullptr;
        }
    for (int p = 0; p < IDK_MAX_PEERS; p++) {
        if (ctx->peerMapped[p] && p != ctx->gatherRank && ctx->peerIsIpc && ctx->peerSlotTable[p]) cudaIpcCloseMemHandle(ctx->peerSlotTable[p]);
        ctx->peerSlotTable[p] = nullptr;
        ctx->peerMapped[p] = false;
    }
    ctx->peerIsIpc = false;
    release(ctx->slotTable);
    for (int i = 0; i < IDK_MAX_LANES; i++) ctx->lanes[i].slotEpoch = 0;
    for (int b = 0; b < 2; b++) { release(ctx->gatherImage[b]); release(ctx->gatherFlags[b]); }
    release(ctx->gatherRows);
    release(ctx->gatherScratch);
    ctx->gatherWorld = 0;
    ctx->gatherCurrent = -1;
    ctx->gatherEpoch = 0;
}

extern "C" {

IDKPT_API uint32_t idkpt_abi_version(void) { return IDKPT_ABI_VERSION; }

IDKPT_API const char* idkpt_last_error(IdkPtCtx* ctx) { return ctx ? ctx->lastError.c_str() : g_createError.c_str(); }

IDKPT_API int idkpt_create(const IdkPtCreateInfo* ci, IdkPtCtx** out) {
    if (!ci || !out) return fail(nullptr, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_create: null argument");
    *out = nullptr;
    if (ci->Width <= 0 || ci->Height <= 0 || ci->Width > 4096 * 4 || ci->Height > 4096 * 4)
        return fail(nullptr, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_create: invalid image size");
    int stripe = ci->TileStripeHeight > 0 ? ci->TileStripeHeight : 8;
    int tcount = ci->TileCount > 1 ? ci->TileCount : 1;
    if ((ci->Flags & IDKPT_CREATE_GLOBAL_SLOTS) && tcount > 1 && (ci->Height + stripe - 1) / stripe > IDK_MAX_STRIPES)
        return fail(nullptr, IDKPT_ERR_UNSUPPORTED, "idkpt_create: IDKPT_CREATE_GLOBAL_SLOTS supports at most 4096 stripes (raise TileStripeHeight)");
    if (tcount > 1 && (ci->TileIndex < 0 || ci->TileIndex >= tcount))
        return fail(nullptr, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_create: TileIndex out of range");
    int deviceCount = 0;
    cudaError_t e = cudaGetDeviceCount(&deviceCount);
    if (e != cudaSuccess || deviceCount == 0)
        return fail(nullptr, IDKPT_ERR_NO_DEVICE, "idkpt_create: no CUDA device (libidkpt has no CPU fallback)");
    if (ci->Device < 0 || ci->Device >= deviceCount)
        return fail(nullptr, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_create: device ordinal out of range");
    if (cudaSetDevice(ci->Device) != cudaSuccess) return fail(nullptr, IDKPT_ERR_CUDA, "idkpt_create: cudaSetDevice failed");
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, ci->Device) != cudaSuccess) return fail(nullptr, IDKPT_ERR_CUDA, "idkpt_create: cudaGetDeviceProperties failed");
    if (prop.major < 10) {
        char buf[512];
        snprintf(buf, sizeof(buf), "idkpt_create: device '%s' is sm_%d%d; libidkpt is built for sm_100a only", prop.name, prop.major, prop.minor);
        return fail(nullptr, IDKPT_ERR_NO_DEVICE, buf);
    }
    IdkPtCtx* ctx = new IdkPtCtx();
    ctx->device = ci->Device;
    ctx->smCount = prop.multiProcessorCount;
    ctx->width = ci->Width;
    ctx->height = ci->Height;
    ctx->stripeH = stripe;
    ctx->tileIndex = tcount > 1 ? ci->TileIndex : 0;
    ctx->tileCount = tcount;
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) {
        delete ctx;
        return fail(nullptr, IDKPT_ERR_CUDA, "idkpt_create: cudaStreamCreate failed");
    }
    // developer knobs (kernel variant / scheduling thresholds); results are identical for every setting
    if (const char* v = getenv("IDKPT_TRAVERSE_VARIANT")) ctx->traverseVariant = std::max(1, std::min(3, atoi(v)));
    if (const char* v = getenv("IDKPT_TUNE_SETUP")) ctx->tune.setupThreshold = std::max(1, std::min(32, atoi(v)));
    if (const char* v = getenv("IDKPT_TUNE_LEAF")) ctx->tune.leafThreshold = std::max(1, std::min(32, atoi(v)));
    if (const char* v = getenv("IDKPT_TUNE_SETUP_STAGED")) ctx->tune.setupThresholdStaged = std::max(1, std::min(32, atoi(v)));
    if (const char* v = getenv("IDKPT_PACK_ASYNC")) ctx->packAsync = atoi(v) != 0;
    if (const char* v = getenv("IDKPT_PACK_CTA")) ctx->packCta = std::max(0, atoi(v));
    if (const int fl = (ci->Flags >> 8) & 15) ctx->laneCount = std::min(IDK_MAX_LANES, fl);   // IDKPT_CREATE_LANES(n)
    ctx->globalSlots = (ci->Flags & IDKPT_CREATE_GLOBAL_SLOTS) != 0;
    if (const char* v = getenv("IDKPT_LANES")) ctx->laneCount = std::max(1, std::min(IDK_MAX_LANES, atoi(v)));
    if (const char* v = getenv("IDKPT_DEBUG_EPOCH_START")) ctx->epochStart = (uint32_t)strtoul(v, nullptr, 0) & IDK_EPOCH_MASK;
    if (const char* v = getenv("IDKPT_DEBUG_SLOT_EPOCH_START")) ctx->slotEpochStart = (uint32_t)strtoul(v, nullptr, 0) & ~1u;   // even: keeps the parity sequence
    if (const char* v = getenv("IDKPT_GATHER_TIMEOUT_MS")) ctx->gatherTimeoutMs = std::max(1.0, atof(v));
    ctx->clockKHz = prop.clockRate;
    compute_tile_rows(ctx);
    int rc = allocate_wavefront(ctx);
    if (rc != IDKPT_OK) {
        g_createError = ctx->lastError;
        idkpt_destroy(ctx);
        return rc;
    }
    ctx->sky[0] = ctx->sky[1] = ctx->sky[2] = 0.0f;
    *out = ctx;
    return IDKPT_OK;
}

IDKPT_API void idkpt_destroy(IdkPtCtx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    drain(ctx);
    DevBuf* all[] = {&ctx->nodes, &ctx->triRec, &ctx->blasTris, &ctx->positions, &ctx->descs, &ctx->instances, &ctx->xforms,
                     &ctx->meshes, &ctx->materials, &ctx->vertices, &ctx->lights, &ctx->tlas, &ctx->vtxFrame, &ctx->surfRec,
                     &ctx->images[0], &ctx->images[1], &ctx->images[2], &ctx->counters, &ctx->countLog, &ctx->skyFaces,
                     &ctx->texPixels, &ctx->texRecs, &ctx->srgbLut, &ctx->bloomDown, &ctx->bloomUp, &ctx->postConsts, &ctx->ldr,
                     &ctx->unskinned, &ctx->joints, &ctx->refitParents, &ctx->refitLocks, &ctx->scratch[0], &ctx->scratch[1], &ctx->scratch[2],
                     &ctx->tlasScratch, &ctx->oidn[0], &ctx->oidn[1], &ctx->oidn[2], &ctx->oidn[3], &ctx->denoiseWork[0], &ctx->denoiseWork[1], &ctx->denoised};
    for (DevBuf* b : all) release(*b);
    for (int i = 0; i < IDK_MAX_LANES; i++) release_lane(ctx->lanes[i], false);
    for (cudaEvent_t ev : ctx->events) cudaEventDestroy(ev);
    gather_teardown(ctx);
    if (ctx->copyStream) { cudaStreamSynchronize(ctx->copyStream); cudaStreamDestroy(ctx->copyStream); }
    if (ctx->snapDone) cudaEventDestroy(ctx->snapDone);
    if (ctx->copyDone) cudaEventDestroy(ctx->copyDone);
    release(ctx->presentSnap);
    for (DevBuf& b : ctx->bb.buf) release(b);
    if (ctx->bb.stream) cudaStreamDestroy(ctx->bb.stream);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

IDKPT_API int idkpt_set_scene(IdkPtCtx* ctx, const IdkPtSceneDesc* s) {
    if (!ctx || !s) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_set_scene: null argument");
    DRAIN_PENDING("idkpt_set_scene");
    CK(cudaSetDevice(ctx->device));
    if (!s->BlasNodes || !s->BlasTriangles || !s->BlasDescs || !s->BlasInstances || !s->MeshTransforms || !s->Meshes ||
        !s->Materials || !s->Vertices || !s->VertexPositions)
        return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_set_scene: a required array is null");
    if (s->LightCount > IDK_GPU_MAX_UBO_LIGHT_COUNT) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_set_scene: more than 256 lights");
    if (s->UseTlas) {
        // TLAS.AllocateRequiredNodes: 2n-1 nodes, root at 0, children adjacent (TLAS.cs:266-269)
        if (!s->TlasNodes || s->BlasInstanceCount == 0 || s->TlasNodeCount != 2 * s->BlasInstanceCount - 1)
            return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_set_scene: UseTlas needs 2*instances-1 TLAS nodes");
        for (uint64_t i = 0; i < s->TlasNodeCount; i++) {
            const uint32_t w = s->TlasNodes[i].IsLeafAndChildOrInstanceId, id = w & 0x7FFFFFFFu;
            if ((w >> 31) ? (id >= s->BlasInstanceCount) : (id <= i || (uint64_t)id + 1 >= s->TlasNodeCount))
                return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_set_scene: malformed TLAS node (child / instance id out of range)");
        }
        if (tlas_height(s->TlasNodes, s->TlasNodeCount) > IDK_TLAS_STACK_SIZE)
            return fail(ctx, IDKPT_ERR_UNSUPPORTED, "idkpt_set_scene: TLAS deeper than the 24-entry traversal stack of the TLAS walk (BVHIntersect.glsl:4)");
    }
    if (s->BlasTriangleCount >= (1ull << 31) || s->BlasNodeCount >= (1ull << 31)) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_set_scene: scene too large");
    // validate indices the kernels will chase (a bad host array must not become a device fault)
    for (uint64_t i = 0; i < s->BlasInstanceCount; i++) {
        if (s->BlasInstances[i].BlasId >= s->BlasDescCount || s->BlasInstances[i].MeshTransformId >= s->MeshTransformCount)
            return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_set_scene: BlasInstance references a missing BLAS or transform");
    }
    for (uint64_t i = 0; i < s->BlasDescCount; i++) {
        const GpuBlasDesc& d = s->BlasDescs[i];
        if (d.NodeOffset < 0 || d.NodeCount < 4 || (uint64_t)d.NodeOffset + d.NodeCount > s->BlasNodeCount || d.TriangleOffset < 0 ||
            (uint64_t)d.TriangleOffset + d.TriangleCount > s->BlasTriangleCount)
            return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_set_scene: GpuBlasDesc range outside the node/triangle arrays");
        if (d.RequiredStackSize > s->BlasStackSize)
            return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_set_scene: BlasStackSize smaller than a BLAS's RequiredStackSize");
        if (const char* err = validate_blas(s->BlasNodes + d.NodeOffset, d, s->BlasStackSize)) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, err);
    }
    for (uint64_t i = 0; i < s->MeshCount; i++)
        if (s->Meshes[i].MaterialId < 0 || (uint64_t)s->Meshes[i].MaterialId >= s->MaterialCount)
            return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_set_scene: GpuMesh.MaterialId out of range");
    if (const char* terr = idk_validate_textures(s)) {
        ctx->lastError = std::string("idkpt_set_scene: ") + terr;
        return strstr(terr, "not supported") ? IDKPT_ERR_UNSUPPORTED : IDKPT_ERR_INVALID_ARGUMENT;
    }

    // triangle vertex ids must index the position / vertex arrays
    // (checked on the host copy: cheap relative to the BVH build that produced it)
    for (uint64_t i = 0; i < s->BlasTriangleCount; i++) {
        const GpuBlasTriangle& t = s->BlasTriangles[i];
        const uint64_t lim = std::min(s->VertexPositionCount, s->VertexCount);
        if ((uint64_t)(uint32_t)t.X >= lim || (uint64_t)(uint32_t)t.Y >= lim || (uint64_t)(uint32_t)t.Z >= lim || t.MeshId < 0 || (uint64_t)t.MeshId >= s->MeshCount)
            return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_set_scene: GpuBlasTriangle index out of range");
    }
    if ((size_t)std::max(1, s->BlasStackSize) * IDK_BLOCK * sizeof(uint32_t) > 200 * 1024)
        return fail(ctx, IDKPT_ERR_UNSUPPORTED, "BlasStackSize too large for the shared-memory traversal stack");

    // Every host-side check has passed; from here on device arrays are overwritten / reallocated. Until the new scene is
    // complete the context has NO scene: a failure below (CUDA error, out of memory) must not leave the previous scene's
    // pointers and counts looking valid.
    ctx->haveScene = false;
    int rc;
    // nodes and triangle records share one allocation ("bvh"): [nodes | triRec], so that one L2 access-policy window covers both
    const size_t nodeBytes = ((s->BlasNodeCount * sizeof(GpuBlasNode)) + 255) & ~(size_t)255;
    const size_t triRecBytes = std::max<size_t>(s->BlasTriangleCount, 1) * (16 * IDK_TRI_STRIDE);
    CK(ensure(ctx->nodes, nodeBytes + triRecBytes));
    ctx->treeletNodes = 0;
    std::vector<GpuBlasNode> relaid;
    {
        const char* env = getenv("IDKPT_TREELET_PAIRS");
        const uint32_t wantPairs = env ? (uint32_t)std::min(768, std::max(0, atoi(env))) : 0u;   // default off: measured no gain over the L1 (profiles/r01d_treelet.txt)
        if (wantPairs > 0 && !s->UseTlas && s->BlasInstanceCount == 1 && s->BlasDescCount == 1 && s->BlasDescs[0].NodeOffset == 0 &&
            s->BlasNodeCount < (1ull << 31) && (s->BlasNodeCount & 1) == 0) {
            const int got = relayout_treelet(s->BlasNodes, (uint32_t)s->BlasNodeCount, wantPairs, relaid);
            if (got > 0) ctx->treeletNodes = 2 * got + 2;
            else relaid.clear();
        }
    }
    CK(cudaMemcpyAsync(ctx->nodes.p, relaid.empty() ? s->BlasNodes : relaid.data(), s->BlasNodeCount * sizeof(GpuBlasNode), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));   // `relaid` is a local
    if ((rc = upload(ctx, ctx->blasTris, s->BlasTriangles, s->BlasTriangleCount * sizeof(GpuBlasTriangle)))) return rc;
    if ((rc = upload(ctx, ctx->positions, s->VertexPositions, s->VertexPositionCount * sizeof(PackedVec3)))) return rc;
    if ((rc = upload(ctx, ctx->descs, s->BlasDescs, s->BlasDescCount * sizeof(GpuBlasDesc)))) return rc;
    if ((rc = upload(ctx, ctx->instances, s->BlasInstances, s->BlasInstanceCount * sizeof(GpuBlasInstance)))) return rc;
    if ((rc = upload(ctx, ctx->xforms, s->MeshTransforms, s->MeshTransformCount * sizeof(GpuMeshTransform)))) return rc;
    if ((rc = upload(ctx, ctx->meshes, s->Meshes, s->MeshCount * sizeof(GpuMesh)))) return rc;
    if ((rc = upload(ctx, ctx->materials, s->Materials, s->MaterialCount * sizeof(GpuMaterial)))) return rc;
    if ((rc = upload(ctx, ctx->vertices, s->Vertices, s->VertexCount * sizeof(GpuVertex)))) return rc;
    if ((rc = upload(ctx, ctx->lights, s->Lights, s->LightCount * sizeof(GpuLight)))) return rc;
    if ((rc = upload(ctx, ctx->tlas, s->TlasNodes, s->UseTlas ? s->TlasNodeCount * sizeof(GpuTlasNode) : 0))) return rc;
    if ((rc = upload_textures(ctx, s->Textures, s->TextureCount))) return rc;
    ctx->hostMaterialMaxHandle.assign(s->MaterialCount, 0);
    for (uint64_t i = 0; i < s->MaterialCount; i++) ctx->hostMaterialMaxHandle[i] = material_max_handle(s->Materials[i]);

    CK(ensure(ctx->vtxFrame, std::max<size_t>(s->VertexCount, 1) * 32));
    CK(ensure(ctx->surfRec, std::max<size_t>(s->MeshCount, 1) * 80));
    if (s->VertexCount) {
        const uint32_t nv = (uint32_t)s->VertexCount;
        k_prepare_vertices<<<(nv + 255) / 256, 256, 0, ctx->stream>>>((const uint4*)ctx->vertices.p, (float4*)ctx->vtxFrame.p, nv);
    }
    if (s->MeshCount) {
        const uint32_t nm = (uint32_t)s->MeshCount;
        k_prepare_surfaces<<<(nm + 255) / 256, 256, 0, ctx->stream>>>((const GpuMesh*)ctx->meshes.p, (const GpuMaterial*)ctx->materials.p, (float4*)ctx->surfRec.p, nm);
    }
    CK(cudaGetLastError());
    if (s->BlasTriangleCount) {
        const uint32_t n = (uint32_t)s->BlasTriangleCount;
        k_prepare_triangles<<<(n + 255) / 256, 256, 0, ctx->stream>>>((const int4*)ctx->blasTris.p, (const float*)ctx->positions.p, (float4*)((char*)ctx->nodes.p + nodeBytes), n);
        CK(cudaGetLastError());
    }

    DeviceScene& sc = ctx->sc;
    sc.nodes = (const float4*)ctx->nodes.p;
    sc.triRec = (const float4*)((char*)ctx->nodes.p + nodeBytes);
    sc.blasTris = (const int4*)ctx->blasTris.p;
    sc.descs = (const GpuBlasDesc*)ctx->descs.p;
    sc.instances = (const GpuBlasInstance*)ctx->instances.p;
    sc.xforms = (const float4*)ctx->xforms.p;
    sc.meshes = (const GpuMesh*)ctx->meshes.p;
    sc.materials = (const GpuMaterial*)ctx->materials.p;
    sc.vertices = (const uint4*)ctx->vertices.p;
    sc.lights = (const GpuLight*)ctx->lights.p;
    sc.instanceCount = (uint32_t)s->BlasInstanceCount;
    sc.lightCount = (uint32_t)s->LightCount;
    sc.skyR = ctx->sky[0]; sc.skyG = ctx->sky[1]; sc.skyB = ctx->sky[2];
    sc.skyFaces = ctx->skyFaceSize ? (const float4*)ctx->skyFaces.p : nullptr;
    sc.skyFaceSize = ctx->skyFaceSize;
    sc.stackSize = std::max(1, s->BlasStackSize);
    sc.tlasNodes = (const float4*)ctx->tlas.p;
    sc.useTlas = s->UseTlas ? 1 : 0;
    sc.treeletNodes = ctx->treeletNodes;
    sc.vtxFrame = (const float4*)ctx->vtxFrame.p;
    sc.surfRec = (const float4*)ctx->surfRec.p;
    sc.textures = (const TexRec*)ctx->texRecs.p;
    sc.textureCount = (uint32_t)s->TextureCount;
    sc.srgbLut = (const float*)ctx->srgbLut.p;
    ctx->counts = *s;
    ctx->hostDescs.assign(s->BlasDescs, s->BlasDescs + s->BlasDescCount);
    ctx->nodeBytes = nodeBytes;
    if ((rc = configure_launches(ctx))) return rc;
    // Keep the BVH resident in the 126 MB L2: persisting access-policy window over [nodes | triRec] on the render stream.
    // The wavefront buffers (hundreds of MB per frame) stream through the rest of the cache without evicting the tree.
    {
        cudaDeviceProp prop;
        CK(cudaGetDeviceProperties(&prop, ctx->device));
        const char* env = getenv("IDKPT_L2_PERSIST");
        const bool want = !(env && atoi(env) == 0);
        cudaStreamAttrValue& attr = ctx->l2Window;
        memset(&attr, 0, sizeof(attr));
        if (want && prop.persistingL2CacheMaxSize > 0 && prop.accessPolicyMaxWindowSize > 0) {
            const size_t bvhBytes = nodeBytes + triRecBytes;
            const size_t setAside = std::min<size_t>((size_t)prop.persistingL2CacheMaxSize, std::max<size_t>(bvhBytes, 1 << 20));
            CK(cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, setAside));
            const size_t window = std::min<size_t>(bvhBytes, (size_t)prop.accessPolicyMaxWindowSize);
            attr.accessPolicyWindow.base_ptr = ctx->nodes.p;
            attr.accessPolicyWindow.num_bytes = window;
            attr.accessPolicyWindow.hitRatio = window <= setAside ? 1.0f : (float)((double)setAside / (double)window);
            attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
            attr.accessPolicyWindow.missProp = cudaAccessPropertyNormal;
        } else {
            attr.accessPolicyWindow.num_bytes = 0;
        }
        CK(cudaStreamSetAttribute(ctx->stream, cudaStreamAttributeAccessPolicyWindow, &attr));
        for (int i = 0; i < IDK_MAX_LANES; i++)    // the asynchronous path launches traverse / shade on the lane streams
            if (ctx->lanes[i].stream) CK(cudaStreamSetAttribute(ctx->lanes[i].stream, cudaStreamAttributeAccessPolicyWindow, &attr));
    }
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->haveScene = true;
    ctx->accumulatedSamples = 0;
    return IDKPT_OK;
}

IDKPT_API int idkpt_update_range(IdkPtCtx* ctx, IdkPtArrayId which, uint64_t first, uint64_t count, const void* data) {
    if (!ctx || !data) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_update_range: null argument");
    DRAIN_PENDING("idkpt_update_range");
    if (!ctx->haveScene) return fail(ctx, IDKPT_ERR_NO_SCENE, "idkpt_update_range: no scene");
    CK(cudaSetDevice(ctx->device));
    DevBuf* b = nullptr;
    size_t elem = 0;
    uint64_t limit = 0;
    switch (which) {
        case IDKPT_ARRAY_MESH_TRANSFORMS: b = &ctx->xforms; elem = sizeof(GpuMeshTransform); limit = ctx->counts.MeshTransformCount; break;
        case IDKPT_ARRAY_MESHES: b = &ctx->meshes; elem = sizeof(GpuMesh); limit = ctx->counts.MeshCount; break;
        case IDKPT_ARRAY_MATERIALS: b = &ctx->materials; elem = sizeof(GpuMaterial); limit = ctx->counts.MaterialCount; break;
        case IDKPT_ARRAY_LIGHTS: b = &ctx->lights; elem = sizeof(GpuLight); limit = ctx->counts.LightCount; break;
        case IDKPT_ARRAY_TLAS_NODES: b = &ctx->tlas; elem = sizeof(GpuTlasNode); limit = ctx->counts.UseTlas ? ctx->counts.TlasNodeCount : 0; break;
        default: return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_update_range: unknown array id");
    }
    if (first > limit || count > limit - first) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_update_range: range outside the array");
    if (which == IDKPT_ARRAY_MESHES) {
        const GpuMesh* m = (const GpuMesh*)data;
        for (uint64_t i = 0; i < count; i++)
            if (m[i].MaterialId < 0 || (uint64_t)m[i].MaterialId >= ctx->counts.MaterialCount)
                return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_update_range: GpuMesh.MaterialId out of range");
    }
    if (which == IDKPT_ARRAY_TLAS_NODES) {
        const GpuTlasNode* t = (const GpuTlasNode*)data;
        for (uint64_t i = 0; i < count; i++) {
            const uint32_t w = t[i].IsLeafAndChildOrInstanceId, id = w & 0x7FFFFFFFu;
            if ((w >> 31) ? (id >= ctx->counts.BlasInstanceCount) : (id <= first + i || (uint64_t)id + 1 >= ctx->counts.TlasNodeCount))
                return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_update_range: malformed TLAS node (child / instance id out of range)");
        }
        if (first == 0 && count == ctx->counts.TlasNodeCount && tlas_height(t, count) > IDK_TLAS_STACK_SIZE)
            return fail(ctx, IDKPT_ERR_UNSUPPORTED, "idkpt_update_range: TLAS deeper than the 24-entry traversal stack of the TLAS walk (BVHIntersect.glsl:4)");
    }
    if (which == IDKPT_ARRAY_MATERIALS) {
        const GpuMaterial* m = (const GpuMaterial*)data;
        for (uint64_t i = 0; i < count; i++)
            if (const char* err = validate_material_textures(m[i], ctx->counts.TextureCount, "idkpt_update_range: material texture handle outside the texture table"))
                return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, err);
        for (uint64_t i = 0; i < count; i++) ctx->hostMaterialMaxHandle[first + i] = material_max_handle(m[i]);
    }
    CK(cudaMemcpyAsync((char*)b->p + first * elem, data, count * elem, cudaMemcpyHostToDevice, ctx->stream));
    if ((which == IDKPT_ARRAY_MESHES || which == IDKPT_ARRAY_MATERIALS) && ctx->counts.MeshCount) {
        const uint32_t nm = (uint32_t)ctx->counts.MeshCount;   // refresh the per-mesh surface records
        k_prepare_surfaces<<<(nm + 255) / 256, 256, 0, ctx->stream>>>((const GpuMesh*)ctx->meshes.p, (const GpuMaterial*)ctx->materials.p, (float4*)ctx->surfRec.p, nm);
        CK(cudaGetLastError());
    }
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->accumulatedSamples = 0;
    return IDKPT_OK;
}

IDKPT_API int idkpt_set_sky(IdkPtCtx* ctx, const IdkPtSkyDesc* sky) {
    if (!ctx || !sky) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_set_sky: null argument");
    DRAIN_PENDING("idkpt_set_sky");
    if (sky->FaceSize < 0 || sky->FaceSize > 8192) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_set_sky: invalid FaceSize");
    CK(cudaSetDevice(ctx->device));
    if (sky->FaceSize > 0) {
        const size_t faceBytes = (size_t)sky->FaceSize * sky->FaceSize * 16;
        for (int i = 0; i < 6; i++) if (!sky->Faces[i]) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_set_sky: a cubemap face is null");
        CK(ensure(ctx->skyFaces, 6 * faceBytes));
        for (int i = 0; i < 6; i++) CK(cudaMemcpyAsync((char*)ctx->skyFaces.p + i * faceBytes, sky->Faces[i], faceBytes, cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    ctx->skyFaceSize = sky->FaceSize;
    for (int i = 0; i < 3; i++) ctx->sky[i] = sky->Color[i];
    ctx->sc.skyR = ctx->sky[0]; ctx->sc.skyG = ctx->sky[1]; ctx->sc.skyB = ctx->sky[2];
    ctx->sc.skyFaces = ctx->skyFaceSize ? (const float4*)ctx->skyFaces.p : nullptr;
    ctx->sc.skyFaceSize = ctx->skyFaceSize;
    ctx->accumulatedSamples = 0;
    return IDKPT_OK;
}

// Replaces the texture table (SURVEY 8b idkpt_set_textures): e.g. streamed-in higher-resolution images. Handles already
// stored in the materials must stay valid.
IDKPT_API int idkpt_set_textures(IdkPtCtx* ctx, const IdkPtTextureDesc* textures, uint64_t count) {
    if (!ctx || (!textures && count)) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_set_textures: null argument");
    DRAIN_PENDING("idkpt_set_textures");
    if (!ctx->haveScene) return fail(ctx, IDKPT_ERR_NO_SCENE, "idkpt_set_textures: no scene");
    IdkPtSceneDesc tmp = {};
    tmp.Textures = textures; tmp.TextureCount = count;
    if (const char* terr = idk_validate_textures(&tmp)) {
        ctx->lastError = std::string("idkpt_set_textures: ") + terr;
        return strstr(terr, "not supported") ? IDKPT_ERR_UNSUPPORTED : IDKPT_ERR_INVALID_ARGUMENT;
    }
    for (uint64_t h : ctx->hostMaterialMaxHandle)
        if (h > count) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_set_textures: a material references a texture beyond the new table");
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    int rc = upload_textures(ctx, textures, count);
    if (rc) return rc;
    ctx->counts.TextureCount = count;
    ctx->accumulatedSamples = 0;
    return IDKPT_OK;
}

IDKPT_API int idkpt_resize(IdkPtCtx* ctx, int32_t width, int32_t height) {
    if (!ctx) return IDKPT_ERR_INVALID_ARGUMENT;
    DRAIN_PENDING("idkpt_resize");
    if (width <= 0 || height <= 0 || width > 16384 || height > 16384) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_resize: invalid size");
    if (ctx->globalSlots && ctx->tileCount > 1 && (height + ctx->stripeH - 1) / ctx->stripeH > IDK_MAX_STRIPES)
        return fail(ctx, IDKPT_ERR_UNSUPPORTED, "idkpt_resize: IDKPT_CREATE_GLOBAL_SLOTS supports at most 4096 stripes");
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    if (ctx->copyPending) { CK(cudaEventSynchronize(ctx->copyDone)); ctx->copyPending = false; }
    gather_teardown(ctx);   // the exported full-frame buffers have the old size: peers must export / import again
    ctx->haveDenoised = false;
    for (int i = 0; i < 4; i++) release(ctx->oidn[i]);
    release(ctx->denoiseWork[0]); release(ctx->denoiseWork[1]); release(ctx->denoised);
    ctx->width = width;
    ctx->height = height;
    compute_tile_rows(ctx);
    int rc = allocate_wavefront(ctx);
    if (rc) return rc;
    for (int i = 0; i < IDK_MAX_LANES; i++) {
        release(ctx->lanes[i].keys);
        release(ctx->lanes[i].keysTmp);
        release(ctx->lanes[i].sortedAlive);
    }
    ctx->accumulatedSamples = 0;
    return IDKPT_OK;
}

IDKPT_API int idkpt_reset_accumulation(IdkPtCtx* ctx) {
    if (!ctx) return IDKPT_ERR_INVALID_ARGUMENT;
    ctx->accumulatedSamples = 0;
    return IDKPT_OK;
}

IDKPT_API uint32_t idkpt_accumulated_samples(IdkPtCtx* ctx) { return ctx ? ctx->accumulatedSamples : 0; }

IDKPT_API int idkpt_set_accumulated_samples(IdkPtCtx* ctx, uint32_t n) {
    if (!ctx) return IDKPT_ERR_INVALID_ARGUMENT;
    ctx->accumulatedSamples = n;
    return IDKPT_OK;
}

struct EventPool {
    IdkPtCtx* ctx;
    size_t used = 0;
    struct Span { size_t a, b; int cat; int bounce; };
    std::vector<Span> spans;
    bool enabled;
    cudaEvent_t get() {
        if (used == ctx->events.size()) {
            cudaEvent_t e;
            cudaEventCreate(&e);
            ctx->events.push_back(e);
        }
        return ctx->events[used++];
    }
    size_t begin() {
        if (!enabled) return 0;
        size_t i = used;
        cudaEventRecord(get(), ctx->stream);
        return i;
    }
    void end(size_t a, int cat, int bounce = -1) {
        if (!enabled) return;
        size_t i = used;
        cudaEventRecord(get(), ctx->stream);
        spans.push_back({a, i, cat, bounce});
    }
};

IDKPT_API int idkpt_stream_handle(IdkPtCtx* ctx, void** stream) {
    if (!ctx || !stream) return IDKPT_ERR_INVALID_ARGUMENT;
    *stream = (void*)ctx->stream;
    return IDKPT_OK;
}

IDKPT_API int idkpt_sync(IdkPtCtx* ctx) {
    if (!ctx) return IDKPT_ERR_INVALID_ARGUMENT;
    CK(cudaSetDevice(ctx->device));
    int rc = check_device_errors(ctx, drain(ctx), "idkpt_sync");
#if IDK_PHASE_STATS
    if (rc == IDKPT_OK && ctx->counters.p) {   // instrumented build: phase statistics of everything since the last dump (asynchronous path included)
        TraceCounters tc;
        CK(cudaMemcpy(&tc, ctx->counters.p, sizeof(tc), cudaMemcpyDeviceToHost));
        CK(cudaMemset(ctx->counters.p, 0, sizeof(tc)));
        const double bs = 32.0 * (double)tc.phaseRounds[1];
        fprintf(stderr, "[idkpt phase stats @sync] rounds SETUP %llu BOX %llu LEAF %llu | lanes/round SETUP %.1f BOX %.1f LEAF %.1f | BOX lane slots: active %.1f%% wait-SETUP %.1f%% wait-LEAF %.1f%% exited %.1f%%\n",
                tc.phaseRounds[0], tc.phaseRounds[1], tc.phaseRounds[2], (double)tc.phaseLanes[0] / std::max(1ull, tc.phaseRounds[0]), (double)tc.phaseLanes[1] / std::max(1ull, tc.phaseRounds[1]),
                (double)tc.phaseLanes[2] / std::max(1ull, tc.phaseRounds[2]), 100.0 * tc.phaseLanes[1] / std::max(1.0, bs), 100.0 * tc.boxIdle[0] / std::max(1.0, bs), 100.0 * tc.boxIdle[1] / std::max(1.0, bs), 100.0 * tc.boxIdle[2] / std::max(1.0, bs));
    }
#endif
    return rc;
}

IDKPT_API int idkpt_compute(IdkPtCtx* ctx, const GpuPerFrameData* frame, const IdkPtSettings* st, IdkPtStats* stats) {
    if (!ctx || !frame || !st) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_compute: null argument");
    if (!ctx->haveScene) return fail(ctx, IDKPT_ERR_NO_SCENE, "idkpt_compute: idkpt_set_scene has not been called");
    if (st->RayDepth < 1 || st->RayDepth > IDKPT_MAX_RAY_DEPTH) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_compute: RayDepth out of range");
    if (st->SamplesPerPixel < 1) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_compute: SamplesPerPixel must be >= 1");
    CK(cudaSetDevice(ctx->device));
    if (stats) memset(stats, 0, sizeof(*stats));
    const uint32_t n = ctx->nLocal;
    if (n == 0) { ctx->accumulatedSamples += st->SamplesPerPixel; return IDKPT_OK; }

    const bool wantStats = st->CollectStats != 0 || st->Gpu.DoDebugBVHTraversal != 0;
    const bool sorting = st->DoRaySorting != 0;
    const bool aovs = st->OutputAOVs != 0;
    // stats == NULL: asynchronous. Samples are issued round-robin onto the lanes and the call returns without waiting
    // (idkpt_sync, or any call that reads device data, waits). With stats the call is synchronous and runs one sample at
    // a time on lane 0, exactly the sequence the per-kernel timings describe.
    const bool async = stats == nullptr && !wantStats && !ctx->exportEnabled && ctx->laneCount > 1;
    const bool globalSlots = ctx->globalSlots && ctx->tileCount > 1;
    if (globalSlots && ctx->gatherWorld < 2)
        return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_compute: IDKPT_CREATE_GLOBAL_SLOTS needs the peers connected (idkpt_gather_import / idkpt_gather_connect)");
    if (globalSlots && sorting)
        return fail(ctx, IDKPT_ERR_UNSUPPORTED, "idkpt_compute: ray sorting reorders the slots by a tile-local key sort; not available with IDKPT_CREATE_GLOBAL_SLOTS");
    if (!async && ctx->asyncPending) {
        int rc = check_device_errors(ctx, drain(ctx), "idkpt_compute");
        if (rc) return rc;
    }

    FrameParams f;
    memcpy(f.invProj, frame->InvProjection, sizeof(f.invProj));
    memcpy(f.invView, frame->InvView, sizeof(f.invView));
    memcpy(f.viewPos, frame->ViewPos, sizeof(f.viewPos));
    f.focalLength = st->Gpu.FocalLength;
    f.lenseRadius = st->Gpu.LenseRadius;
    f.width = ctx->width; f.height = ctx->height;
    f.stripeH = ctx->stripeH; f.tileIndex = ctx->tileIndex; f.tileCount = ctx->tileCount;
    f.doDebugTraversal = st->Gpu.DoDebugBVHTraversal;
    f.doTraceLights = st->Gpu.DoTraceLights;
    f.doRussianRoulette = st->Gpu.DoRussianRoulette;

    EventPool ev{ctx, 0, {}, stats != nullptr};
    const size_t evTotal = ev.begin();
    uint32_t launches = 0, traverseLaunches = 0;
    std::vector<uint32_t> hostCounts(stats ? (size_t)st->SamplesPerPixel * (IDKPT_MAX_RAY_DEPTH + 1) : 0, 0);
    DevBuf& countLog = ctx->countLog;   // per-sample copy of counts for the stats (device-side, read once at the end)
    if (stats) CK(ensure(countLog, hostCounts.size() * sizeof(uint32_t)));
    if (wantStats) CK(cudaMemsetAsync(ctx->counters.p, 0, sizeof(TraceCounters), ctx->stream));

    const dim3 rgGrid((ctx->width + 7) / 8, (ctx->height + 7) / 8), rgBlock(8, 8);
    const int accBlocks = std::min<int>((int)((n + IDK_BLOCK - 1) / IDK_BLOCK), ctx->smCount * 8);

    for (int s = 0; s < st->SamplesPerPixel; s++) {
        Lane& ln = ctx->lanes[async ? ctx->nextLane : 0];
        if (async) {
            ctx->nextLane = (ctx->nextLane + 1) % ctx->laneCount;
            if (!ln.allocated)   // first asynchronous call (or first after a resize): bring up every lane now, not one per call
                for (int i = 0; i < ctx->laneCount; i++)
                    if (!ctx->lanes[i].allocated) { int rc = allocate_lane(ctx, ctx->lanes[i]); if (rc) return rc; }
            if (ln.accPending) CK(cudaStreamWaitEvent(ln.stream, ln.accDone, 0));   // its previous sample's radiance has been consumed
        }
        const cudaStream_t ls = async ? ln.stream : ctx->stream;   // the wavefront chain of this sample
        if (sorting) {
            CK(ensure(ln.keys, (size_t)n * 4));
            CK(ensure(ln.keysTmp, (size_t)n * 4));
            CK(ensure(ln.sortedAlive, (size_t)n * 4));
            if (idk_sort_prepare(ln.sortScratch, n)) return fail(ctx, IDKPT_ERR_OUT_OF_MEMORY, "idkpt_compute: sort scratch allocation failed");
        }
        uint32_t* counts = (uint32_t*)ln.countsDev.p;
        uint32_t* tickets = (uint32_t*)ln.tickets.p;
        f.accumulatedSamples = ctx->accumulatedSamples;
        // zero the alive counts and work tickets, counts[0] = n (every pixel of the tile traces a primary ray)
        k_init_sample<<<1, 256, 0, ls>>>(counts, IDKPT_MAX_RAY_DEPTH + 1, tickets, 2 * (IDKPT_MAX_RAY_DEPTH + 1), n);
        launches++;

        size_t e0 = ev.begin();
        k_raygen<<<rgGrid, rgBlock, 0, ls>>>(f, (PathState*)ln.state.p);
        ev.end(e0, 3);
        launches++;

        for (int j = 0; j < st->RayDepth; j++) {
            const bool first = j == 0;
            const bool last = j == st->RayDepth - 1;
            // alive list of this bounce: slot -> tile pixel (identity for the first hit)
            const uint32_t* alive = first ? nullptr : (const uint32_t*)ln.alive[j & 1].p;
            if (sorting && j > 1) {
                // PathTracer.RaySorting(), PathTracer.cs:273-297: stable sort of the alive list by cached key
                e0 = ev.begin();
                int nl = idk_sort_by_key(ln.sortScratch, (const uint32_t*)ln.keys.p, alive, (uint32_t*)ln.sortedAlive.p, counts + j, n, ctx->smCount, ls);
                ev.end(e0, 2);
                if (nl < 0) return fail(ctx, IDKPT_ERR_CUDA, "idkpt_compute: sort launch failed");
                launches += (uint32_t)nl;
                alive = (const uint32_t*)ln.sortedAlive.p;
            }

            if (globalSlots && !first) {
                // per-stripe alive counts of this bounce to every peer, everybody's counts back: global slot = local slot + delta[stripe]
                SlotExchangeArgs xa;
                memset(&xa, 0, sizeof(xa));
                // 32-bit epoch (~20 days at 2,400 exchanges per second and lane). Wrap: 0 means "nothing published" and the parity
                // must keep alternating (0xFFFFFFFF is odd), so the successor of 0xFFFFFFFF is 2. A table word always holds the
                // epoch of two exchanges ago, so a reused value can never be mistaken for the current one.
                if (++ln.slotEpoch == 0u) ln.slotEpoch = 2u;
                const uint32_t epoch = ln.slotEpoch;
                const size_t laneIdx = (size_t)(&ln - ctx->lanes);
                for (int p = 0; p < ctx->gatherWorld; p++)
                    xa.peerTable[p] = (unsigned long long*)ctx->peerSlotTable[p] + (laneIdx * 2 + (epoch & 1u)) * (size_t)ctx->nStripes;
                xa.alive = alive; xa.count = counts + j;
                xa.delta = (uint32_t*)ln.slotDelta.p;
                xa.timedOut = (uint32_t*)ctx->gatherScratch.p + 1;
                xa.timeoutCycles = (long long)(ctx->gatherTimeoutMs * (double)ctx->clockKHz);
                xa.epoch = epoch;
                xa.world = ctx->gatherWorld; xa.rank = ctx->gatherRank;
                xa.stripePixels = (uint32_t)ctx->stripeH * (uint32_t)ctx->width;
                xa.nLocalStripes = (uint32_t)ctx->nLocalStripes; xa.nStripes = (uint32_t)ctx->nStripes;
                k_slot_exchange<<<1, 256, 0, ls>>>(xa);
                launches++;
            }

            TraverseArgs ta;
            ta.sc = ctx->sc;
            ta.state = (const PathState*)ln.state.p;
            ta.perm = alive;
            ta.count = counts + j;
            ta.ticket = tickets + 2 * j;
            ta.hits = (HitRec*)ln.hits.p;
            ta.hitXform = (uint32_t*)ln.hitXform.p;
            ta.debugCost = (float*)ln.debugCost.p;
            ta.counters = (TraceCounters*)ctx->counters.p;
            ta.traceLights = st->Gpu.DoTraceLights;
            ta.bounce = j;
            e0 = ev.begin();
            if (ctx->traverseVariant == 1 || (ctx->traverseVariant == 3 && first)) {
                if (wantStats) k_traverse<true><<<ctx->traverse1BlocksStats, IDK_BLOCK, ctx->stackBytes, ls>>>(ta);
                else k_traverse<false><<<async ? ctx->traverse1BlocksLane : ctx->traverse1Blocks, IDK_BLOCK, ctx->stackBytes, ls>>>(ta);
            } else {
                const int tb = async ? ctx->traverseBlocksLane : ctx->traverseBlocks;
                TraverseTuning tune = ctx->tune;
                tune.packRays = (async && ctx->packAsync) ? 1 : 0;
                tune.packCta = (async && ctx->packAsync) ? ctx->packCta : 0;
                if (ctx->sc.useTlas) {       // the TLAS walk is a fourth phase of the production kernel (BVHIntersect.glsl:205-272)
                    if (wantStats) k_traverse2<true, false, true><<<ctx->traverseBlocksStats, IDK_T2_BLOCK, ctx->traverse2Smem, ls>>>(ta, tune);
                    else k_traverse2<false, false, true><<<tb, IDK_T2_BLOCK, ctx->traverse2Smem, ls>>>(ta, tune);
                } else if (ctx->treeletNodes) {
                    if (wantStats) k_traverse2<true, true, false><<<ctx->traverseBlocksStats, IDK_T2_BLOCK, ctx->traverse2Smem, ls>>>(ta, tune);
                    else k_traverse2<false, true, false><<<tb, IDK_T2_BLOCK, ctx->traverse2Smem, ls>>>(ta, tune);
                } else {
                    if (wantStats) k_traverse2<true, false, false><<<ctx->traverseBlocksStats, IDK_T2_BLOCK, ctx->traverse2Smem, ls>>>(ta, tune);
                    else k_traverse2<false, false, false><<<tb, IDK_T2_BLOCK, ctx->traverse2Smem, ls>>>(ta, tune);
                }
            }
            ev.end(e0, 0, j);
            launches++;
            traverseLaunches++;

            ShadeArgs sa;
            sa.sc = ctx->sc;
            sa.f = f;
            sa.state = (PathState*)ln.state.p;
            sa.aov = (float4*)ln.aov.p;
            sa.alive = alive;
            sa.hits = (const HitRec*)ln.hits.p;
            sa.hitXform = (const uint32_t*)ln.hitXform.p;
            sa.debugCost = (const float*)ln.debugCost.p;
            sa.count = counts + j;
            sa.survivors = (uint32_t*)ln.survivors.p;
            sa.keysTmp = sorting ? (uint32_t*)ln.keysTmp.p : nullptr;
            sa.radiance = (float4*)ln.radiance.p;
            sa.aovAlbedoFinal = (float4*)ln.aovAlbedoFinal.p;
            sa.aovNormalFinal = (float4*)ln.aovNormalFinal.p;
            sa.slotDelta = (globalSlots && !first) ? (const uint32_t*)ln.slotDelta.p : nullptr;
            sa.stripePixels = (uint32_t)ctx->stripeH * (uint32_t)ctx->width;
            sa.exportState = ctx->exportEnabled ? 1 : 0;
            sa.firstHit = first ? 1 : 0;
            sa.lastBounce = last ? 1 : 0;
            sa.outputAovs = aovs ? 1 : 0;
            e0 = ev.begin();
            if (ctx->sc.textureCount) k_shade<true><<<ctx->shadeBlocks, IDK_BLOCK, 0, ls>>>(sa);
            else k_shade<false><<<ctx->shadeBlocks, IDK_BLOCK, 0, ls>>>(sa);
            launches++;
            if (!last) {
                CompactArgs ca;
                ca.survivors = (const uint32_t*)ln.survivors.p;
                ca.keysTmp = sorting ? (const uint32_t*)ln.keysTmp.p : nullptr;
                ca.count = counts + j;
                ca.aliveOut = (uint32_t*)ln.alive[(j + 1) & 1].p;
                ca.keysOut = sorting ? (uint32_t*)ln.keys.p : nullptr;
                ca.countOut = counts + j + 1;
                ca.ticket = tickets + 2 * j + 1;
                ca.tileStatus = (unsigned long long*)ln.tileStatus.p;
                if (ln.epoch >= IDK_EPOCH_MASK) {   // 30-bit epoch wrapped: clear this lane's status words (ordered on its stream) and restart at 1
                    CK(cudaMemsetAsync(ln.tileStatus.p, 0, ln.tileStatus.bytes, ls));
                    ln.epoch = 0;
                }
                ca.epoch = ++ln.epoch;
                const size_t ec = ev.begin();
                k_compact<<<ctx->compactBlocks, IDK_BLOCK, 0, ls>>>(ca);
                ev.end(ec, 5);
                launches++;
            }
            ev.end(e0, 1, j);
        }

        // FinalDraw runs on the main (image) stream in issue order: samples accumulate in the order they were submitted
        // whichever lane finishes first, and presents / read-backs queued on the main stream see a consistent image.
        if (async) {
            CK(cudaEventRecord(ln.radianceReady, ls));
            CK(cudaStreamWaitEvent(ctx->stream, ln.radianceReady, 0));
        }
        e0 = ev.begin();
        const bool gatherNow = ctx->gatherWorld > 1 && s == st->SamplesPerPixel - 1;
        if (gatherNow) {
            // FinalDraw fused with the all-gather: Result pixels go straight to every rank's full image over NVLink
            const int b = (int)((ctx->gatherEpoch + 1) & 1u);
            GatherArgs g;
            memset(&g, 0, sizeof(g));
            for (int p = 0; p < ctx->gatherWorld; p++) { g.peerImage[p] = (float4*)ctx->peerImage[b][p]; g.peerFlags[p] = (uint32_t*)ctx->peerFlags[b][p]; }
            g.tileRows = (const int*)ctx->gatherRows.p;
            g.doneCounter = (uint32_t*)ctx->gatherScratch.p;
            g.world = ctx->gatherWorld; g.rank = ctx->gatherRank; g.width = ctx->width;
            g.epoch = ++ctx->gatherEpoch;
            CK(cudaMemsetAsync(ctx->gatherScratch.p, 0, 4, ctx->stream));
            k_accumulate_scatter<<<accBlocks, IDK_BLOCK, 0, ctx->stream>>>((const float4*)ln.radiance.p, (float4*)ctx->images[0].p, n,
                                                                           ctx->accumulatedSamples, st->Gpu.DoDebugBVHTraversal, g);
            if (aovs)   // AOV images stay local to the tile (only Result is gathered)
                k_accumulate_aov<<<accBlocks, IDK_BLOCK, 0, ctx->stream>>>((const float4*)ln.aovAlbedoFinal.p, (const float4*)ln.aovNormalFinal.p,
                                                                           (float4*)ctx->images[1].p, (float4*)ctx->images[2].p, n, ctx->accumulatedSamples);
            if (async) { CK(cudaEventRecord(ln.accDone, ctx->stream)); ln.accPending = true; }   // before the arrival wait: the lane may go on
            k_gather_wait<<<1, 32, 0, ctx->stream>>>((const uint32_t*)ctx->gatherFlags[b].p, ctx->gatherWorld, g.epoch, (uint32_t*)ctx->gatherScratch.p + 1,
                                                     (long long)(ctx->gatherTimeoutMs * (double)ctx->clockKHz));
            ctx->gatherCurrent = b;
            launches += aovs ? 3 : 2;
        } else {
            k_accumulate<<<accBlocks, IDK_BLOCK, 0, ctx->stream>>>((const float4*)ln.radiance.p, (const float4*)ln.aovAlbedoFinal.p,
                                                                   (const float4*)ln.aovNormalFinal.p, (float4*)ctx->images[0].p,
                                                                   (float4*)ctx->images[1].p, (float4*)ctx->images[2].p, n,
                                                                   ctx->accumulatedSamples, st->Gpu.DoDebugBVHTraversal, aovs ? 1 : 0);
            if (async) { CK(cudaEventRecord(ln.accDone, ctx->stream)); ln.accPending = true; }
            launches++;
        }
        ev.end(e0, 3);
        ev.end(e0, 6);
        if (stats) CK(cudaMemcpyAsync((uint32_t*)countLog.p + (size_t)s * (IDKPT_MAX_RAY_DEPTH + 1), counts,
                                      (IDKPT_MAX_RAY_DEPTH + 1) * sizeof(uint32_t), cudaMemcpyDeviceToDevice, ctx->stream));
        ctx->accumulatedSamples++;   // PathTracer.cs:269
    }
    ev.end(evTotal, 4);
    CK(cudaGetLastError());
    if (async) {
        ctx->asyncPending = true;
        return IDKPT_OK;
    }
    {
        int rc = check_device_errors(ctx, cudaStreamSynchronize(ctx->stream), "idkpt_compute");
        if (rc) return rc;
    }
    if (stats) {
        CK(cudaMemcpy(hostCounts.data(), countLog.p, hostCounts.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost));
        for (int s = 0; s < st->SamplesPerPixel; s++)
            for (int j = 0; j < st->RayDepth; j++) {
                const uint64_t c = hostCounts[(size_t)s * (IDKPT_MAX_RAY_DEPTH + 1) + j];
                stats->BounceRays[j] += c;
                stats->Rays += c;
            }
        if (wantStats) {
            TraceCounters tc;
            CK(cudaMemcpy(&tc, ctx->counters.p, sizeof(tc), cudaMemcpyDeviceToHost));
            stats->NodePairFetches = tc.steps;
            stats->TriangleTests = tc.tris;
            stats->InstanceVisits = tc.instances;
            stats->Hits = tc.hits;
#if IDK_PHASE_STATS
            fprintf(stderr, "[idkpt phase stats] SETUP rounds %llu lanes %llu | BOX rounds %llu lanes %llu | LEAF rounds %llu lanes %llu\n", tc.phaseRounds[0], tc.phaseLanes[0],
                    tc.phaseRounds[1], tc.phaseLanes[1], tc.phaseRounds[2], tc.phaseLanes[2]);
            fprintf(stderr, "[idkpt phase stats] during BOX rounds, idle lanes: waiting SETUP %llu, waiting LEAF %llu, exited %llu\n", tc.boxIdle[0], tc.boxIdle[1], tc.boxIdle[2]);
            { double mx = 0; for (int j = 0; j < st->RayDepth; j++) mx += tc.maxSteps[j]; fprintf(stderr, "[idkpt phase stats] sum over bounces of the longest ray: %.0f steps\n", mx); }
#endif
            for (int j = 0; j < IDKPT_MAX_RAY_DEPTH; j++) stats->BounceMaxSteps[j] = tc.maxSteps[j];
        }
        for (const EventPool::Span& sp : ev.spans) {
            float ms = 0.0f;
            cudaEventElapsedTime(&ms, ctx->events[sp.a], ctx->events[sp.b]);
            switch (sp.cat) {
                case 0: stats->TraverseMs += ms; if (sp.bounce >= 0) stats->BounceTraverseMs[sp.bounce] += ms; break;
                case 1: stats->ShadeMs += ms; if (sp.bounce >= 0) stats->BounceShadeMs[sp.bounce] += ms; break;
                case 2: stats->SortMs += ms; break;
                case 3: stats->OtherMs += ms; break;
                case 5: stats->CompactMs += ms; break;
                case 6: stats->AccumulateMs += ms; break;
                default: stats->TotalMs = ms; break;
            }
        }
        stats->KernelLaunches = launches;
        stats->TraverseLaunches = traverseLaunches;
    }
    return IDKPT_OK;
}

static int image_copy(IdkPtCtx* ctx, IdkPtImage which, void* host, uint64_t bytes, bool toHost) {
    if (!ctx || !host) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt image copy: null argument");
    if (which == IDKPT_IMAGE_DENOISED) {
        if (!toHost || !ctx->haveDenoised) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt image copy: no denoised image (call idkpt_denoise)");
        if (bytes < (uint64_t)ctx->width * ctx->height * 16) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt image copy: buffer smaller than width*height*16");
        CK(cudaSetDevice(ctx->device));
        CK(cudaMemcpyAsync(host, ctx->denoised.p, (size_t)ctx->width * ctx->height * 16, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        return IDKPT_OK;
    }
    if ((int)which < 0 || (int)which > 2) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt image copy: unknown image");
    if (bytes < (uint64_t)ctx->width * ctx->height * 16) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt image copy: buffer smaller than width*height*16");
    CK(cudaSetDevice(ctx->device));
    const size_t rowBytes = (size_t)ctx->width * 16;
    // owned rows are stored compactly; copy stripe by stripe into the full-image layout
    size_t i = 0;
    while (i < ctx->rows.size()) {
        size_t j = i;
        while (j + 1 < ctx->rows.size() && ctx->rows[j + 1] == ctx->rows[j] + 1) j++;
        char* h = (char*)host + (size_t)ctx->rows[i] * rowBytes;
        char* d = (char*)ctx->images[which].p + i * rowBytes;
        if (toHost) CK(cudaMemcpyAsync(h, d, (j - i + 1) * rowBytes, cudaMemcpyDeviceToHost, ctx->stream));
        else CK(cudaMemcpyAsync(d, h, (j - i + 1) * rowBytes, cudaMemcpyHostToDevice, ctx->stream));
        i = j + 1;
    }
    CK(cudaStreamSynchronize(ctx->stream));
    return IDKPT_OK;
}

IDKPT_API int idkpt_read_result(IdkPtCtx* ctx, IdkPtImage which, void* dst, uint64_t bytes) { return image_copy(ctx, which, dst, bytes, true); }
IDKPT_API int idkpt_write_result(IdkPtCtx* ctx, IdkPtImage which, const void* src, uint64_t bytes) { return image_copy(ctx, which, (void*)src, bytes, false); }

// Present without stalling the renderer: snapshot the image on the device (ordered after the Compute that produced it)
// and copy the snapshot to (ideally pinned) host memory on a second stream, so the transfer overlaps the next Compute.
IDKPT_API int idkpt_present_async(IdkPtCtx* ctx, IdkPtImage which, void* dstHost, uint64_t bytes) {
    if (!ctx || !dstHost) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_present_async: null argument");
    if ((int)which < 0 || (int)which > 3) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_present_async: unknown image");
    if (bytes < (uint64_t)ctx->width * ctx->height * 16) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_present_async: buffer smaller than width*height*16");
    CK(cudaSetDevice(ctx->device));
    if ((int)which == 3) {
        // IDKPT_IMAGE_GATHERED: the full multi-GPU frame. Snapshot it on the main stream first: with several frames in flight
        // a peer may start scattering frame k+2 into this buffer as soon as every rank has finished frame k+1, and that is
        // ordered after this snapshot (main stream: wait(k) -> snapshot(k) -> scatter(k+1)) but not after a slow D2H copy.
        if (ctx->gatherWorld < 2 || ctx->gatherCurrent < 0) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_present_async: no gathered frame yet");
        if (!ctx->copyStream) {
            CK(cudaStreamCreateWithFlags(&ctx->copyStream, cudaStreamNonBlocking));
            CK(cudaEventCreateWithFlags(&ctx->snapDone, cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&ctx->copyDone, cudaEventDisableTiming));
        }
        const size_t full = (size_t)ctx->width * ctx->height * 16;
        CK(ensure(ctx->presentSnap, full));
        if (ctx->copyPending) CK(cudaStreamWaitEvent(ctx->stream, ctx->copyDone, 0));   // previous transfer still reads the snapshot
        CK(cudaMemcpyAsync(ctx->presentSnap.p, ctx->gatherImage[ctx->gatherCurrent].p, full, cudaMemcpyDeviceToDevice, ctx->stream));
        CK(cudaEventRecord(ctx->snapDone, ctx->stream));
        CK(cudaStreamWaitEvent(ctx->copyStream, ctx->snapDone, 0));
        CK(cudaMemcpyAsync(dstHost, ctx->presentSnap.p, full, cudaMemcpyDeviceToHost, ctx->copyStream));
        CK(cudaEventRecord(ctx->copyDone, ctx->copyStream));
        ctx->copyPending = true;
        return IDKPT_OK;
    }
    if (!ctx->copyStream) {
        CK(cudaStreamCreateWithFlags(&ctx->copyStream, cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&ctx->snapDone, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&ctx->copyDone, cudaEventDisableTiming));
    }
    const size_t n = (size_t)ctx->nLocal * 16;
    CK(ensure(ctx->presentSnap, std::max<size_t>(n, 16)));
    if (ctx->copyPending) CK(cudaStreamWaitEvent(ctx->stream, ctx->copyDone, 0));   // previous transfer still reads the snapshot
    CK(cudaMemcpyAsync(ctx->presentSnap.p, ctx->images[which].p, n, cudaMemcpyDeviceToDevice, ctx->stream));
    CK(cudaEventRecord(ctx->snapDone, ctx->stream));
    CK(cudaStreamWaitEvent(ctx->copyStream, ctx->snapDone, 0));
    // The tile's rows are stored compactly, stripe after stripe; in the full-frame host layout its stripes are tileCount stripes
    // apart: ONE strided (2-D) copy moves all complete stripes, a second one the partial last stripe of the image if it is ours.
    // With a host frame shared by all ranks (idkpt_register_host_buffer on the same mapping in every process) each GPU
    // delivers its own 1/N of the frame over its own PCIe link -- no rank has to download the whole gathered image.
    const size_t rowBytes = (size_t)ctx->width * 16;
    if (!ctx->rows.empty()) {
        const size_t stripeBytes = (size_t)ctx->stripeH * rowBytes;
        const size_t fullStripes = ctx->rows.size() / (size_t)ctx->stripeH, tailRows = ctx->rows.size() % (size_t)ctx->stripeH;
        char* h0 = (char*)dstHost + (size_t)ctx->rows[0] * rowBytes;
        if (fullStripes)
            CK(cudaMemcpy2DAsync(h0, stripeBytes * (size_t)ctx->tileCount, ctx->presentSnap.p, stripeBytes, stripeBytes, fullStripes,
                                 cudaMemcpyDeviceToHost, ctx->copyStream));
        if (tailRows)
            CK(cudaMemcpyAsync((char*)dstHost + (size_t)ctx->rows[fullStripes * ctx->stripeH] * rowBytes, (char*)ctx->presentSnap.p + fullStripes * stripeBytes,
                               tailRows * rowBytes, cudaMemcpyDeviceToHost, ctx->copyStream));
    }
    CK(cudaEventRecord(ctx->copyDone, ctx->copyStream));
    ctx->copyPending = true;
    return IDKPT_OK;
}

IDKPT_API int idkpt_present_wait(IdkPtCtx* ctx) {
    if (!ctx) return IDKPT_ERR_INVALID_ARGUMENT;
    if (ctx->copyPending) {
        CK(cudaSetDevice(ctx->device));
        CK(cudaEventSynchronize(ctx->copyDone));
        ctx->copyPending = false;
    }
    return IDKPT_OK;
}

// Page-lock a host buffer the engine owns (e.g. the POSIX shared-memory frame all ranks present into) so that
// idkpt_present_async's copies are truly asynchronous. The C# host has no CUDA runtime of its own to call cudaHostRegister.
IDKPT_API int idkpt_register_host_buffer(IdkPtCtx* ctx, void* hostPtr, uint64_t bytes) {
    if (!ctx || !hostPtr || !bytes) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_register_host_buffer: null argument");
    CK(cudaSetDevice(ctx->device));
    CK(cudaHostRegister(hostPtr, bytes, cudaHostRegisterPortable));
    return IDKPT_OK;
}

IDKPT_API int idkpt_unregister_host_buffer(IdkPtCtx* ctx, void* hostPtr) {
    if (!ctx || !hostPtr) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_unregister_host_buffer: null argument");
    CK(cudaSetDevice(ctx->device));
    if (ctx->copyPending) { CK(cudaEventSynchronize(ctx->copyDone)); ctx->copyPending = false; }   // a transfer may still target it
    CK(cudaHostUnregister(hostPtr));
    return IDKPT_OK;
}

// ---- multi-GPU gather over peer memory -----------------------------------------------------------------------------
// Step 1 (every rank): allocate the exported buffers and return their CUDA IPC handles (4 x 64 bytes:
// image[0], image[1], flags[0], flags[1]). Step 2: exchange the handles (any transport) and import all ranks' handles.
// The buffers peers write into: full-size images + arrival flags (double-buffered), the per-stripe count tables of the
// global-slot exchange. Stand-alone cudaMalloc allocations (IPC export needs that).
// CUDA loads kernels lazily, and loading one may have to wait for the kernels that are running. Once contexts wait for each
// other ON THE DEVICE (arrival wait, slot exchange) a first launch from the host thread that still has to submit the peer's
// work would deadlock against them -- so everything a connected context can launch is loaded before the first wait exists.
__global__ void k_denoise_import(const float* __restrict__ rgb, float4* __restrict__ out, int count);
static int preload_kernels(IdkPtCtx* ctx) {
    cudaFuncAttributes fa;
#define IDK_PRELOAD(k) CK(cudaFuncGetAttributes(&fa, k))
    IDK_PRELOAD(k_init_sample); IDK_PRELOAD(k_prepare_triangles); IDK_PRELOAD(k_prepare_vertices); IDK_PRELOAD(k_prepare_surfaces);
    IDK_PRELOAD(k_raygen); IDK_PRELOAD(k_traverse<false>); IDK_PRELOAD(k_traverse<true>);
    IDK_PRELOAD((k_traverse2<false, false, false>)); IDK_PRELOAD((k_traverse2<true, false, false>)); IDK_PRELOAD((k_traverse2<false, true, false>));
    IDK_PRELOAD((k_traverse2<true, true, false>)); IDK_PRELOAD((k_traverse2<false, false, true>)); IDK_PRELOAD((k_traverse2<true, false, true>));
    IDK_PRELOAD(k_shade<false>); IDK_PRELOAD(k_shade<true>); IDK_PRELOAD(k_compact); IDK_PRELOAD(k_slot_exchange);
    IDK_PRELOAD(k_accumulate); IDK_PRELOAD(k_accumulate_aov); IDK_PRELOAD(k_accumulate_scatter); IDK_PRELOAD(k_gather_wait);
    IDK_PRELOAD(k_sort_histogram); IDK_PRELOAD(k_sort_scan); IDK_PRELOAD(k_sort_scatter);
    IDK_PRELOAD(k_trace_rays); IDK_PRELOAD(k_trace_rays_any); IDK_PRELOAD(k_shadows_ray_traced);
    IDK_PRELOAD(k_skin_vertices); IDK_PRELOAD(k_refit_prepare); IDK_PRELOAD(k_refit_climb); IDK_PRELOAD(k_tlas_build);
    IDK_PRELOAD(k_bloom_down); IDK_PRELOAD(k_bloom_up); IDK_PRELOAD(k_agx_matrices); IDK_PRELOAD(k_tonemap);
    IDK_PRELOAD(k_denoise_prepare); IDK_PRELOAD(k_denoise_atrous); IDK_PRELOAD(k_denoise_finish); IDK_PRELOAD(k_denoise_import);
    IDK_PRELOAD(k_bcn_decode);
#undef IDK_PRELOAD
    return IDKPT_OK;
}

static size_t slot_table_words(const IdkPtCtx* ctx) { return (size_t)IDK_MAX_LANES * 2 * (size_t)std::max(1, ctx->nStripes); }
static int gather_allocate(IdkPtCtx* ctx) {
    { int rc = preload_kernels(ctx); if (rc) return rc; }
    const size_t imgBytes = (size_t)ctx->width * ctx->height * 16;
    for (int b = 0; b < 2; b++) {
        CK(ensure(ctx->gatherImage[b], imgBytes));
        CK(ensure(ctx->gatherFlags[b], IDK_MAX_PEERS * sizeof(uint32_t)));
        CK(cudaMemsetAsync(ctx->gatherImage[b].p, 0, imgBytes, ctx->stream));
        CK(cudaMemsetAsync(ctx->gatherFlags[b].p, 0, IDK_MAX_PEERS * sizeof(uint32_t), ctx->stream));
    }
    // every lane is brought up NOW: once peers wait for each other on the device, a later allocation (an implicit device
    // synchronisation in the worst case) from the thread that still has to submit a peer's work could deadlock
    if (ctx->laneCount > 1)
        for (int i = 0; i < ctx->laneCount; i++)
            if (!ctx->lanes[i].allocated) { int rc = allocate_lane(ctx, ctx->lanes[i]); if (rc) return rc; }
    CK(ensure(ctx->slotTable, slot_table_words(ctx) * sizeof(unsigned long long)));
    CK(cudaMemsetAsync(ctx->slotTable.p, 0, ctx->slotTable.bytes, ctx->stream));   // epoch 0 = nothing published
    CK(ensure(ctx->gatherScratch, 16));
    CK(cudaMemsetAsync(ctx->gatherScratch.p, 0, 16, ctx->stream));
    CK(ensure(ctx->gatherRows, std::max<size_t>(ctx->rows.size(), 1) * sizeof(int)));
    if (!ctx->rows.empty()) CK(cudaMemcpyAsync(ctx->gatherRows.p, ctx->rows.data(), ctx->rows.size() * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return IDKPT_OK;
}

IDKPT_API int idkpt_gather_export(IdkPtCtx* ctx, void* handlesOut, uint64_t bytes) {
    if (!ctx || !handlesOut) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_gather_export: null argument");
    DRAIN_PENDING("idkpt_gather_export");
    if (bytes < IDKPT_GATHER_HANDLE_BYTES) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_gather_export: need IDKPT_GATHER_HANDLE_BYTES (320) bytes");
    CK(cudaSetDevice(ctx->device));
    { int rc = gather_allocate(ctx); if (rc) return rc; }
    cudaIpcMemHandle_t* out = (cudaIpcMemHandle_t*)handlesOut;
    for (int b = 0; b < 2; b++) {
        CK(cudaIpcGetMemHandle(&out[b], ctx->gatherImage[b].p));
        CK(cudaIpcGetMemHandle(&out[2 + b], ctx->gatherFlags[b].p));
    }
    CK(cudaIpcGetMemHandle(&out[4], ctx->slotTable.p));
    return IDKPT_OK;
}

// allHandles = world x 256 bytes in rank order (this rank's own entry is ignored and replaced by the local pointers).
IDKPT_API int idkpt_gather_import(IdkPtCtx* ctx, int32_t rank, int32_t world, const void* allHandles, uint64_t bytes) {
    if (!ctx || !allHandles) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_gather_import: null argument");
    DRAIN_PENDING("idkpt_gather_import");
    if (world < 2 || world > IDK_MAX_PEERS || rank < 0 || rank >= world) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_gather_import: invalid rank / world");
    if (world != ctx->tileCount || rank != ctx->tileIndex) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_gather_import: rank / world must equal TileIndex / TileCount");
    if (bytes < (uint64_t)world * IDKPT_GATHER_HANDLE_BYTES) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_gather_import: handle buffer too small");
    if (!ctx->gatherImage[0].p) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_gather_import: call idkpt_gather_export first");
    if (ctx->gatherWorld > 1) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_gather_import: peers are already connected (idkpt_resize disconnects them)");
    CK(cudaSetDevice(ctx->device));
    const cudaIpcMemHandle_t* hs = (const cudaIpcMemHandle_t*)allHandles;
    ctx->peerIsIpc = true;
    for (int p = 0; p < world; p++) {
        for (int b = 0; b < 2; b++) {
            if (p == rank) {
                ctx->peerImage[b][p] = ctx->gatherImage[b].p;
                ctx->peerFlags[b][p] = ctx->gatherFlags[b].p;
            } else {
                CK(cudaIpcOpenMemHandle(&ctx->peerImage[b][p], hs[5 * p + b], cudaIpcMemLazyEnablePeerAccess));
                CK(cudaIpcOpenMemHandle(&ctx->peerFlags[b][p], hs[5 * p + 2 + b], cudaIpcMemLazyEnablePeerAccess));
            }
        }
        if (p == rank) ctx->peerSlotTable[p] = ctx->slotTable.p;
        else CK(cudaIpcOpenMemHandle(&ctx->peerSlotTable[p], hs[5 * p + 4], cudaIpcMemLazyEnablePeerAccess));
        ctx->peerMapped[p] = true;
    }
    ctx->gatherWorld = world;
    ctx->gatherRank = rank;
    ctx->gatherEpoch = 0;
    ctx->gatherCurrent = -1;
    for (int i = 0; i < IDK_MAX_LANES; i++) ctx->lanes[i].slotEpoch = ctx->slotEpochStart;
    return IDKPT_OK;
}

// The same wiring for a host that drives all GPUs from ONE process (the reference engine is a single process): contexts
// [0, world) in tile order, each created with TileIndex = its position and TileCount = world. No IPC: the contexts hand each
// other their device pointers; peer access between different devices is enabled here.
IDKPT_API int idkpt_gather_connect(IdkPtCtx** ctxs, int32_t world) {
    if (!ctxs || world < 2 || world > IDK_MAX_PEERS) return fail(ctxs && world > 0 ? ctxs[0] : nullptr, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_gather_connect: invalid argument");
    for (int r = 0; r < world; r++) {
        IdkPtCtx* ctx = ctxs[r];
        if (!ctx) return fail(ctxs[0], IDKPT_ERR_INVALID_ARGUMENT, "idkpt_gather_connect: null context");
        if (ctx->tileCount != world || ctx->tileIndex != r) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_gather_connect: context r must have TileIndex r and TileCount world");
        if (ctx->width != ctxs[0]->width || ctx->height != ctxs[0]->height || ctx->stripeH != ctxs[0]->stripeH || ctx->laneCount != ctxs[0]->laneCount ||
            ctx->globalSlots != ctxs[0]->globalSlots)
            return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_gather_connect: contexts differ in size, stripe height, lanes or flags");
        DRAIN_PENDING("idkpt_gather_connect");
        if (ctx->gatherWorld > 1) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_gather_connect: peers are already connected");
        CK(cudaSetDevice(ctx->device));
        int rc = gather_allocate(ctx);
        if (rc) return rc;
    }
    for (int r = 0; r < world; r++) {
        IdkPtCtx* ctx = ctxs[r];
        CK(cudaSetDevice(ctx->device));
        for (int p = 0; p < world; p++) {
            if (ctxs[p]->device != ctx->device) {
                int can = 0;
                CK(cudaDeviceCanAccessPeer(&can, ctx->device, ctxs[p]->device));
                if (!can) return fail(ctx, IDKPT_ERR_UNSUPPORTED, "idkpt_gather_connect: no peer access between two of the devices");
                const cudaError_t e = cudaDeviceEnablePeerAccess(ctxs[p]->device, 0);
                if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
                else CK(e);
            }
            for (int b = 0; b < 2; b++) {
                ctx->peerImage[b][p] = ctxs[p]->gatherImage[b].p;
                ctx->peerFlags[b][p] = ctxs[p]->gatherFlags[b].p;
            }
            ctx->peerSlotTable[p] = ctxs[p]->slotTable.p;
            ctx->peerMapped[p] = true;
        }
        ctx->peerIsIpc = false;
        ctx->gatherWorld = world;
        ctx->gatherRank = r;
        ctx->gatherEpoch = 0;
        ctx->gatherCurrent = -1;
        for (int i = 0; i < IDK_MAX_LANES; i++) ctx->lanes[i].slotEpoch = ctx->slotEpochStart;
    }
    return IDKPT_OK;
}

// Full image (all ranks' tiles) of the last idkpt_compute; valid until the compute after next (double-buffered).
IDKPT_API int idkpt_gather_device_ptr(IdkPtCtx* ctx, void** devPtr, uint64_t* bytes) {
    if (!ctx || !devPtr) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_gather_device_ptr: null argument");
    DRAIN_PENDING("idkpt_gather_device_ptr");
    if (ctx->gatherWorld < 2 || ctx->gatherCurrent < 0) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_gather_device_ptr: no gathered frame yet");
    *devPtr = ctx->gatherImage[ctx->gatherCurrent].p;
    if (bytes) *bytes = (uint64_t)ctx->width * ctx->height * 16;
    return IDKPT_OK;
}

IDKPT_API int idkpt_result_device_ptr(IdkPtCtx* ctx, IdkPtImage which, void** devPtr, uint64_t* bytes) {
    if (!ctx || !devPtr || (int)which < 0 || (int)which > 2) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_result_device_ptr: invalid argument");
    DRAIN_PENDING("idkpt_result_device_ptr");
    *devPtr = ctx->images[which].p;
    if (bytes) *bytes = (uint64_t)ctx->nLocal * 16;
    return IDKPT_OK;
}

IDKPT_API int idkpt_tile_rows(IdkPtCtx* ctx, int32_t* rowCount, int32_t* rowsOut, int32_t capacity) {
    if (!ctx || !rowCount) return IDKPT_ERR_INVALID_ARGUMENT;
    *rowCount = (int32_t)ctx->rows.size();
    if (rowsOut) for (int i = 0; i < capacity && i < (int)ctx->rows.size(); i++) rowsOut[i] = ctx->rows[i];
    return IDKPT_OK;
}

IDKPT_API int idkpt_read_wavefront_rays(IdkPtCtx* ctx, GpuWavefrontRay* dst, uint64_t count) {
    if (!ctx) return IDKPT_ERR_INVALID_ARGUMENT;
    DRAIN_PENDING("idkpt_read_wavefront_rays");
    if (!dst) {   // dst == NULL arms the export for subsequent idkpt_compute calls (debug / parity feature)
        ctx->exportEnabled = count != 0;
        return IDKPT_OK;
    }
    if (!ctx->exportEnabled) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_read_wavefront_rays: arm the export first (dst = NULL, count = 1) and call idkpt_compute");
    if (count < (uint64_t)ctx->width * ctx->height) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_read_wavefront_rays: buffer smaller than width*height");
    CK(cudaSetDevice(ctx->device));
    std::vector<PathState> tmp(ctx->nLocal);
    CK(cudaMemcpyAsync(tmp.data(), ctx->lanes[0].state.p, (size_t)ctx->nLocal * sizeof(PathState), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    for (size_t i = 0; i < ctx->rows.size(); i++) {
        for (int x = 0; x < ctx->width; x++) {
            const PathState& s = tmp[i * (size_t)ctx->width + x];
            GpuWavefrontRay& w = dst[(size_t)ctx->rows[i] * ctx->width + x];
            w.Origin[0] = s.ox; w.Origin[1] = s.oy; w.Origin[2] = s.oz; w.PreviousIOROrTraverseCost = s.prevIor;
            w.Throughput[0] = s.tx; w.Throughput[1] = s.ty; w.Throughput[2] = s.tz; w.PackedDirectionX = s.pdx;
            w.Radiance[0] = s.rx; w.Radiance[1] = s.ry; w.Radiance[2] = s.rz; w.PackedDirectionY = s.pdy;
        }
    }
    return IDKPT_OK;
}

// ---- present chain (SURVEY.md 8f.3) ----------------------------------------------------------------------------------------

static inline int ilogb_int(int v) { int r = 0; while (v > 1) { v >>= 1; r++; } return r; }

IDKPT_API int idkpt_post_process(IdkPtCtx* ctx, const IdkPtPostSettings* s, IdkPtImage source, uint8_t* rgba8Out, float* kernelMs) {
    if (!ctx || !s) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_post_process: null argument");
    if (kernelMs) *kernelMs = 0.0f;
    const int w = ctx->width, h = ctx->height;
    const float4* src = nullptr;
    if (source == IDKPT_IMAGE_GATHERED) {
        if (ctx->gatherWorld < 2 || ctx->gatherCurrent < 0) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_post_process: no gathered frame yet");
        src = (const float4*)ctx->gatherImage[ctx->gatherCurrent].p;
    } else if (source == IDKPT_IMAGE_DENOISED) {
        if (!ctx->haveDenoised) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_post_process: no denoised image (call idkpt_denoise)");
        src = (const float4*)ctx->denoised.p;
    } else if ((int)source >= 0 && (int)source <= 2) {
        if (ctx->tileCount != 1) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_post_process: a tiled context holds only its own rows; use IDKPT_IMAGE_GATHERED");
        src = (const float4*)ctx->images[source].p;
    } else return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_post_process: unknown image");
    if (s->IsBloom && (w < 2 || h < 2)) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_post_process: bloom needs an image of at least 2x2");
    if (s->IsBloom && (s->BloomMinusLods < 0 || s->BloomMinusLods > 30)) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_post_process: BloomMinusLods out of range");
    CK(cudaSetDevice(ctx->device));
    CK(ensure(ctx->ldr, (size_t)w * h * 4));
    CK(ensure(ctx->postConsts, sizeof(PostTonemapConsts)));
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    cudaEventRecord(e0, ctx->stream);
    const dim3 blk(256);
    auto grid = [](int gw, int gh) { return dim3((unsigned)((gw + 31) / 32), (unsigned)((gh + 7) / 8)); };
    PostImage bloomResult = {nullptr, nullptr, 0, 0};
    if (s->IsBloom) {
        // Bloom.SetSize (Bloom.cs:132-150): half resolution, levels = max(MaxMipmapLevel - MinusLods, 2); the upsample chain has one level less
        const int w2 = w / 2, h2 = h / 2;
        const int levels = std::max(ilogb_int(std::max(w2, h2)) + 1 - s->BloomMinusLods, 2);
        std::vector<size_t> off(levels + 1, 0);
        std::vector<int> lw(levels), lh(levels);
        for (int l = 0; l < levels; l++) {
            lw[l] = std::max(1, w2 / (1 << std::min(l, 30))); lh[l] = std::max(1, h2 / (1 << std::min(l, 30)));
            off[l + 1] = off[l] + (size_t)lw[l] * lh[l];
        }
        cudaError_t ce = ensure(ctx->bloomDown, off[levels] * 8);
        if (ce == cudaSuccess) ce = ensure(ctx->bloomUp, off[levels - 1] * 8);
        if (ce != cudaSuccess) { cudaEventDestroy(e0); cudaEventDestroy(e1); return fail(ctx, IDKPT_ERR_OUT_OF_MEMORY, "idkpt_post_process: bloom allocation failed"); }
        uint2* down = (uint2*)ctx->bloomDown.p;
        uint2* up = (uint2*)ctx->bloomUp.p;
        for (int l = 0; l < levels; l++) {
            BloomDownArgs a;
            a.src = l == 0 ? PostImage{src, nullptr, w, h} : PostImage{nullptr, down + off[l - 1], lw[l - 1], lh[l - 1]};
            a.dst = down + off[l]; a.dw = lw[l]; a.dh = lh[l];
            a.prefilter = l == 0; a.maxColor = s->BloomMaxColor; a.threshold = s->BloomThreshold;
            k_bloom_down<<<grid(a.dw, a.dh), blk, 0, ctx->stream>>>(a);
        }
        for (int l = levels - 2; l >= 0; l--) {
            BloomUpArgs a;
            a.up = l == levels - 2 ? PostImage{nullptr, down + off[l + 1], lw[l + 1], lh[l + 1]} : PostImage{nullptr, up + off[l + 1], lw[l + 1], lh[l + 1]};
            a.down = PostImage{nullptr, down + off[l + 1], lw[l + 1], lh[l + 1]};
            a.dst = up + off[l]; a.dw = lw[l]; a.dh = lh[l];
            k_bloom_up<<<grid(a.dw, a.dh), blk, 0, ctx->stream>>>(a);
        }
        bloomResult = PostImage{nullptr, up, lw[0], lh[0]};
    }
    k_agx_matrices<<<1, 1, 0, ctx->stream>>>(s->Exposure, s->Compression, (PostTonemapConsts*)ctx->postConsts.p);
    TonemapArgs t;
    t.src0 = PostImage{src, nullptr, w, h};
    t.src1 = bloomResult;
    t.dst = (uchar4*)ctx->ldr.p; t.w = w; t.h = h;
    t.saturation = s->Saturation; t.linear = s->Linear; t.peak = s->Peak; t.doTonemap = s->DoTonemapAndSrgbTransform ? 1 : 0;
    t.consts = (const PostTonemapConsts*)ctx->postConsts.p;
    k_tonemap<<<grid(w, h), blk, 0, ctx->stream>>>(t);
    cudaEventRecord(e1, ctx->stream);
    if (rgba8Out) cudaMemcpyAsync(rgba8Out, ctx->ldr.p, (size_t)w * h * 4, cudaMemcpyDeviceToHost, ctx->stream);
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e == cudaSuccess && kernelMs) cudaEventElapsedTime(kernelMs, e0, e1);
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    if (e != cudaSuccess) { ctx->lastError = std::string("idkpt_post_process: ") + cudaGetErrorString(e); return IDKPT_ERR_CUDA; }
    return IDKPT_OK;
}

IDKPT_API int idkpt_ldr_device_ptr(IdkPtCtx* ctx, void** devPtr, uint64_t* bytes) {
    if (!ctx || !devPtr) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_ldr_device_ptr: null argument");
    DRAIN_PENDING("idkpt_ldr_device_ptr");
    if (!ctx->ldr.p) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_ldr_device_ptr: call idkpt_post_process first");
    *devPtr = ctx->ldr.p;
    if (bytes) *bytes = (uint64_t)ctx->width * ctx->height * 4;
    return IDKPT_OK;
}

// ---- denoise hand-off (SURVEY.md 8f.3) ---------------------------------------------------------------------------------------
static int denoise_alloc(IdkPtCtx* ctx) {
    const size_t n = (size_t)ctx->width * ctx->height;
    for (int i = 0; i < 4; i++) CK(ensure(ctx->oidn[i], n * 12));
    for (int i = 0; i < 2; i++) CK(ensure(ctx->denoiseWork[i], n * 16));
    CK(ensure(ctx->denoised, n * 16));
    return IDKPT_OK;
}

IDKPT_API int idkpt_denoise(IdkPtCtx* ctx, const IdkPtDenoiseSettings* s, float* kernelMs) {
    if (!ctx || !s) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_denoise: null argument");
    if (kernelMs) *kernelMs = 0.0f;
    if (ctx->tileCount != 1) return fail(ctx, IDKPT_ERR_UNSUPPORTED, "idkpt_denoise: the AOV images of a tiled context hold only its own rows");
    if (s->Iterations < 0 || s->Iterations > 12 || !(s->SigmaColor > 0.0f) || !(s->SigmaNormal > 0.0f) || !(s->SigmaAlbedo > 0.0f))
        return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_denoise: Iterations must be 0..12 and the sigmas positive");
    DRAIN_PENDING("idkpt_denoise");
    CK(cudaSetDevice(ctx->device));
    int rc = denoise_alloc(ctx);
    if (rc) return rc;
    const int w = ctx->width, h = ctx->height, n = w * h;
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    cudaEventRecord(e0, ctx->stream);
    DenoisePrepareArgs pa;
    pa.result = (const float4*)ctx->images[0].p; pa.albedo = (const float4*)ctx->images[1].p; pa.normal = (const float4*)ctx->images[2].p;
    pa.oidnBeauty = (float*)ctx->oidn[0].p; pa.oidnAlbedo = (float*)ctx->oidn[1].p; pa.oidnNormal = (float*)ctx->oidn[2].p;
    pa.work = (float4*)ctx->denoiseWork[0].p; pa.count = n; pa.demodulate = s->Demodulate ? 1 : 0;
    k_denoise_prepare<<<(n + 255) / 256, 256, 0, ctx->stream>>>(pa);
    int cur = 0;
    for (int it = 0; it < s->Iterations; it++) {
        const int step = 1 << it;
        const float sc = s->SigmaColor / (float)step;
        DenoiseAtrousArgs a;
        a.in = (const float4*)ctx->denoiseWork[cur].p; a.out = (float4*)ctx->denoiseWork[cur ^ 1].p;
        a.albedo = pa.albedo; a.normal = pa.normal; a.w = w; a.h = h; a.step = step;
        a.invSigmaColor2 = 1.0f / (sc * sc); a.invSigmaNormal2 = 1.0f / (s->SigmaNormal * s->SigmaNormal);
        a.invSigmaAlbedo2 = 1.0f / (s->SigmaAlbedo * s->SigmaAlbedo); a.invStep2 = 1.0f / ((float)step * (float)step);
        k_denoise_atrous<<<dim3((unsigned)((w + 31) / 32), (unsigned)((h + 7) / 8)), 256, 0, ctx->stream>>>(a);
        cur ^= 1;
    }
    if (s->Iterations > 0) {
        DenoiseFinishArgs fa;
        fa.filtered = (const float4*)ctx->denoiseWork[cur].p; fa.albedo = pa.albedo; fa.denoised = (float4*)ctx->denoised.p;
        fa.oidnOutput = (float*)ctx->oidn[3].p; fa.count = n; fa.demodulate = pa.demodulate;
        k_denoise_finish<<<(n + 255) / 256, 256, 0, ctx->stream>>>(fa);
    }
    cudaEventRecord(e1, ctx->stream);
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e == cudaSuccess && kernelMs) cudaEventElapsedTime(kernelMs, e0, e1);
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    if (e != cudaSuccess) { ctx->lastError = std::string("idkpt_denoise: ") + cudaGetErrorString(e); return IDKPT_ERR_CUDA; }
    if (s->Iterations > 0) ctx->haveDenoised = true;
    return IDKPT_OK;
}

IDKPT_API int idkpt_denoise_device_ptrs(IdkPtCtx* ctx, void** beauty, void** albedo, void** normal, void** output, uint64_t* bytesEach) {
    if (!ctx) return IDKPT_ERR_INVALID_ARGUMENT;
    DRAIN_PENDING("idkpt_denoise_device_ptrs");
    CK(cudaSetDevice(ctx->device));
    int rc = denoise_alloc(ctx);
    if (rc) return rc;
    if (beauty) *beauty = ctx->oidn[0].p;
    if (albedo) *albedo = ctx->oidn[1].p;
    if (normal) *normal = ctx->oidn[2].p;
    if (output) *output = ctx->oidn[3].p;
    if (bytesEach) *bytesEach = (uint64_t)ctx->width * ctx->height * 12;
    return IDKPT_OK;
}

// The OIDN output buffer (written by the host's OIDN CUDA device) becomes the denoised image.
__global__ void __launch_bounds__(256) k_denoise_import(const float* __restrict__ rgb, float4* __restrict__ out, int count) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) out[i] = make_float4(rgb[3 * (size_t)i], rgb[3 * (size_t)i + 1], rgb[3 * (size_t)i + 2], 1.0f);
}

IDKPT_API int idkpt_denoise_import_output(IdkPtCtx* ctx) {
    if (!ctx) return IDKPT_ERR_INVALID_ARGUMENT;
    DRAIN_PENDING("idkpt_denoise_import_output");
    if (!ctx->oidn[3].p || !ctx->denoised.p) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_denoise_import_output: call idkpt_denoise_device_ptrs / idkpt_denoise first");
    CK(cudaSetDevice(ctx->device));
    const int n = ctx->width * ctx->height;
    k_denoise_import<<<(n + 255) / 256, 256, 0, ctx->stream>>>((const float*)ctx->oidn[3].p, (float4*)ctx->denoised.p, n);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->haveDenoised = true;
    return IDKPT_OK;
}

// ---- dynamic geometry (SURVEY.md 8f.2) -----------------------------------------------------------------------------------

IDKPT_API int idkpt_set_skinning_data(IdkPtCtx* ctx, const GpuUnskinnedVertex* vertices, uint64_t count) {
    if (!ctx || (!vertices && count)) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_set_skinning_data: null argument");
    DRAIN_PENDING("idkpt_set_skinning_data");
    CK(cudaSetDevice(ctx->device));
    int rc;
    if ((rc = upload(ctx, ctx->unskinned, vertices, count * sizeof(GpuUnskinnedVertex)))) return rc;
    ctx->unskinnedMaxJoint.resize(count);
    for (uint64_t i = 0; i < count; i++) {
        const uint32_t* j = vertices[i].JointIndices;
        ctx->unskinnedMaxJoint[i] = std::max(std::max(j[0], j[1]), std::max(j[2], j[3]));
    }
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->unskinnedCount = count;
    return IDKPT_OK;
}

IDKPT_API int idkpt_skin_vertices(IdkPtCtx* ctx, const float* jointMatrices, uint64_t jointCount, const IdkPtSkinningCmd* cmds, uint32_t cmdCount, float* kernelMs) {
    if (!ctx || (!jointMatrices && jointCount) || (!cmds && cmdCount)) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_skin_vertices: null argument");
    DRAIN_PENDING("idkpt_skin_vertices");
    if (!ctx->haveScene) return fail(ctx, IDKPT_ERR_NO_SCENE, "idkpt_skin_vertices: no scene");
    if (kernelMs) *kernelMs = 0.0f;
    const uint64_t vtxLimit = std::min(ctx->counts.VertexPositionCount, ctx->counts.VertexCount);
    for (uint32_t c = 0; c < cmdCount; c++) {
        const IdkPtSkinningCmd& k = cmds[c];
        if ((uint64_t)k.InputVertexOffset + k.VertexCount > ctx->unskinnedCount) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_skin_vertices: input range outside the unskinned vertices (idkpt_set_skinning_data)");
        if ((uint64_t)k.OutputVertexOffset + k.VertexCount > vtxLimit) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_skin_vertices: output range outside the vertex arrays");
        uint32_t maxJoint = 0;
        for (uint64_t i = k.InputVertexOffset; i < (uint64_t)k.InputVertexOffset + k.VertexCount; i++) maxJoint = std::max(maxJoint, ctx->unskinnedMaxJoint[i]);
        if (k.VertexCount && (uint64_t)k.JointMatricesOffset + maxJoint >= jointCount) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_skin_vertices: a joint index points past the joint matrices");
    }
    CK(cudaSetDevice(ctx->device));
    int rc;
    if ((rc = upload(ctx, ctx->joints, jointMatrices, jointCount * 48))) return rc;   // jointMatricesBuffer.UploadElements (ModelManager.cs:277)
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    cudaEventRecord(e0, ctx->stream);
    for (uint32_t c = 0; c < cmdCount; c++) {
        if (!cmds[c].VertexCount) continue;
        SkinArgs a;
        a.unskinned = (const uint32_t*)ctx->unskinned.p; a.joints = (const float4*)ctx->joints.p;
        a.positions = (float*)ctx->positions.p; a.vertices = (uint4*)ctx->vertices.p; a.vtxFrame = (float4*)ctx->vtxFrame.p;
        a.inOffset = cmds[c].InputVertexOffset; a.outOffset = cmds[c].OutputVertexOffset; a.jointOffset = cmds[c].JointMatricesOffset; a.count = cmds[c].VertexCount;
        k_skin_vertices<<<(a.count + 255) / 256, 256, 0, ctx->stream>>>(a);
    }
    cudaEventRecord(e1, ctx->stream);
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e == cudaSuccess && kernelMs) cudaEventElapsedTime(kernelMs, e0, e1);
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    if (e != cudaSuccess) { ctx->lastError = std::string("idkpt_skin_vertices: ") + cudaGetErrorString(e); return IDKPT_ERR_CUDA; }
    ctx->accumulatedSamples = 0;
    return IDKPT_OK;
}

IDKPT_API int idkpt_blas_refit(IdkPtCtx* ctx, uint32_t first, uint32_t count, float* kernelMs) {
    if (!ctx) return IDKPT_ERR_INVALID_ARGUMENT;
    DRAIN_PENDING("idkpt_blas_refit");
    if (!ctx->haveScene) return fail(ctx, IDKPT_ERR_NO_SCENE, "idkpt_blas_refit: no scene");
    if ((uint64_t)first + count > ctx->hostDescs.size()) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_blas_refit: BLAS range outside BlasDescs");
    if (ctx->treeletNodes) return fail(ctx, IDKPT_ERR_UNSUPPORTED, "idkpt_blas_refit: not available with the treelet node layout (IDKPT_TREELET_PAIRS)");
    if (kernelMs) *kernelMs = 0.0f;
    CK(cudaSetDevice(ctx->device));
    int maxNodes = 0;
    for (uint32_t b = first; b < first + count; b++) maxNodes = std::max(maxNodes, ctx->hostDescs[b].NodeCount);
    CK(ensure(ctx->refitParents, std::max<size_t>((size_t)maxNodes, 4) * 4));   // blasRefitLockBuffer sizing, BVH.cs:451
    CK(ensure(ctx->refitLocks, std::max<size_t>((size_t)maxNodes, 4) * 4));
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    cudaEventRecord(e0, ctx->stream);
    for (uint32_t b = first; b < first + count; b++) {
        const GpuBlasDesc& d = ctx->hostDescs[b];
        RefitArgs a;
        a.nodes = (float4*)ctx->nodes.p + 2 * (size_t)d.NodeOffset;
        a.blasTris = (const int4*)ctx->blasTris.p; a.positions = (const float*)ctx->positions.p;
        a.triRec = (float4*)((char*)ctx->nodes.p + ctx->nodeBytes);
        a.parents = (int32_t*)ctx->refitParents.p; a.locks = (uint32_t*)ctx->refitLocks.p;
        a.nodeCount = (uint32_t)d.NodeCount; a.triOffset = (uint32_t)d.TriangleOffset; a.triCount = (uint32_t)d.TriangleCount;
        k_refit_prepare<<<(a.nodeCount + 255) / 256, 256, 0, ctx->stream>>>(a);
        k_refit_climb<<<(a.nodeCount + 255) / 256, 256, 0, ctx->stream>>>(a);
    }
    cudaEventRecord(e1, ctx->stream);
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e == cudaSuccess && kernelMs) cudaEventElapsedTime(kernelMs, e0, e1);
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    if (e != cudaSuccess) { ctx->lastError = std::string("idkpt_blas_refit: ") + cudaGetErrorString(e); return IDKPT_ERR_CUDA; }
    ctx->accumulatedSamples = 0;
    return IDKPT_OK;
}

// BVH.TlasBuild on the device (BVH.cs:278-298, TLAS.cs:28-141): see k_tlas_build.
IDKPT_API int idkpt_tlas_build(IdkPtCtx* ctx, int32_t searchRadius, float* kernelMs) {
    if (!ctx) return IDKPT_ERR_INVALID_ARGUMENT;
    DRAIN_PENDING("idkpt_tlas_build");
    if (kernelMs) *kernelMs = 0.0f;
    if (!ctx->haveScene) return fail(ctx, IDKPT_ERR_NO_SCENE, "idkpt_tlas_build: no scene");
    if (!ctx->counts.UseTlas) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_tlas_build: the scene was set without UseTlas (no TLAS node array to fill)");
    if (searchRadius < 1 || searchRadius > 1024) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_tlas_build: search radius out of range (TLAS.BuildSettings.SearchRadius, default 15)");
    const uint64_t n = ctx->counts.BlasInstanceCount;
    if (n > 16384) return fail(ctx, IDKPT_ERR_UNSUPPORTED, "idkpt_tlas_build: more than 16384 instances (single-CTA build); build on the host and idkpt_update_range");
    if (ctx->treeletNodes) return fail(ctx, IDKPT_ERR_UNSUPPORTED, "idkpt_tlas_build: not available with the treelet node layout (IDKPT_TREELET_PAIRS)");
    CK(cudaSetDevice(ctx->device));
    const size_t nodeCount = 2 * n - 1;
    const size_t tempOff = 0, leavesOff = nodeCount * 32, keysOff = leavesOff + n * 32, prefOff = keysOff + n * 4, needOff = prefOff + n * 4;
    CK(ensure(ctx->tlasScratch, needOff + nodeCount * 4 + 64));
    TlasBuildArgs a;
    a.blasNodes = (const float4*)ctx->nodes.p; a.descs = (const GpuBlasDesc*)ctx->descs.p; a.instances = (const GpuBlasInstance*)ctx->instances.p;
    a.xforms = (const float4*)ctx->xforms.p; a.nodes = (float4*)ctx->tlas.p;
    a.temp = (float4*)((char*)ctx->tlasScratch.p + tempOff); a.leaves = (float4*)((char*)ctx->tlasScratch.p + leavesOff);
    a.keys = (uint32_t*)((char*)ctx->tlasScratch.p + keysOff); a.pref = (int*)((char*)ctx->tlasScratch.p + prefOff);
    a.need = (int*)((char*)ctx->tlasScratch.p + needOff);
    a.n = (int)n; a.searchRadius = searchRadius;
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    cudaEventRecord(e0, ctx->stream);
    k_tlas_build<<<1, 1024, 0, ctx->stream>>>(a);
    cudaEventRecord(e1, ctx->stream);
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e == cudaSuccess && kernelMs) cudaEventElapsedTime(kernelMs, e0, e1);
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    if (e != cudaSuccess) { ctx->lastError = std::string("idkpt_tlas_build: ") + cudaGetErrorString(e); return IDKPT_ERR_CUDA; }
    ctx->accumulatedSamples = 0;
    int need = 0;
    CK(cudaMemcpy(&need, a.need, 4, cudaMemcpyDeviceToHost));
    if (need > IDK_TLAS_STACK_SIZE) {     // the walk's stack is fixed (BVHIntersect.glsl:4): refuse to trace through a TLAS it cannot hold
        ctx->haveScene = false;
        return fail(ctx, IDKPT_ERR_UNSUPPORTED, "idkpt_tlas_build: the built TLAS is deeper than the 24-entry traversal stack of the TLAS walk (scene invalidated; set it again)");
    }
    return IDKPT_OK;
}

IDKPT_API int idkpt_read_range(IdkPtCtx* ctx, IdkPtArrayId which, uint64_t first, uint64_t count, void* out) {
    if (!ctx || (!out && count)) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_read_range: null argument");
    if (!ctx->haveScene) return fail(ctx, IDKPT_ERR_NO_SCENE, "idkpt_read_range: no scene");
    const DevBuf* b = nullptr;
    size_t elem = 0;
    uint64_t limit = 0;
    switch (which) {
        case IDKPT_ARRAY_BLAS_NODES: b = &ctx->nodes; elem = sizeof(GpuBlasNode); limit = ctx->counts.BlasNodeCount; break;
        case IDKPT_ARRAY_VERTEX_POSITIONS: b = &ctx->positions; elem = sizeof(PackedVec3); limit = ctx->counts.VertexPositionCount; break;
        case IDKPT_ARRAY_VERTICES: b = &ctx->vertices; elem = sizeof(GpuVertex); limit = ctx->counts.VertexCount; break;
        case IDKPT_ARRAY_TLAS_NODES: b = &ctx->tlas; elem = sizeof(GpuTlasNode); limit = ctx->counts.UseTlas ? ctx->counts.TlasNodeCount : 0; break;
        default: return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_read_range: array id not readable");
    }
    if (which == IDKPT_ARRAY_BLAS_NODES && ctx->treeletNodes) return fail(ctx, IDKPT_ERR_UNSUPPORTED, "idkpt_read_range: BLAS nodes are re-laid out (IDKPT_TREELET_PAIRS)");
    if (first > limit || count > limit - first) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_read_range: range outside the array");
    CK(cudaSetDevice(ctx->device));
    if (count) CK(cudaMemcpyAsync(out, (const char*)b->p + first * elem, count * elem, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return IDKPT_OK;
}

static int trace_rays_impl(IdkPtCtx* ctx, const IdkPtRay* rays, uint64_t count, int32_t traceLights, IdkPtHit* hitsOut, float* kernelMs, bool anyHit);

IDKPT_API int idkpt_trace_rays(IdkPtCtx* ctx, const IdkPtRay* rays, uint64_t count, int32_t traceLights, IdkPtHit* hitsOut, float* kernelMs) {
    return trace_rays_impl(ctx, rays, count, traceLights, hitsOut, kernelMs, false);
}

IDKPT_API int idkpt_trace_rays_any(IdkPtCtx* ctx, const IdkPtRay* rays, uint64_t count, int32_t traceLights, IdkPtHit* hitsOut, float* kernelMs) {
    return trace_rays_impl(ctx, rays, count, traceLights, hitsOut, kernelMs, true);
}

IDKPT_API int idkpt_shadows_ray_traced(IdkPtCtx* ctx, const GpuPerFrameData* frame, const float* depth, const float* normalRG, int32_t width,
                                       int32_t height, int32_t lightIndex, int32_t samples, uint32_t noiseIndex, const float* taaJitter,
                                       float* visibilityOut, float* kernelMs) {
    if (!ctx || !frame || !depth || !normalRG || !visibilityOut) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_shadows_ray_traced: null argument");
    if (!ctx->haveScene) return fail(ctx, IDKPT_ERR_NO_SCENE, "idkpt_shadows_ray_traced: no scene");
    if (width < 1 || height < 1 || width > 16384 || height > 16384 || samples < 1 || samples > 1024) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_shadows_ray_traced: invalid size / sample count");
    if (lightIndex < 0 || (uint64_t)lightIndex >= ctx->counts.LightCount) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_shadows_ray_traced: light index out of range");
    CK(cudaSetDevice(ctx->device));
    if (kernelMs) *kernelMs = 0.0f;
    const size_t n = (size_t)width * height;
    DevBuf &dDepth = ctx->scratch[0], &dN = ctx->scratch[1], &dVis = ctx->scratch[2];
    int rc = IDKPT_OK;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    do {
        if (ensure(dDepth, n * 4) != cudaSuccess || ensure(dN, n * 8) != cudaSuccess || ensure(dVis, n * 4) != cudaSuccess) { rc = fail(ctx, IDKPT_ERR_OUT_OF_MEMORY, "idkpt_shadows_ray_traced: device allocation failed"); break; }
        cudaMemcpyAsync(dDepth.p, depth, n * 4, cudaMemcpyHostToDevice, ctx->stream);
        cudaMemcpyAsync(dN.p, normalRG, n * 8, cudaMemcpyHostToDevice, ctx->stream);
        cudaMemcpyAsync(dVis.p, visibilityOut, n * 4, cudaMemcpyHostToDevice, ctx->stream);   // pixels with depth == 1 keep the caller's value
        ShadowArgs a;
        a.sc = ctx->sc;
        memcpy(a.invProjView, frame->InvProjView, sizeof(a.invProjView));
        a.jitter[0] = taaJitter ? taaJitter[0] : 0.0f; a.jitter[1] = taaJitter ? taaJitter[1] : 0.0f;
        a.depth = (const float*)dDepth.p; a.normalRG = (const float2*)dN.p; a.visibility = (float*)dVis.p;
        a.width = width; a.height = height; a.lightIndex = lightIndex; a.samples = samples; a.noiseIndex = noiseIndex;
        cudaEventCreate(&e0); cudaEventCreate(&e1);
        cudaEventRecord(e0, ctx->stream);
        k_shadows_ray_traced<<<ctx->traceRaysBlocks, IDK_BLOCK, ctx->stackBytes, ctx->stream>>>(a);
        cudaEventRecord(e1, ctx->stream);
        cudaMemcpyAsync(visibilityOut, dVis.p, n * 4, cudaMemcpyDeviceToHost, ctx->stream);
        cudaError_t e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) { ctx->lastError = std::string("idkpt_shadows_ray_traced: ") + cudaGetErrorString(e); rc = IDKPT_ERR_CUDA; break; }
        if (kernelMs) cudaEventElapsedTime(kernelMs, e0, e1);
    } while (0);
    if (e0) cudaEventDestroy(e0);
    if (e1) cudaEventDestroy(e1);
    return rc;
}

static int trace_rays_impl(IdkPtCtx* ctx, const IdkPtRay* rays, uint64_t count, int32_t traceLights, IdkPtHit* hitsOut, float* kernelMs, bool anyHit) {
    if (!ctx || (!rays && count) || (!hitsOut && count)) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_trace_rays: null argument");
    if (!ctx->haveScene) return fail(ctx, IDKPT_ERR_NO_SCENE, "idkpt_trace_rays: no scene");
    if (count >= (1ull << 31)) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_trace_rays: too many rays");
    if (kernelMs) *kernelMs = 0.0f;
    if (count == 0) return IDKPT_OK;
    CK(cudaSetDevice(ctx->device));
    DevBuf &dr = ctx->scratch[0], &dh = ctx->scratch[1], &dt = ctx->scratch[2];
    int rc = IDKPT_OK;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    do {
        if (ensure(dr, count * 32) != cudaSuccess || ensure(dh, count * 32) != cudaSuccess || ensure(dt, 16) != cudaSuccess) { rc = fail(ctx, IDKPT_ERR_OUT_OF_MEMORY, "idkpt_trace_rays: device allocation failed"); break; }
        cudaMemcpyAsync(dr.p, rays, count * 32, cudaMemcpyHostToDevice, ctx->stream);
        cudaMemsetAsync(dt.p, 0, 16, ctx->stream);
        TraceRaysArgs a;
        a.sc = ctx->sc;
        a.rays = (const float4*)dr.p;
        a.hits = (uint4*)dh.p;
        a.count = (uint32_t)count;
        a.ticket = (uint32_t*)dt.p;
        a.traceLights = traceLights;
        cudaEventCreate(&e0);
        cudaEventCreate(&e1);
        cudaEventRecord(e0, ctx->stream);
        if (anyHit) k_trace_rays_any<<<ctx->traceRaysBlocks, IDK_BLOCK, ctx->stackBytes, ctx->stream>>>(a);
        else k_trace_rays<<<ctx->traceRaysBlocks, IDK_BLOCK, ctx->stackBytes, ctx->stream>>>(a);
        cudaEventRecord(e1, ctx->stream);
        cudaMemcpyAsync(hitsOut, dh.p, count * 32, cudaMemcpyDeviceToHost, ctx->stream);
        cudaError_t e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) { ctx->lastError = std::string("idkpt_trace_rays: ") + cudaGetErrorString(e); rc = IDKPT_ERR_CUDA; break; }
        if (kernelMs) cudaEventElapsedTime(kernelMs, e0, e1);
    } while (0);
    if (e0) cudaEventDestroy(e0);
    if (e1) cudaEventDestroy(e1);
    return rc;
}


// ---- device BLAS build (idk_blas_build.cuh) ----
enum BbBuf {
    BB_POS, BB_TRIS, BB_ITEMSTART, BB_TRIOFF, BB_PRESPLIT, BB_PRIO, BB_TOTALPRIO, BB_GBOX, BB_SPLITCOUNT, BB_ITEMBLAS,
    BB_BLASOFF, BB_BOUNDS, BB_FRAGTRI, BB_FRAGBLAS, BB_KEYS, BB_KEYS2, BB_VALS, BB_SORTED0, BB_SORTED1, BB_SORTED2,
    BB_TABLE, BB_AUX, BB_R0, BB_R1, BB_R2, BB_STACK, BB_NODES, BB_OUT, BB_DEPTH, BB_PARENT, BB_RSTART, BB_RCOUNT,
    BB_FRAGOFF, BB_FRAGCOUNT, BB_NODEBASE, BB_TASKS0, BB_TASKS1, BB_SMALL, BB_COUNTERS, BB_PERBLAS, BB_NODEI0, BB_NODEI1,
    BB_NODEI2, BB_NODEI3, BB_NODED0, BB_NODED1, BB_TRIOUT, BB_TEMP, BB_COUNT
};
static_assert(BB_COUNT <= 48, "IdkPtCtx::BlasBuild::buf");

__global__ void k_bb_gather_offsets(const long long* offset, const int* itemStart, int blasCount, long long* out) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b <= blasCount) out[b] = offset[itemStart[b]];
}

__global__ void k_bb_init_roots(idkbb::SplitArgs a, const int* fragCount, int blasCount) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= blasCount) return;
    const int n = fragCount[b];
    idkbb::createChild(a, a.nodeBase[b], 1, -1, 0, n, 0);
    idkbb::pushTask(a, {b, 1, 2, 0}, n);
}

static int bits_for(uint64_t v) { int b = 0; while (v) { b++; v >>= 1; } return b; }

IDKPT_API void idkpt_blas_default_build_settings(IdkPtBlasBuildSettings* s) {
    if (!s) return;
    s->StopSplittingThreshold = 1;
    s->MaxLeafTriangleCount = 2;
    s->TriangleCost = 1.1f;
    s->StackOptThreshold = 16;
    s->StackOptSahIncreaseAcceptance = 0.0009745f;
    s->SplitFactor = 0.3f;
    s->DoPreSplit = 1;
}

static inline float bb_half_area(const float mn[3], const float mx[3]) {
    const float sx = mx[0] - mn[0], sy = mx[1] - mn[1], sz = mx[2] - mn[2];
    return fmaf(sx + sy, sz, sx * sy);
}

IDKPT_API int idkpt_blas_build(IdkPtCtx* ctx, const PackedVec3* positions, uint64_t positionCount, const GpuBlasTriangle* triangles,
                               uint64_t triangleCount, const IdkPtBlasBuildDesc* descs, uint32_t blasCount,
                               const IdkPtBlasBuildSettings* settings, IdkPtBlasBuildInfo* infosOut, float* kernelMs) {
    if (!ctx) return IDKPT_ERR_INVALID_ARGUMENT;
    if (kernelMs) *kernelMs = 0.0f;
    auto& bb = ctx->bb;
    bb.infos.clear();
    bb.nodeBase.clear();
    bb.fragOffset.clear();
    if (blasCount == 0) return IDKPT_OK;
    if (!descs || !infosOut || (!positions && positionCount) || (!triangles && triangleCount))
        return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_blas_build: null argument");
    if (blasCount > 65535) return fail(ctx, IDKPT_ERR_UNSUPPORTED, "idkpt_blas_build: more than 65535 BLASes in one call");
    IdkPtBlasBuildSettings st;
    if (settings) st = *settings; else idkpt_blas_default_build_settings(&st);

    // ---- validation (host arrays, before any device work)
    for (uint64_t i = 0; i < positionCount; i++)
        if (!std::isfinite(positions[i].x) || !std::isfinite(positions[i].y) || !std::isfinite(positions[i].z))
            return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_blas_build: non-finite vertex position");
    uint64_t items = 0;
    for (uint32_t b = 0; b < blasCount; b++) {
        const IdkPtBlasBuildDesc& d = descs[b];
        if (d.TriangleCount == 0) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_blas_build: empty BLAS");
        if ((uint64_t)d.TriangleOffset + d.TriangleCount > triangleCount) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_blas_build: BLAS triangle range outside the triangle array");
        if (d.TriangleCount >= (uint32_t)idkbb::MAX_FRAGMENTS) return fail(ctx, IDKPT_ERR_UNSUPPORTED, "idkpt_blas_build: a BLAS of 2^24 or more fragments");
        float mn[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, mx[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
        for (uint32_t t = d.TriangleOffset; t < d.TriangleOffset + d.TriangleCount; t++) {
            const int32_t id[3] = {triangles[t].X, triangles[t].Y, triangles[t].Z};
            for (int v = 0; v < 3; v++) {
                if (id[v] < 0 || (uint64_t)id[v] >= positionCount) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_blas_build: vertex index outside the position array");
                const float p[3] = {positions[id[v]].x, positions[id[v]].y, positions[id[v]].z};
                for (int k = 0; k < 3; k++) { mn[k] = std::min(mn[k], p[k]); mx[k] = std::max(mx[k], p[k]); }
            }
        }
        if (!std::isfinite(bb_half_area(mn, mx))) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_blas_build: BLAS bounding box with a non-finite half-area");
        items += d.TriangleCount;
    }
    if (items >= (1ull << 31)) return fail(ctx, IDKPT_ERR_UNSUPPORTED, "idkpt_blas_build: 2^31 or more triangles in one call");
    const int B = (int)blasCount, W = (int)items;
    std::vector<int> itemStart(B + 1), triOff(B), presplit(B);
    for (int b = 0; b < B; b++) {
        itemStart[b + 1] = itemStart[b] + (int)descs[b].TriangleCount;
        triOff[b] = (int)descs[b].TriangleOffset;
        presplit[b] = st.DoPreSplit && !descs[b].IsRefittable;
    }

    CK(cudaSetDevice(ctx->device));
    if (!bb.stream) CK(cudaStreamCreateWithFlags(&bb.stream, cudaStreamNonBlocking));
    cudaStream_t s = bb.stream;
    DevBuf* buf = bb.buf;
    auto need = [&](int id, size_t bytes) { return ensure(buf[id], std::max<size_t>(bytes, 16)); };
#define BB_NEED(id, bytes) do { if (need(id, bytes) != cudaSuccess) return fail(ctx, IDKPT_ERR_OUT_OF_MEMORY, "idkpt_blas_build: device allocation failed"); } while (0)
#define BB_P(id, T) ((T*)buf[id].p)
    size_t tempBytes = 0;
    auto temp = [&](size_t bytes) -> cudaError_t { tempBytes = bytes; return need(BB_TEMP, bytes); };

    cudaEvent_t ev[7];
    for (int i = 0; i < 7; i++) CK(cudaEventCreate(&ev[i]));
    struct EvGuard { cudaEvent_t* e; ~EvGuard() { for (int i = 0; i < 7; i++) cudaEventDestroy(e[i]); } } evGuard{ev};

    // ---- pre-splitting
    BB_NEED(BB_POS, positionCount * 12); BB_NEED(BB_TRIS, triangleCount * 16);
    BB_NEED(BB_ITEMSTART, (B + 1) * 4); BB_NEED(BB_TRIOFF, B * 4); BB_NEED(BB_PRESPLIT, B * 4);
    BB_NEED(BB_PRIO, (size_t)W * 4); BB_NEED(BB_TOTALPRIO, B * 4); BB_NEED(BB_GBOX, B * sizeof(idkbb::Box));
    BB_NEED(BB_SPLITCOUNT, ((size_t)W + 1) * 8); BB_NEED(BB_ITEMBLAS, (size_t)W * 4); BB_NEED(BB_BLASOFF, (B + 1) * 8);
    if (positionCount) CK(cudaMemcpyAsync(buf[BB_POS].p, positions, positionCount * 12, cudaMemcpyHostToDevice, s));
    if (triangleCount) CK(cudaMemcpyAsync(buf[BB_TRIS].p, triangles, triangleCount * 16, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(buf[BB_ITEMSTART].p, itemStart.data(), (B + 1) * 4, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(buf[BB_TRIOFF].p, triOff.data(), B * 4, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(buf[BB_PRESPLIT].p, presplit.data(), B * 4, cudaMemcpyHostToDevice, s));
    cudaEventRecord(ev[0], s);
    idkbb::PreArgs pa;
    pa.pos = BB_P(BB_POS, float); pa.tris = BB_P(BB_TRIS, int4); pa.blasItemStart = BB_P(BB_ITEMSTART, int);
    pa.blasTriOffset = BB_P(BB_TRIOFF, int); pa.blasPresplit = BB_P(BB_PRESPLIT, int); pa.itemCount = W; pa.blasCount = B;
    pa.prio = BB_P(BB_PRIO, float); pa.totalPrio = BB_P(BB_TOTALPRIO, float); pa.globalBox = BB_P(BB_GBOX, idkbb::Box);
    pa.splitCount = BB_P(BB_SPLITCOUNT, long long); pa.itemBlas = BB_P(BB_ITEMBLAS, int); pa.splitFactor = st.SplitFactor;
    idkbb::k_item_prepare<<<(W + 255) / 256, 256, 0, s>>>(pa);
    idkbb::k_total_priority<<<(B + 127) / 128, 128, 0, s>>>(pa);
    idkbb::k_global_box<<<B, idkbb::NT, 0, s>>>(pa);
    idkbb::k_split_counts<<<(W + 256) / 256, 256, 0, s>>>(pa);
    CK(cub::DeviceScan::ExclusiveSum(nullptr, tempBytes, pa.splitCount, pa.splitCount, W + 1, s));
    CK(temp(tempBytes));
    CK(cub::DeviceScan::ExclusiveSum(buf[BB_TEMP].p, tempBytes, pa.splitCount, pa.splitCount, W + 1, s));
    k_bb_gather_offsets<<<(B + 128) / 128, 128, 0, s>>>(pa.splitCount, pa.blasItemStart, B, BB_P(BB_BLASOFF, long long));
    std::vector<long long> blasOff(B + 1);
    CK(cudaMemcpyAsync(blasOff.data(), buf[BB_BLASOFF].p, (B + 1) * 8, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    std::vector<int> fragOff(B), fragCount(B), nodeBase(B + 1);
    long long nodeSlots = 0;
    for (int b = 0; b < B; b++) {
        const long long n = blasOff[b + 1] - blasOff[b];
        if (n >= idkbb::MAX_FRAGMENTS) return fail(ctx, IDKPT_ERR_UNSUPPORTED, "idkpt_blas_build: a BLAS of 2^24 or more fragments");
        fragOff[b] = (int)blasOff[b];
        fragCount[b] = (int)n;
        nodeBase[b] = (int)nodeSlots;
        nodeSlots += std::max<long long>(2 * n, 4);
        if (nodeSlots >= (1ll << 31) || blasOff[b + 1] >= (1ll << 30)) return fail(ctx, IDKPT_ERR_UNSUPPORTED, "idkpt_blas_build: too many fragments in one call");
    }
    nodeBase[B] = (int)nodeSlots;
    const int F = (int)blasOff[B], NS = (int)nodeSlots;

    BB_NEED(BB_BOUNDS, (size_t)F * sizeof(idkbb::Box)); BB_NEED(BB_FRAGTRI, (size_t)F * 4); BB_NEED(BB_FRAGBLAS, (size_t)F * 4);
    idkbb::FragArgs fa;
    fa.pos = pa.pos; fa.tris = pa.tris; fa.blasItemStart = pa.blasItemStart; fa.blasTriOffset = pa.blasTriOffset;
    fa.blasPresplit = pa.blasPresplit; fa.itemBlas = pa.itemBlas; fa.offset = pa.splitCount; fa.globalBox = pa.globalBox;
    fa.itemCount = W; fa.fragCount = F;
    fa.bounds = BB_P(BB_BOUNDS, idkbb::Box); fa.fragTri = BB_P(BB_FRAGTRI, int); fa.fragBlas = BB_P(BB_FRAGBLAS, int);
    idkbb::k_fragments<<<(F + 255) / 256, 256, 0, s>>>(fa);
    cudaEventRecord(ev[1], s);

    // ---- three stable sorts by centroid key (the BLAS id in the high bits keeps every BLAS in its own range)
    const size_t keyN = std::max<size_t>(F, NS);
    BB_NEED(BB_KEYS, keyN * 8); BB_NEED(BB_KEYS2, keyN * 8); BB_NEED(BB_VALS, keyN * 4);
    BB_NEED(BB_SORTED0, (size_t)F * 4); BB_NEED(BB_SORTED1, (size_t)F * 4); BB_NEED(BB_SORTED2, (size_t)F * 4);
    unsigned long long *keys = BB_P(BB_KEYS, unsigned long long), *keys2 = BB_P(BB_KEYS2, unsigned long long);
    int* vals = BB_P(BB_VALS, int);
    int* sorted[3] = {BB_P(BB_SORTED0, int), BB_P(BB_SORTED1, int), BB_P(BB_SORTED2, int)};
    const int fragEndBit = 32 + bits_for((uint64_t)(B - 1));
    CK(cub::DeviceRadixSort::SortPairs(nullptr, tempBytes, keys, keys2, vals, sorted[0], F, 0, fragEndBit, s));
    CK(temp(tempBytes));
    for (int axis = 0; axis < 3; axis++) {
        idkbb::k_sort_keys<<<(F + 255) / 256, 256, 0, s>>>(fa.bounds, fa.fragBlas, F, axis, keys, vals);
        CK(cub::DeviceRadixSort::SortPairs(buf[BB_TEMP].p, tempBytes, keys, keys2, vals, sorted[axis], F, 0, fragEndBit, s));
    }
    cudaEventRecord(ev[2], s);

    // ---- splits: the top of every tree level by level, one block per node; subtrees of <= SMALL fragments one thread each
    BB_NEED(BB_TABLE, F); BB_NEED(BB_AUX, (size_t)F * 4); BB_NEED(BB_R0, (size_t)F * 4); BB_NEED(BB_R1, (size_t)F * 4);
    BB_NEED(BB_R2, (size_t)F * 4); BB_NEED(BB_STACK, (size_t)F * 12);
    BB_NEED(BB_NODES, (size_t)NS * 32); BB_NEED(BB_OUT, (size_t)NS * 32); BB_NEED(BB_DEPTH, (size_t)NS * 4);
    BB_NEED(BB_PARENT, (size_t)NS * 4); BB_NEED(BB_RSTART, (size_t)NS * 4); BB_NEED(BB_RCOUNT, (size_t)NS * 4);
    BB_NEED(BB_FRAGOFF, B * 4); BB_NEED(BB_FRAGCOUNT, B * 4); BB_NEED(BB_NODEBASE, (B + 1) * 4);
    const size_t bigCap = (size_t)F / idkbb::SMALL + 2 * (size_t)B + 16, smallCap = 2 * (size_t)F + 2 * (size_t)B + 16;
    BB_NEED(BB_TASKS0, bigCap * 16); BB_NEED(BB_TASKS1, bigCap * 16); BB_NEED(BB_SMALL, smallCap * 16); BB_NEED(BB_COUNTERS, 64);
    CK(cudaMemcpyAsync(buf[BB_FRAGOFF].p, fragOff.data(), B * 4, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(buf[BB_FRAGCOUNT].p, fragCount.data(), B * 4, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(buf[BB_NODEBASE].p, nodeBase.data(), (B + 1) * 4, cudaMemcpyHostToDevice, s));
    CK(cudaMemsetAsync(buf[BB_NODES].p, 0, (size_t)NS * 32, s));
    CK(cudaMemsetAsync(buf[BB_DEPTH].p, 0xFF, (size_t)NS * 4, s));
    CK(cudaMemsetAsync(buf[BB_COUNTERS].p, 0, 64, s));
    int* counters = BB_P(BB_COUNTERS, int);     // [0], [1]: big-task counts (ping-pong), [2]: small-task count
    idkbb::SplitArgs sa;
    sa.bounds = fa.bounds;
    for (int i = 0; i < 3; i++) sa.sorted[i] = sorted[i];
    sa.table = BB_P(BB_TABLE, uint8_t); sa.aux = BB_P(BB_AUX, int);
    sa.R[0] = BB_P(BB_R0, float); sa.R[1] = BB_P(BB_R1, float); sa.R[2] = BB_P(BB_R2, float);
    sa.stack = BB_P(BB_STACK, int); sa.nodes = BB_P(BB_NODES, GpuBlasNode);
    sa.depth = BB_P(BB_DEPTH, int); sa.parent = BB_P(BB_PARENT, int); sa.rangeStart = BB_P(BB_RSTART, int); sa.rangeCount = BB_P(BB_RCOUNT, int);
    sa.fragOffset = BB_P(BB_FRAGOFF, int); sa.nodeBase = BB_P(BB_NODEBASE, int);
    sa.s = {st.StopSplittingThreshold, st.MaxLeafTriangleCount, st.TriangleCost, st.StackOptThreshold, st.StackOptSahIncreaseAcceptance, st.SplitFactor};
    sa.small = BB_P(BB_SMALL, idkbb::Task); sa.smallCount = counters + 2;
    idkbb::Task* lists[2] = {BB_P(BB_TASKS0, idkbb::Task), BB_P(BB_TASKS1, idkbb::Task)};
    sa.in = nullptr; sa.inCount = 0; sa.outBig = lists[0]; sa.outBigCount = counters + 0;
    k_bb_init_roots<<<(B + 127) / 128, 128, 0, s>>>(sa, BB_P(BB_FRAGCOUNT, int), B);
    for (int level = 0;; level++) {
        const int cur = level & 1;
        int bigCount = 0;
        CK(cudaMemcpyAsync(&bigCount, counters + cur, 4, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        if (bigCount == 0) break;
        sa.in = lists[cur]; sa.inCount = bigCount;
        sa.outBig = lists[cur ^ 1]; sa.outBigCount = counters + (cur ^ 1);
        CK(cudaMemsetAsync(counters + (cur ^ 1), 0, 4, s));
        idkbb::k_split_big<<<bigCount, idkbb::NT, 0, s>>>(sa);
    }
    int smallCount = 0;
    CK(cudaMemcpyAsync(&smallCount, counters + 2, 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    if (smallCount) idkbb::k_split_small<<<(smallCount + 63) / 64, 64, 0, s>>>(sa, smallCount);
    cudaEventRecord(ev[3], s);

    // ---- stack optimisation
    BB_NEED(BB_PERBLAS, (size_t)B * 64);
    BB_NEED(BB_NODEI0, ((size_t)NS + 1) * 4); BB_NEED(BB_NODEI1, ((size_t)NS + 1) * 4); BB_NEED(BB_NODEI2, ((size_t)NS + 1) * 4);
    BB_NEED(BB_NODEI3, ((size_t)NS + 1) * 4 * 8); BB_NEED(BB_NODED0, ((size_t)NS + 1) * 8); BB_NEED(BB_NODED1, ((size_t)NS + 1) * 8 * 2);
    BB_NEED(BB_TRIOUT, (size_t)F * 16);
    int* perBlas = BB_P(BB_PERBLAS, int);      // 16 ints per BLAS slot group, laid out as arrays of B
    CK(cudaMemsetAsync(perBlas, 0, (size_t)B * 64, s));
    int* nodeI3 = BB_P(BB_NODEI3, int);
    const size_t NS1 = (size_t)NS + 1;
    idkbb::PostArgs q;
    q.nodes = sa.nodes; q.out = BB_P(BB_OUT, GpuBlasNode);
    q.depth = sa.depth; q.parent = sa.parent; q.rangeStart = sa.rangeStart; q.rangeCount = sa.rangeCount;
    q.nodeBase = sa.nodeBase; q.fragOffset = sa.fragOffset; q.fragCount = BB_P(BB_FRAGCOUNT, int);
    q.blasCount = B; q.nodeSlots = NS; q.s = sa.s;
    q.rootWasLeaf = perBlas; q.created = perBlas + B; q.rs0 = perBlas + 2 * B; q.finalK = perBlas + 3 * B; q.rsOut = perBlas + 4 * B;
    q.newCount = perBlas + 5 * B; q.triOutCount = perBlas + 6 * B; q.sah = (double*)(perBlas + 8 * B);
    q.keys = keys; q.vals = vals;
    q.pre = BB_P(BB_NODEI0, int); q.byDepth = BB_P(BB_NODEI1, int); q.prePos = BB_P(BB_NODEI2, int);
    q.cflag = nodeI3; q.size = nodeI3 + NS1; q.diff = nodeI3 + 2 * NS1; q.qualPre = nodeI3 + 3 * NS1; q.depthPre = nodeI3 + 4 * NS1;
    q.internalDep = nodeI3 + 5 * NS1; q.depthDep = nodeI3 + 6 * NS1; q.flag = nodeI3 + 7 * NS1;
    q.sahPre = BB_P(BB_NODED0, double); q.collPre = BB_P(BB_NODED1, double); q.collDep = q.collPre + NS1;
    q.newId = q.size;                 // sizes are dead once the stack optimisation has run
    q.pairCount = q.internalDep; q.uniqCount = q.depthDep; q.uniq = sa.aux;
    q.sorted0 = sorted[0]; q.fragTri = fa.fragTri; q.tris = pa.tris; q.triOut = BB_P(BB_TRIOUT, int4); q.presplit = pa.blasPresplit;
    const int nsBlocks = (NS + 256) / 256, bBlocks = (B + 127) / 128;
    const int nodeEndBit = 48 + bits_for((uint64_t)(B - 1));
    idkbb::k_root_fix<<<bBlocks, 128, 0, s>>>(q);
    idkbb::k_node_keys<<<nsBlocks, 256, 0, s>>>(q, 0);
    CK(cub::DeviceRadixSort::SortPairs(nullptr, tempBytes, keys, keys2, vals, q.pre, NS, 0, nodeEndBit, s));
    CK(temp(std::max(tempBytes, buf[BB_TEMP].bytes)));
    tempBytes = buf[BB_TEMP].bytes;
    CK(cub::DeviceRadixSort::SortPairs(buf[BB_TEMP].p, tempBytes, keys, keys2, vals, q.pre, NS, 0, nodeEndBit, s));
    idkbb::k_pre_pos<<<nsBlocks, 256, 0, s>>>(q);
    size_t scanBytes = 0;
    CK(cub::DeviceScan::ExclusiveSum(nullptr, scanBytes, q.cflag, q.cflag, NS + 1, s));
    size_t incBytes = 0;
    CK(cub::DeviceScan::InclusiveSum(nullptr, incBytes, q.diff, q.diff, NS + 1, s));
    CK(temp(std::max(std::max(scanBytes, incBytes), buf[BB_TEMP].bytes)));
    tempBytes = buf[BB_TEMP].bytes;
    size_t tb = tempBytes;
    CK(cub::DeviceScan::ExclusiveSum(buf[BB_TEMP].p, tb, q.cflag, q.cflag, NS + 1, s));
    idkbb::k_sizes_both<<<nsBlocks, 256, 0, s>>>(q);
    tb = tempBytes;
    CK(cub::DeviceScan::InclusiveSum(buf[BB_TEMP].p, tb, q.diff, q.diff, NS + 1, s));
    idkbb::k_terms<<<nsBlocks, 256, 0, s>>>(q);
    idkbb::k_node_keys<<<nsBlocks, 256, 0, s>>>(q, 1);
    tb = tempBytes;
    CK(cub::DeviceRadixSort::SortPairs(buf[BB_TEMP].p, tb, keys, keys2, vals, q.byDepth, NS, 0, nodeEndBit, s));
    idkbb::k_dep_arrays<<<nsBlocks, 256, 0, s>>>(q);
    idkbb::k_stack_opt<<<B, 32, 0, s>>>(q);
    cudaEventRecord(ev[4], s);

    // ---- compaction (RemoveEmptySubtrees)
    CK(cudaMemsetAsync(q.out, 0, (size_t)NS * 32, s));
    idkbb::k_survivors<<<nsBlocks, 256, 0, s>>>(q);
    tb = tempBytes;
    CK(cub::DeviceScan::ExclusiveSum(buf[BB_TEMP].p, tb, q.flag, q.flag, NS + 1, s));
    idkbb::k_emit<<<nsBlocks, 256, 0, s>>>(q);
    cudaEventRecord(ev[5], s);

    // ---- unindexing, SAH of the result
    idkbb::k_pair_counts<<<nsBlocks, 256, 0, s>>>(q);
    idkbb::k_leaf_counts<<<nsBlocks, 256, 0, s>>>(q);
    tb = tempBytes;
    CK(cub::DeviceScan::ExclusiveSum(buf[BB_TEMP].p, tb, q.flag, q.flag, NS + 1, s));
    idkbb::k_unindex_plain<<<nsBlocks, 256, 0, s>>>(q);
    idkbb::k_unindex_pairs<<<nsBlocks, 256, 0, s>>>(q);
    idkbb::k_final_terms<<<nsBlocks, 256, 0, s>>>(q);
    idkbb::k_final_sah<<<B, 32, 0, s>>>(q);
    cudaEventRecord(ev[6], s);
    std::vector<int> hostPer((size_t)B * 16);
    CK(cudaMemcpyAsync(hostPer.data(), perBlas, (size_t)B * 64, cudaMemcpyDeviceToHost, s));
    cudaError_t e = cudaStreamSynchronize(s);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) { ctx->lastError = std::string("idkpt_blas_build: ") + cudaGetErrorString(e); return IDKPT_ERR_CUDA; }
    for (int i = 0; i < 6; i++) cudaEventElapsedTime(&bb.phaseMs[i], ev[i], ev[i + 1]);
    if (kernelMs) cudaEventElapsedTime(kernelMs, ev[0], ev[6]);
    const double* sah = (const double*)(hostPer.data() + 8 * B);
    bb.infos.resize(B);
    for (int b = 0; b < B; b++) {
        IdkPtBlasBuildInfo& in = bb.infos[b];
        in.NodeCount = (uint32_t)hostPer[5 * B + b];
        in.TriangleCount = presplit[b] ? (uint32_t)hostPer[6 * B + b] : (uint32_t)fragCount[b];
        in.FragmentCount = (uint32_t)fragCount[b];
        in.RequiredStackSize = hostPer[4 * B + b];
        memcpy(&in.SahBits, &sah[b], 8);
        infosOut[b] = in;
    }
    bb.nodeBase = nodeBase;
    bb.fragOffset = fragOff;
#undef BB_NEED
#undef BB_P
    return IDKPT_OK;
}

IDKPT_API int idkpt_blas_build_read(IdkPtCtx* ctx, uint32_t blas, GpuBlasNode* nodesOut, GpuBlasTriangle* trianglesOut) {
    if (!ctx) return IDKPT_ERR_INVALID_ARGUMENT;
    auto& bb = ctx->bb;
    if (blas >= bb.infos.size()) return fail(ctx, IDKPT_ERR_INVALID_ARGUMENT, "idkpt_blas_build_read: no such BLAS in the last build");
    CK(cudaSetDevice(ctx->device));
    const IdkPtBlasBuildInfo& in = bb.infos[blas];
    if (nodesOut) CK(cudaMemcpyAsync(nodesOut, (const GpuBlasNode*)bb.buf[BB_OUT].p + bb.nodeBase[blas], (size_t)in.NodeCount * 32, cudaMemcpyDeviceToHost, bb.stream));
    if (trianglesOut) CK(cudaMemcpyAsync(trianglesOut, (const GpuBlasTriangle*)bb.buf[BB_TRIOUT].p + bb.fragOffset[blas], (size_t)in.TriangleCount * 16, cudaMemcpyDeviceToHost, bb.stream));
    CK(cudaStreamSynchronize(bb.stream));
    return IDKPT_OK;
}

IDKPT_API int idkpt_blas_build_phase_ms(IdkPtCtx* ctx, float* phaseMs, int32_t count) {
    if (!ctx || (!phaseMs && count > 0)) return IDKPT_ERR_INVALID_ARGUMENT;
    for (int i = 0; i < count && i < 6; i++) phaseMs[i] = ctx->bb.phaseMs[i];
    return IDKPT_OK;
}

} // extern "C"

#include "idkvx_impl.cuh"
