/*
 * idkpt.h -- C ABI of libidkpt, the B200-native replacement for the body of
 * IDKEngine.Render.PathTracer (reference: IDKEngine/Source/Render/PathTracer.cs).
 *
 * The C# class keeps its public surface (ctor / Compute / SetSize /
 * ResetAccumulation / properties, PathTracer.cs:10-125,170-346); its GL
 * dispatch sequence (PathTracer.cs:214-297) is replaced by P/Invoke calls into
 * the functions below (binding shown in INTEGRATION.md). Scene data that the
 * reference binds implicitly to fixed SSBO/UBO slots (ModelManager.cs:103-119,
 * BVH.cs:145-152, LightManager.cs:80) is handed over explicitly, in the same
 * struct layouts (idk_gpu_types.h).
 *
 * Conventions (mirroring the reference's own native interop, SRC/OIDN/OIDN.cs:
 * opaque handles, plain pointers + sizes, error string getter):
 *   - every function returns IDKPT_OK (0) or a negative IdkPtStatus;
 *   - idkpt_last_error() returns a UTF-8 string owned by the library;
 *   - host arrays are borrowed only for the duration of the call (copied);
 *   - a context is single-threaded (the engine's render thread);
 *   - there is NO CPU fallback: without a usable CUDA device idkpt_create fails.
 */
#ifndef IDKPT_H
#define IDKPT_H

#include "idk_gpu_types.h"

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define IDKPT_API __declspec(dllexport)
#else
#define IDKPT_API __attribute__((visibility("default")))
#endif

typedef struct IdkPtCtx IdkPtCtx;

typedef enum IdkPtStatus {
    IDKPT_OK = 0,
    IDKPT_ERR_INVALID_ARGUMENT = -1,
    IDKPT_ERR_NO_DEVICE = -2,
    IDKPT_ERR_CUDA = -3,
    IDKPT_ERR_NO_SCENE = -4,
    IDKPT_ERR_OUT_OF_MEMORY = -5,
    IDKPT_ERR_UNSUPPORTED = -6
} IdkPtStatus;

#define IDKPT_MAX_RAY_DEPTH 64

/* Replaces: new PathTracer(width, height, settings)   (PathTracer.cs:170-212).
 * Tile fields implement the multi-GPU screen split (one context per GPU):
 * image rows are cut into stripes of TileStripeHeight rows, stripe s belongs to
 * context (s % TileCount) == TileIndex. TileCount <= 1 => the whole image. */
#define IDKPT_CREATE_LANES(n) (((uint32_t)(n) & 15u) << 8)
/* Multi-GPU, strict parity: NHit seeds a ray's random numbers with its slot in the alive list (NHit/compute.glsl:
 * gl_GlobalInvocationID.x). By default a tile numbers its own alive rays (the N-GPU image is then a valid, but different,
 * Monte-Carlo estimate than the 1-GPU image, reproducible per GPU count). With this flag the ranks exchange their per-stripe
 * alive counts over NVLink once per bounce so that every ray gets its WHOLE-IMAGE slot: the N-GPU image is bit-identical to
 * the 1-GPU image. Needs the peers connected (idkpt_gather_import / idkpt_gather_connect) and every rank issuing the same
 * idkpt_compute calls; not available together with DoRaySorting. Ignored when TileCount <= 1. */
#define IDKPT_CREATE_GLOBAL_SLOTS (1u << 12)

typedef struct IdkPtCreateInfo {
    int32_t Device;            /* CUDA device ordinal */
    int32_t Width;
    int32_t Height;
    int32_t TileStripeHeight;  /* rows per stripe (multiple of 8), 0 => 8 */
    int32_t TileIndex;
    int32_t TileCount;
    uint32_t Flags;            /* 0, IDKPT_CREATE_LANES(n): samples in flight for asynchronous idkpt_compute (default 8, 1 = off), IDKPT_CREATE_GLOBAL_SLOTS */
} IdkPtCreateInfo;

/* Replaces the implicit SSBO bindings 4,5(vertices),8,9..: ModelManager.cs:103-119
 * (meshes, materials, vertices, positions, transforms) and BVH.cs:145-152,445-451
 * (nodes, triangles, descs, instances, tlas) plus LightManager.cs:80 (UBO 2). */
/* Material textures. The reference stores 64-bit GL bindless sampler handles in GpuMaterial (GpuMaterial.cs:8-67); here a
 * handle is an index into this table: 0 = the 1x1 white fallback (ModelLoader.cs:1855-1870), k > 0 = Textures[k-1]. Base
 * level only: the path tracer's compute shaders sample lod 0 (Surface.glsl:57-60). Uncompressed RGBA8 as the loader
 * creates for non-KTX images (BaseColor/Emissive sRGB, ModelLoader.cs:938-945), or the BC7 / BC5 / BC4 level-0 block stream of
 * a KTX2 image as it comes out of the loader's transcoder (decoded on the GPU at upload).
 * Channel use as in Surface.glsl:49-77: BaseColor rgba, MetallicRoughness r = metallic g = roughness, Normal rg,
 * Emissive rgb, Transmission r. */
typedef enum IdkPtTextureFormat {
    IDKPT_TEX_RGBA8_UNORM = 0, IDKPT_TEX_RGBA8_SRGB = 1,   /* what the loader creates for PNG / JPG images (ModelLoader.cs:938-945) */
    /* ABI 3: the KTX2 formats of ModelLoader.cs:954-968, handed over as the level-0 block stream exactly as the loader gives it
     * to glCompressedTextureSubImage2D: ceil(W/4) x ceil(H/4) blocks, row-major. Decoded once at upload (csrc/idk_bcn.cuh). */
    IDKPT_TEX_BC7_UNORM = 2, IDKPT_TEX_BC7_SRGB = 3,       /* 16-byte blocks -> exact RGBA8 */
    IDKPT_TEX_BC5_RG_UNORM = 4,                            /* 16-byte blocks (RGTC2) -> (R, G, 0, 1) in fp32 */
    IDKPT_TEX_BC4_R_UNORM = 5,                             /* 8-byte blocks (RGTC1) -> (R, 0, 0, 1) in fp32 */
    IDKPT_TEX_RG32F = 6, IDKPT_TEX_R32F = 7, IDKPT_TEX_RGBA32F = 8   /* uncompressed float texels (e.g. the R11G11B10F metallic-roughness image) */
} IdkPtTextureFormat;
#define IDKPT_TEX_FLAG_R_FROM_B 1   /* texture.SetSwizzleR(Swizzle.B): BC7 / RGBA metallic-roughness images keep metallic in B (ModelLoader.cs:989-994) */
#define IDKPT_TEX_FLAG_MAG_NEAREST 2 /* the glTF sampler's magFilter is NEAREST (9728; ModelLoader.cs:1166-1196): compute shaders sample at lod 0, i.e.
                                      * under MAGNIFICATION, so the sampler's MagFilter decides between this and bilinear (the default, LINEAR 9729) */
typedef struct IdkPtTextureDesc {
    const void* Pixels;       /* level 0, row 0 first (v = 0): Width*Height texels of the format, or its block stream for BCn */
    int32_t Width, Height;
    int32_t Format;           /* IdkPtTextureFormat */
    int32_t WrapS, WrapT;     /* GL enums as in the glTF sampler: 10497 REPEAT, 33071 CLAMP_TO_EDGE, 33648 MIRRORED_REPEAT */
    int32_t Flags;            /* IDKPT_TEX_FLAG_* (was padding before ABI 3: 0 keeps the old meaning) */
} IdkPtTextureDesc;

typedef struct IdkPtSceneDesc {
    const GpuBlasNode*      BlasNodes;       uint64_t BlasNodeCount;
    const GpuBlasTriangle*  BlasTriangles;   uint64_t BlasTriangleCount;
    const GpuBlasDesc*      BlasDescs;       uint64_t BlasDescCount;
    const GpuBlasInstance*  BlasInstances;   uint64_t BlasInstanceCount;
    const GpuTlasNode*      TlasNodes;       uint64_t TlasNodeCount;     /* may be NULL/0 */
    const GpuMeshTransform* MeshTransforms;  uint64_t MeshTransformCount;
    const GpuMesh*          Meshes;          uint64_t MeshCount;
    const GpuMaterial*      Materials;       uint64_t MaterialCount;
    const GpuVertex*        Vertices;        uint64_t VertexCount;
    const PackedVec3*       VertexPositions; uint64_t VertexPositionCount;
    const GpuLight*         Lights;          uint64_t LightCount;        /* <= 256 */
    int32_t UseTlas;        /* BVH.GpuUseTlas (BVH.cs:18-27); default 0 */
    int32_t BlasStackSize;  /* BVH.BlasStackSize (BVH.cs:29-45,559-567) = max RequiredStackSize */
    const IdkPtTextureDesc* Textures; uint64_t TextureCount;             /* may be NULL/0: every material handle must then be 0 */
} IdkPtSceneDesc;

typedef enum IdkPtArrayId {
    IDKPT_ARRAY_MESH_TRANSFORMS = 0,
    IDKPT_ARRAY_MESHES = 1,
    IDKPT_ARRAY_MATERIALS = 2,
    IDKPT_ARRAY_LIGHTS = 3,
    IDKPT_ARRAY_TLAS_NODES = 4,        /* update + read: BVH.TlasBuild re-upload (BVH.cs:278-283); needs a scene set with UseTlas */
    IDKPT_ARRAY_BLAS_NODES = 5,        /* read only (idkpt_read_range): refitted boxes for the host-side TLAS build */
    IDKPT_ARRAY_VERTEX_POSITIONS = 6,  /* read only: skinned positions (the download behind fenceCopiedSkinnedVerticesToHost, ModelManager.cs:282) */
    IDKPT_ARRAY_VERTICES = 7           /* read only: skinned normals / tangents */
} IdkPtArrayId;

/* Replaces SkyBoxManager's bindless samplerCube in UBO 5 (SkyBoxManager.cs:87):
 * either a constant colour or six rgba32f faces (+X,-X,+Y,-Y,+Z,-Z), FaceSize^2
 * texels each (row-major, GL face orientation), sampled with GL face selection +
 * bilinear filtering inside the face (clamp to edge). */
typedef struct IdkPtSkyDesc {
    float        Color[3];
    int32_t      FaceSize;       /* 0 => constant Color */
    const float* Faces[6];
} IdkPtSkyDesc;

/* PathTracer's runtime-mutable properties (PathTracer.cs:12-125). */
typedef struct IdkPtSettings {
    IdkPtGpuSettings Gpu;        /* FocalLength.. DoRussianRoulette */
    int32_t RayDepth;            /* default 7 (PathTracer.cs:211) */
    int32_t SamplesPerPixel;     /* default 1 (PathTracer.cs:12) */
    int32_t DoRaySorting;        /* default 0 (PathTracer.cs:173) */
    int32_t OutputAOVs;          /* default 0 (PathTracer.cs:174) */
    int32_t CollectStats;        /* count node-pair fetches / triangle tests (debugCost semantics, BVHIntersect.glsl:45,60) */
} IdkPtSettings;

typedef struct IdkPtStats {
    uint64_t Rays;                               /* TraceRay invocations of this call */
    uint64_t BounceRays[IDKPT_MAX_RAY_DEPTH];    /* per bounce, summed over samples */
    uint64_t NodePairFetches;                    /* S (valid if CollectStats) */
    uint64_t TriangleTests;                      /* T (valid if CollectStats) */
    uint64_t InstanceVisits;                     /* I (valid if CollectStats) */
    uint64_t Hits;                               /* rays that hit scene geometry (valid if CollectStats) */
    float    TotalMs;                            /* CUDA-event time of the whole call */
    float    TraverseMs;                         /* sum over traversal launches */
    float    ShadeMs;                            /* sum over shade launches */
    float    SortMs;
    float    OtherMs;                            /* ray-gen + accumulate */
    uint32_t KernelLaunches;
    uint32_t TraverseLaunches;
    float    BounceTraverseMs[IDKPT_MAX_RAY_DEPTH];   /* per bounce, summed over samples */
    float    BounceShadeMs[IDKPT_MAX_RAY_DEPTH];      /* shade + compaction */
    uint32_t BounceMaxSteps[IDKPT_MAX_RAY_DEPTH];     /* longest ray (node-pair fetches) per bounce (valid if CollectStats) */
    float    CompactMs;                          /* ABI 3: the ordered compaction launches alone (also contained in ShadeMs / BounceShadeMs) */
    float    AccumulateMs;                       /* ABI 3: FinalDraw (+ fused peer scatter and arrival wait) alone (also contained in OtherMs) */
} IdkPtStats;

typedef enum IdkPtImage {
    IDKPT_IMAGE_RESULT = 0,   /* PathTracer.Result        (PathTracer.cs:143) */
    IDKPT_IMAGE_ALBEDO = 1,   /* PathTracer.AlbedoTexture (PathTracer.cs:167) */
    IDKPT_IMAGE_NORMAL = 2,   /* PathTracer.NormalTexture (PathTracer.cs:168) */
    IDKPT_IMAGE_GATHERED = 3, /* full multi-GPU Result (idkpt_present_async only; needs idkpt_gather_import) */
    IDKPT_IMAGE_DENOISED = 4  /* PathTracerPipeline's denoised output texture (idkpt_denoise; untiled contexts) */
} IdkPtImage;

/* One ray / hit record of the stand-alone closest-hit query (the GPU analogue of
 * BVH.Intersect(in Ray, out RayHitInfo), SRC/Bvh/BVH.cs:162-193, with the GLSL
 * acceptance rules of SH/include/BVHIntersect.glsl:183-291). */
typedef struct IdkPtRay {
    float Origin[3];
    float TMax;
    float Direction[3];
    float _pad0;
} IdkPtRay;
IDK_STATIC_ASSERT(sizeof(IdkPtRay) == 32, "IdkPtRay must be 32 bytes");

typedef struct IdkPtHit {
    float    BaryX, BaryY;      /* HitInfo.BaryXY (BVHIntersect.glsl:10-16) */
    float    T;                 /* == TMax on miss */
    uint32_t TriangleId;        /* global index into BlasTriangles, ~0u on miss / light */
    uint32_t MeshTransformId;   /* or light index when TriangleId == ~0u and T < TMax */
    uint32_t NodePairFetches;   /* per-ray S */
    uint32_t TriangleTests;     /* per-ray T */
    uint32_t _pad0;
} IdkPtHit;
IDK_STATIC_ASSERT(sizeof(IdkPtHit) == 32, "IdkPtHit must be 32 bytes");

IDKPT_API int idkpt_create(const IdkPtCreateInfo* ci, IdkPtCtx** out);
IDKPT_API void idkpt_destroy(IdkPtCtx* ctx);                                  /* PathTracer.Dispose, PathTracer.cs:344 */
IDKPT_API const char* idkpt_last_error(IdkPtCtx* ctx);                        /* ctx may be NULL: error of the last failed create */

IDKPT_API int idkpt_set_scene(IdkPtCtx* ctx, const IdkPtSceneDesc* scene);    /* ModelManager.Add -> UpdateBuffers + BVH.BlasesBuild uploads (ModelManager.cs:207-213, BVH.cs:445-451) */
IDKPT_API int idkpt_update_range(IdkPtCtx* ctx, IdkPtArrayId which, uint64_t first, uint64_t count, const void* data); /* dirty-range uploads, ModelManager.cs:236-261; LightManager.cs:363-380 */
IDKPT_API int idkpt_set_sky(IdkPtCtx* ctx, const IdkPtSkyDesc* sky);
/* Replace the material texture table of the current scene (same rules as IdkPtSceneDesc.Textures); every handle stored in
 * a material must remain inside the new table. Resets the accumulation. */
IDKPT_API int idkpt_set_textures(IdkPtCtx* ctx, const IdkPtTextureDesc* textures, uint64_t count);

IDKPT_API int idkpt_resize(IdkPtCtx* ctx, int32_t width, int32_t height);     /* PathTracer.SetSize, PathTracer.cs:299-332 */
IDKPT_API int idkpt_reset_accumulation(IdkPtCtx* ctx);                        /* PathTracer.ResetAccumulation, PathTracer.cs:334 */
IDKPT_API uint32_t idkpt_accumulated_samples(IdkPtCtx* ctx);                  /* PathTracer.AccumulatedSamples, PathTracer.cs:27-37 */
IDKPT_API int idkpt_set_accumulated_samples(IdkPtCtx* ctx, uint32_t n);       /* restore a snapshot taken with idkpt_read_result */

/* PathTracer.Compute(), PathTracer.cs:214-271. Images stay on the device.
 * With stats: synchronous, one sample at a time, per-kernel CUDA-event times filled in.
 * With stats == NULL (and CollectStats / DoDebugBVHTraversal / the wavefront export off): ASYNCHRONOUS. The call queues its
 * samples and returns; up to `lanes` samples are in flight on separate streams, so the few-ray tail bounces of one sample
 * overlap the next sample's first bounces. Each sample's values, and the order in which samples are folded into the
 * images, are exactly those of the synchronous path. idkpt_present_async / idkpt_post_process / idkpt_read_result are
 * ordered after every queued sample; calls that change the scene or hand out device pointers wait for the queue to
 * drain; idkpt_sync waits explicitly and reports device-side errors (kernel fault, multi-GPU gather time-out). */
IDKPT_API int idkpt_compute(IdkPtCtx* ctx, const GpuPerFrameData* frame, const IdkPtSettings* settings, IdkPtStats* stats);
IDKPT_API int idkpt_sync(IdkPtCtx* ctx);
/* The context's main (image) stream as a cudaStream_t: FinalDraw of every sample, presents and post-processing run on it in
 * submission order, so an event recorded on it after N idkpt_compute calls completes when those N samples are in the image. */
IDKPT_API int idkpt_stream_handle(IdkPtCtx* ctx, void** stream);

/* Host read-back / restore of an rgba32f image of this context's tile rows in
 * full-image layout (rows not owned by the tile are left untouched). */
IDKPT_API int idkpt_read_result(IdkPtCtx* ctx, IdkPtImage which, void* dst_rgba32f, uint64_t bytes);
IDKPT_API int idkpt_write_result(IdkPtCtx* ctx, IdkPtImage which, const void* src_rgba32f, uint64_t bytes);

/* Asynchronous presentation: snapshot the image (ordered after the Compute that produced it) and copy it to host memory
 * (pinned for full overlap) on a second stream while the next idkpt_compute runs; idkpt_present_wait blocks until the
 * most recent transfer has landed. The GL-free analogue of handing Result to the presenter each frame. */
IDKPT_API int idkpt_present_async(IdkPtCtx* ctx, IdkPtImage which, void* dst_rgba32f_host, uint64_t bytes);
IDKPT_API int idkpt_present_wait(IdkPtCtx* ctx);
/* Page-lock (cudaHostRegister) a host buffer owned by the engine so that idkpt_present_async into it is asynchronous, e.g.
 * ONE frame in POSIX shared memory registered by every rank: each rank's idkpt_present_async(IDKPT_IMAGE_RESULT) then
 * delivers its own stripes to their final position over its own PCIe link (multi-GPU presentation without a root copy). */
IDKPT_API int idkpt_register_host_buffer(IdkPtCtx* ctx, void* host_ptr, uint64_t bytes);
IDKPT_API int idkpt_unregister_host_buffer(IdkPtCtx* ctx, void* host_ptr);

/* Multi-GPU tile gather over NVLink peer memory (no NCCL in the data path). Every rank calls idkpt_gather_export
 * (allocates a double-buffered full-size image + arrival flags + the global-slot table and returns 5 CUDA IPC handles =
 * 320 bytes; 4 handles / 256 bytes before ABI 4), the ranks
 * exchange the handles (torch.distributed, MPI, a socket...) and call idkpt_gather_import with all of them in rank
 * order. From then on the FinalDraw of every idkpt_compute also stores this rank's pixels into every rank's full image
 * at their final position and idkpt_compute returns once all ranks' tiles of that frame have arrived (or fails after
 * IDKPT_GATHER_TIMEOUT_MS, default 30 s, if a peer never delivers). idkpt_resize drops the mappings: export / exchange /
 * import again afterwards.
 * idkpt_gather_connect does the same for a host that drives every GPU from ONE process (like the reference engine): pass
 * the contexts in tile order (context r created with TileIndex r, TileCount world); no IPC, peer access is enabled here.
 * With ONE host thread feeding all contexts only queue work afterwards (idkpt_compute with stats == NULL): a synchronous call
 * would wait for peers whose work has not been submitted yet (and fail after the time-out). Resizing or destroying one
 * context invalidates what its peers hold of it: resize all, then connect again. */
#define IDKPT_GATHER_HANDLE_BYTES 320
IDKPT_API int idkpt_gather_export(IdkPtCtx* ctx, void* handles_out, uint64_t bytes);
IDKPT_API int idkpt_gather_import(IdkPtCtx* ctx, int32_t rank, int32_t world, const void* all_handles, uint64_t bytes);
IDKPT_API int idkpt_gather_connect(IdkPtCtx** ctxs, int32_t world);
IDKPT_API int idkpt_gather_device_ptr(IdkPtCtx* ctx, void** dev_ptr, uint64_t* bytes);

/* Device-side access for zero-copy hand-over (GL interop / NCCL gather):
 * pointer to this tile's compact rgba32f rows (TileRowCount*Width float4). */
IDKPT_API int idkpt_result_device_ptr(IdkPtCtx* ctx, IdkPtImage which, void** dev_ptr, uint64_t* bytes);
IDKPT_API int idkpt_tile_rows(IdkPtCtx* ctx, int32_t* row_count, int32_t* rows_out, int32_t capacity);

/* Export the wavefront state of the last compute() call in the reference's
 * per-pixel layout (GpuWavefrontRay[W*H], SSBO 30) for inspection / parity. */
IDKPT_API int idkpt_read_wavefront_rays(IdkPtCtx* ctx, GpuWavefrontRay* dst, uint64_t count);

/* Stand-alone closest-hit batch with host buffers (H2D + kernel + D2H inside). */
IDKPT_API int idkpt_trace_rays(IdkPtCtx* ctx, const IdkPtRay* rays, uint64_t count, int32_t trace_lights, IdkPtHit* hits_out, float* kernel_ms);

/* ---- "next" rows of the scope table (SURVEY.md 8f.1), built on the same traversal code ----
 * Any-hit (occlusion) batch: TraceRayAny / IntersectBlasAny (BVHIntersect.glsl:107-181,299-411). hits_out[i].NodePairFetches
 * is 1 if the ray is occluded, 0 otherwise; T/TriangleId/Bary describe the first accepted (not the closest) hit. */
IDKPT_API int idkpt_trace_rays_any(IdkPtCtx* ctx, const IdkPtRay* rays, uint64_t count, int32_t trace_lights, IdkPtHit* hits_out, float* kernel_ms);

/* Ray-traced point-light shadows: ShadowsRayTraced/compute.glsl for one light (PointShadowManager.ComputeRayTracedShadowMaps,
 * Source/Render/PointShadowManager.cs:53-75). Host arrays: depth [w*h], octahedral normal rg [w*h*2]; visibility_out [w*h] is
 * read-modify-write (pixels with depth == 1 are left untouched, as the shader returns early). noise_index = the
 * (Frame % SampleCount) * samples term (0 without TAA); taa_jitter may be NULL. */
IDKPT_API int idkpt_shadows_ray_traced(IdkPtCtx* ctx, const GpuPerFrameData* frame, const float* depth, const float* normalRG,
                                       int32_t width, int32_t height, int32_t light_index, int32_t samples, uint32_t noise_index,
                                       const float* taa_jitter, float* visibility_out, float* kernel_ms);

/* ---- dynamic geometry (SURVEY.md 8f.2): ModelManager.Update = skin -> refit -> TLAS (ModelManager.cs:236-261) ----
 * idkpt_set_skinning_data: unskinnedVertexSSBO upload (52-byte GpuUnskinnedVertex records).
 * idkpt_skin_vertices: uploads the joint matrices (row-major mat4x3 = 3 x vec4 each, ModelManager.cs:272-277) and runs
 *   Skinning/compute.glsl once per command; positions, normals and tangents are rewritten in place on the device.
 * idkpt_blas_refit: BVH.GpuBlasesRefit(first, count) (BVH.cs:472-489, BLASRefit/compute.glsl); also refreshes the derived
 *   triangle records of the refitted BLASes. Call it for every BLAS whose vertices moved.
 * idkpt_read_range: device -> host read-back (refitted BLAS nodes for the host TLAS build, skinned vertices).
 * All of them reset the accumulation like any other scene edit. */
typedef struct IdkPtSkinningCmd {     /* ModelManager.SkinningCmd, Skinning/compute.glsl:9-12 uniforms */
    uint32_t InputVertexOffset;
    uint32_t OutputVertexOffset;
    uint32_t JointMatricesOffset;
    uint32_t VertexCount;
} IdkPtSkinningCmd;

IDKPT_API int idkpt_set_skinning_data(IdkPtCtx* ctx, const GpuUnskinnedVertex* vertices, uint64_t count);
IDKPT_API int idkpt_skin_vertices(IdkPtCtx* ctx, const float* joint_matrices, uint64_t joint_count, const IdkPtSkinningCmd* cmds, uint32_t cmd_count, float* kernel_ms);
IDKPT_API int idkpt_blas_refit(IdkPtCtx* ctx, uint32_t first_blas, uint32_t count, float* kernel_ms);
IDKPT_API int idkpt_read_range(IdkPtCtx* ctx, IdkPtArrayId which, uint64_t first, uint64_t count, void* out);
/* BVH.TlasBuild() on the device (BVH.cs:278-298 + TLAS.Build, TLAS.cs:28-141, serial PLOC with TLAS.BuildSettings.SearchRadius = 15):
 * world bounds of every instance from the (refitted) BLAS roots and the current mesh transforms, both already in HBM; fills the
 * scene's TLAS node array (UseTlas scenes) with exactly the nodes the host build produces -- a moving scene reads nothing back. */
IDKPT_API int idkpt_tlas_build(IdkPtCtx* ctx, int32_t search_radius, float* kernel_ms);

/* ---- BLAS build on the device (SURVEY.md 8f row 4): BVH.BlasesBuild(start, count) (BVH.cs:300-377) for a batch of BLASes.
 * SweepSAH with pre-splitting, node for node and byte for byte equal to the host builder (host_mirror/bvh_build.cpp, the
 * C# BLAS.Build it mirrors). A pure function of its inputs: it reads and writes no scene, image or accumulation state and
 * works on a context without a scene. Results live in the context until the next build or idkpt_destroy.
 *   positions: PackedVec3[positionCount]; triangles: GpuBlasTriangle[triangleCount] with global vertex ids and MeshId set
 *   (what BVH.Add produces); descs[blasCount]: one BLAS each, over triangles[TriangleOffset, TriangleOffset + TriangleCount).
 *   settings: NULL = idkpt_blas_default_build_settings. infos_out[blasCount] receives each BLAS's sizes.
 * IDKPT_ERR_INVALID_ARGUMENT: a vertex index outside positionCount, an empty BLAS, a range outside the triangle array,
 *   a non-finite position, or a BLAS whose bounding box has a non-finite half-area (NaN split costs).
 * IDKPT_ERR_UNSUPPORTED: a BLAS of 2^24 fragments or more (the builder counts in floats), more than 65535 BLASes or
 *   2^31 fragments in one call. */
typedef struct IdkPtBlasBuildSettings {   /* BLAS.BuildSettings (BLAS.cs:31-48) + PreSplitting.Settings (PreSplitting.cs:17-24) */
    int32_t StopSplittingThreshold;       /* 1 */
    int32_t MaxLeafTriangleCount;         /* 2 */
    float   TriangleCost;                 /* 1.1 */
    int32_t StackOptThreshold;            /* 16 */
    float   StackOptSahIncreaseAcceptance;/* 0.0009745 */
    float   SplitFactor;                  /* 0.3 */
    int32_t DoPreSplit;                   /* 1: pre-split every BLAS whose IsRefittable is 0 */
} IdkPtBlasBuildSettings;
IDK_STATIC_ASSERT(sizeof(IdkPtBlasBuildSettings) == 28, "IdkPtBlasBuildSettings must be 28 bytes");

typedef struct IdkPtBlasBuildDesc {
    uint32_t TriangleOffset;              /* into the call's triangle array */
    uint32_t TriangleCount;
    int32_t  IsRefittable;                /* 0 selects pre-splitting (BVH.cs:324-333) */
    int32_t  _pad0;
} IdkPtBlasBuildDesc;
IDK_STATIC_ASSERT(sizeof(IdkPtBlasBuildDesc) == 16, "IdkPtBlasBuildDesc must be 16 bytes");

typedef struct IdkPtBlasBuildInfo {       /* what the host builder reports for the same BLAS */
    uint32_t NodeCount;                   /* GpuBlasNode records, node 0 = pad, node 1 = root */
    uint32_t TriangleCount;               /* GpuBlasTriangle records (unindexed) */
    uint32_t FragmentCount;               /* triangles after pre-splitting */
    int32_t  RequiredStackSize;
    uint64_t SahBits;                     /* BLAS.ComputeGlobalSAH of the result: the bits of the double (memcpy / BitConverter) */
} IdkPtBlasBuildInfo;
IDK_STATIC_ASSERT(sizeof(IdkPtBlasBuildInfo) == 24, "IdkPtBlasBuildInfo must be 24 bytes");

IDKPT_API void idkpt_blas_default_build_settings(IdkPtBlasBuildSettings* settings);
IDKPT_API int idkpt_blas_build(IdkPtCtx* ctx, const PackedVec3* positions, uint64_t positionCount, const GpuBlasTriangle* triangles,
                               uint64_t triangleCount, const IdkPtBlasBuildDesc* descs, uint32_t blasCount,
                               const IdkPtBlasBuildSettings* settings, IdkPtBlasBuildInfo* infos_out, float* kernel_ms);
/* Copies BLAS `blas` of the last build: nodes_out[NodeCount], triangles_out[TriangleCount] (either may be NULL). */
IDKPT_API int idkpt_blas_build_read(IdkPtCtx* ctx, uint32_t blas, GpuBlasNode* nodes_out, GpuBlasTriangle* triangles_out);
/* Device time of the last build's phases in ms: pre-split, sort, splits, stack optimisation, compaction, unindexing. */
IDKPT_API int idkpt_blas_build_phase_ms(IdkPtCtx* ctx, float* phase_ms_out, int32_t count);

/* ---- present chain (SURVEY.md 8f.3): Bloom.Compute(Result) + TonemapAndGamma.Compute(Result, Bloom.Result)
 * (Application.cs:217-223) -> the RGBA8 frame the reference copies to the swapchain, produced on the device. ---- */
typedef struct IdkPtPostSettings {
    float   Exposure;                    /* TonemapAndGammaCorrect.GpuSettings (TonemapAndGammaCorrecter.cs:10-22): 0.45 */
    float   Saturation;                  /* 1.06 */
    float   Linear;                      /* 0.18 */
    float   Peak;                        /* 1.0 */
    float   Compression;                 /* 0.1 */
    int32_t DoTonemapAndSrgbTransform;   /* 1 */
    int32_t IsBloom;                     /* Application.IsBloom, default 1 */
    float   BloomThreshold;              /* Bloom.GpuSettings (Bloom.cs:10-19): 1.5 */
    float   BloomMaxColor;               /* 3.8 */
    int32_t BloomMinusLods;              /* Bloom.MinusLods, default 3 */
} IdkPtPostSettings;

/* source: IDKPT_IMAGE_RESULT/ALBEDO/NORMAL of an untiled context, or IDKPT_IMAGE_GATHERED (full multi-GPU frame).
 * rgba8_out: host buffer of width*height*4 bytes (row-major, R8G8B8A8Unorm), or NULL to keep the frame on the device
 * (idkpt_ldr_device_ptr). */
IDKPT_API int idkpt_post_process(IdkPtCtx* ctx, const IdkPtPostSettings* settings, IdkPtImage source, uint8_t* rgba8_out, float* kernel_ms);
IDKPT_API int idkpt_ldr_device_ptr(IdkPtCtx* ctx, void** dev_ptr, uint64_t* bytes);

/* ---- denoise hand-off (SURVEY.md 8f.3): PathTracerPipeline.Denoise (PathTracerPipeline.cs:165-194) without the host round trip.
 * idkpt_denoise packs Result / AlbedoTexture / NormalTexture into OIDN-layout buffers on the device (packed RGB floats,
 * Format.Float3: what Texture.Download(PixelFormat.RGB, Float) fills today) and runs the built-in guided a-trous filter into
 * the denoised image (IDKPT_IMAGE_DENOISED: idkpt_read_result, idkpt_post_process source) and into the OIDN output buffer.
 * A host that links OIDN's CUDA device wraps the four pointers of idkpt_denoise_device_ptrs with oidnNewSharedBuffer, calls
 * idkpt_denoise with Iterations = 0 (pack only), executes its filters, and then idkpt_denoise_import_output takes the
 * output buffer over as the denoised image -- nothing crosses PCIe. Needs OutputAOVs samples in the AOV images. ---- */
typedef struct IdkPtDenoiseSettings {
    int32_t Iterations;      /* a-trous passes (step 1, 2, 4, ...); 5 = default; 0 = only pack the OIDN buffers */
    float   SigmaColor;      /* 3.0: colour edge-stopping on the (demodulated) radiance, halved every pass */
    float   SigmaNormal;     /* 0.35 */
    float   SigmaAlbedo;     /* 0.25 */
    int32_t Demodulate;      /* 1: filter colour / max(albedo, 1e-3) and re-apply the albedo afterwards */
} IdkPtDenoiseSettings;
IDKPT_API int idkpt_denoise(IdkPtCtx* ctx, const IdkPtDenoiseSettings* settings, float* kernel_ms);
IDKPT_API int idkpt_denoise_device_ptrs(IdkPtCtx* ctx, void** beauty, void** albedo, void** normal, void** output, uint64_t* bytes_each);
IDKPT_API int idkpt_denoise_import_output(IdkPtCtx* ctx);

IDKPT_API uint32_t idkpt_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* IDKPT_H */
