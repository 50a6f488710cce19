"""PathTracer: host-side mirror of IDKEngine.Render.PathTracer (SRC/Render/PathTracer.cs:10-346) whose body is the
libidkpt C ABI instead of GL dispatches -- the Python twin of the C# PathTracerNative class in INTEGRATION.md.

Same public members and meaning: ctor(width, height, settings), Compute(), SetSize(), ResetAccumulation(),
properties SamplesPerPixel, RayDepth, AccumulatedSamples, FocalLength, LenseRadius, DoDebugBVHTraversal,
DoTraceLights, DoRussianRoulette, DoRaySorting, OutputAOVs, images Result / AlbedoTexture / NormalTexture.
Setters reset the accumulation exactly where the C# setters do (PathTracer.cs:16-97).
Scene data the reference binds globally (SSBO/UBO slots) is handed over with SetScene()/SetSky()/SetFrame().
"""
import ctypes

import numpy as np

from . import capi
from . import gpu_types as gt


class IdkPtError(RuntimeError):
    pass


class PathTracer:
    def __init__(self, width, height, settings=None, device=0, tile=(8, 0, 1), lib_path=None, lanes=0, global_slots=False):
        """global_slots: IDKPT_CREATE_GLOBAL_SLOTS -- a tiled (multi-GPU) context numbers its alive rays over the WHOLE image, so the
        N-GPU image is bit-identical to the 1-GPU image (needs EnablePeerGather / ConnectPeers)."""
        self._lib = capi.load(lib_path)
        self._ctx = ctypes.c_void_p()
        self._settings = settings or capi.default_settings()
        flags = ((int(lanes) & 15) << 8) | (capi.IDKPT_CREATE_GLOBAL_SLOTS if global_slots else 0)   # IDKPT_CREATE_LANES
        ci = capi.IdkPtCreateInfo(device, width, height, tile[0], tile[1], tile[2], flags)
        rc = self._lib.idkpt_create(ctypes.byref(ci), ctypes.byref(self._ctx))
        if rc != 0:
            msg = self._lib.idkpt_last_error(None)
            raise IdkPtError(f"idkpt_create failed ({rc}): {msg.decode() if msg else ''}")
        self.width, self.height = width, height
        self.tile = tile
        self._frame = None
        self._keep = None
        self.last_stats = None
        self._export = False

    # ------------------------------------------------------------------ plumbing
    def _check(self, rc, what):
        if rc != 0:
            msg = self._lib.idkpt_last_error(self._ctx)
            raise IdkPtError(f"{what} failed ({rc}): {msg.decode() if msg else ''}")

    def Dispose(self):
        if self._ctx:
            self._lib.idkpt_destroy(self._ctx)
            self._ctx = ctypes.c_void_p()

    def __del__(self):
        try:
            self.Dispose()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.Dispose()

    # ------------------------------------------------------------------ scene hand-over
    def SetScene(self, scene):
        d, keep = capi.scene_desc(scene)
        self._check(self._lib.idkpt_set_scene(self._ctx, ctypes.byref(d)), "idkpt_set_scene")

    def UpdateRange(self, which, first, data):
        data = np.ascontiguousarray(data)
        self._check(self._lib.idkpt_update_range(self._ctx, which, first, len(data), data.ctypes.data), "idkpt_update_range")

    _READ_DTYPES = {capi.IDKPT_ARRAY_TLAS_NODES: gt.GpuTlasNode, capi.IDKPT_ARRAY_BLAS_NODES: gt.GpuBlasNode,
                    capi.IDKPT_ARRAY_VERTEX_POSITIONS: gt.PackedVec3, capi.IDKPT_ARRAY_VERTICES: gt.GpuVertex}

    def ReadRange(self, which, first, count):
        out = np.zeros(count, self._READ_DTYPES[which])
        self._check(self._lib.idkpt_read_range(self._ctx, which, first, count, out.ctypes.data), "idkpt_read_range")
        return out

    # ------------------------------------------------------------------ present chain (Application.cs:217-223)
    def PostProcess(self, settings=None, source=capi.IDKPT_IMAGE_RESULT, download=True):
        """Bloom + TonemapAndGammaCorrect of the accumulated frame. Returns (rgba8 [H, W, 4] or None, kernel ms)."""
        st = settings if settings is not None else capi.default_post_settings()
        out = np.zeros((self.height, self.width, 4), np.uint8) if download else None
        ms = ctypes.c_float()
        self._check(self._lib.idkpt_post_process(self._ctx, ctypes.byref(st), source, out.ctypes.data if download else None, ctypes.byref(ms)),
                    "idkpt_post_process")
        return out, ms.value

    # ------------------------------------------------------------------ denoise hand-off (PathTracerPipeline.Denoise, PathTracerPipeline.cs:165-194)
    def Denoise(self, settings=None):
        """Pack Result / Albedo / Normal into the OIDN-layout device buffers and run the built-in guided a-trous filter.
        Returns kernel ms; the output is `Denoised` (and PostProcess(source=IDKPT_IMAGE_DENOISED))."""
        st = settings if settings is not None else capi.default_denoise_settings()
        ms = ctypes.c_float()
        self._check(self._lib.idkpt_denoise(self._ctx, ctypes.byref(st), ctypes.byref(ms)), "idkpt_denoise")
        return ms.value

    @property
    def Denoised(self):
        return self._read(capi.IDKPT_IMAGE_DENOISED)

    def DenoiseDevicePtrs(self):
        """(beauty, albedo, normal, output) device pointers of the packed-RGB float buffers (OIDN Format.Float3) and their size."""
        p = [ctypes.c_void_p() for _ in range(4)]
        n = ctypes.c_uint64()
        self._check(self._lib.idkpt_denoise_device_ptrs(self._ctx, *[ctypes.byref(x) for x in p], ctypes.byref(n)), "idkpt_denoise_device_ptrs")
        return [x.value for x in p], n.value

    def DenoiseImportOutput(self):
        self._check(self._lib.idkpt_denoise_import_output(self._ctx), "idkpt_denoise_import_output")

    # ------------------------------------------------------------------ dynamic geometry (ModelManager.Update, ModelManager.cs:236-261)
    def SetSkinningData(self, unskinned):
        unskinned = np.ascontiguousarray(unskinned)
        assert unskinned.dtype == gt.GpuUnskinnedVertex
        self._check(self._lib.idkpt_set_skinning_data(self._ctx, unskinned.ctypes.data, len(unskinned)), "idkpt_set_skinning_data")

    def SkinVertices(self, joint_matrices, cmds):
        """joint_matrices: [J, 3, 4] float32 (row-major mat4x3); cmds: IdkPtSkinningCmd array. Returns kernel ms."""
        jm = np.ascontiguousarray(joint_matrices, np.float32).reshape(-1, 3, 4)
        cmds = np.ascontiguousarray(cmds)
        assert cmds.dtype == gt.IdkPtSkinningCmd
        ms = ctypes.c_float()
        self._check(self._lib.idkpt_skin_vertices(self._ctx, jm.ctypes.data, len(jm), cmds.ctypes.data, len(cmds), ctypes.byref(ms)), "idkpt_skin_vertices")
        return ms.value

    def BlasRefit(self, first, count=1):
        """BVH.GpuBlasesRefit (BVH.cs:472-489). Returns kernel ms."""
        ms = ctypes.c_float()
        self._check(self._lib.idkpt_blas_refit(self._ctx, first, count, ctypes.byref(ms)), "idkpt_blas_refit")
        return ms.value

    def TlasBuild(self, search_radius=15):
        """BVH.TlasBuild on the device (BVH.cs:278-298, TLAS.cs:28-141) from the refitted roots and current transforms. Returns kernel ms."""
        ms = ctypes.c_float()
        self._check(self._lib.idkpt_tlas_build(self._ctx, search_radius, ctypes.byref(ms)), "idkpt_tlas_build")
        return ms.value

    def BuildBlases(self, positions, jobs, settings=None):
        """BVH.BlasesBuild (BVH.cs:300-377) on the device, every BLAS of the batch in one call. positions: PackedVec3[V];
        jobs: list of (triangles: GpuBlasTriangle[T] with global vertex ids, presplit). settings: host.IdkBlasBuildSettings
        or capi.IdkPtBlasBuildSettings (Threads and DoPreSplit are ignored; presplit decides). Returns one dict per job,
        equal to what host.build_blas returns for the same input."""
        positions = np.ascontiguousarray(positions)
        assert positions.dtype == gt.PackedVec3
        tris = [np.ascontiguousarray(t) for t, _ in jobs]
        assert all(t.dtype == gt.GpuBlasTriangle for t in tris)
        allt = np.concatenate(tris) if tris else np.zeros(0, gt.GpuBlasTriangle)
        descs = np.zeros(len(jobs), gt.IdkPtBlasBuildDesc)
        descs["TriangleCount"] = [len(t) for t in tris]
        descs["TriangleOffset"] = np.concatenate([[0], np.cumsum(descs["TriangleCount"])[:-1]]) if len(jobs) else []
        descs["IsRefittable"] = [0 if presplit else 1 for _, presplit in jobs]
        st = capi.IdkPtBlasBuildSettings()
        self._lib.idkpt_blas_default_build_settings(ctypes.byref(st))
        if settings is not None:
            for name, _ in capi.IdkPtBlasBuildSettings._fields_:
                if name != "DoPreSplit":
                    setattr(st, name, getattr(settings, name))
        st.DoPreSplit = 1
        infos = np.zeros(len(jobs), gt.IdkPtBlasBuildInfo)
        ms = ctypes.c_float()
        self._check(self._lib.idkpt_blas_build(self._ctx, positions.ctypes.data, len(positions), allt.ctypes.data if len(allt) else None,
                                               len(allt), descs.ctypes.data, len(jobs), ctypes.byref(st), infos.ctypes.data,
                                               ctypes.byref(ms)), "idkpt_blas_build")
        self.last_blas_build_ms = ms.value
        out = []
        for b, info in enumerate(infos):
            nodes = np.zeros(int(info["NodeCount"]), gt.GpuBlasNode)
            tri = np.zeros(int(info["TriangleCount"]), gt.GpuBlasTriangle)
            self._check(self._lib.idkpt_blas_build_read(self._ctx, b, nodes.ctypes.data, tri.ctypes.data), "idkpt_blas_build_read")
            out.append(dict(nodes=nodes, triangles=tri, required_stack_size=int(info["RequiredStackSize"]),
                            fragment_count=int(info["FragmentCount"]), sah=float(np.array(info["SahBits"], np.uint64).view(np.float64))))
        return out

    def BuildBlas(self, positions, triangles, presplit=True, settings=None, threads=None):
        """One BLAS on the device: the same dict as host.build_blas(positions, triangles, presplit, settings=settings).
        threads is accepted for signature compatibility and ignored."""
        return self.BuildBlases(positions, [(triangles, presplit)], settings)[0]

    @property
    def BlasBuilder(self):
        """A builder for host.Scene.add(builder=...): called like host.build_blas, with .batch building all models of one add()."""
        pt = self

        def build(positions, triangles, presplit=True, threads=None, settings=None):
            return pt.BuildBlas(positions, triangles, presplit, settings)
        build.batch = lambda positions, jobs, settings=None: pt.BuildBlases(positions, jobs, settings)
        return build

    def BlasBuildPhaseMs(self):
        """Device ms of the last build: pre-split, sort, splits, stack optimisation, compaction, unindexing."""
        ms = (ctypes.c_float * 6)()
        self._check(self._lib.idkpt_blas_build_phase_ms(self._ctx, ms, 6), "idkpt_blas_build_phase_ms")
        return dict(zip(("presplit", "sort", "splits", "stack_opt", "compaction", "unindex"), list(ms)))

    def SetTextures(self, textures):
        """Replace the material texture table (list of dict(pixels, srgb, wrap_s, wrap_t), as host.Scene.textures)."""
        arr, keep = capi.texture_descs(textures)
        self._check(self._lib.idkpt_set_textures(self._ctx, ctypes.addressof(arr) if textures else None, len(textures)), "idkpt_set_textures")

    def SetSky(self, color, faces=None):
        """Constant colour, or cubemap faces [6, N, N, 4] float32 (SkyBoxManager's samplerCube, UBO 5)."""
        s = capi.sky_desc(color, faces)
        self._check(self._lib.idkpt_set_sky(self._ctx, ctypes.byref(s)), "idkpt_set_sky")

    def SetFrame(self, per_frame_data):
        """GpuPerFrameData (UBO 1). A changed camera resets the accumulation like Application.OnRender does
        (SRC/Application.cs:209-213)."""
        pf = np.ascontiguousarray(per_frame_data)
        assert pf.dtype == gt.GpuPerFrameData
        if self._frame is not None and pf.tobytes() != self._frame.tobytes():
            self.ResetAccumulation()
        self._frame = pf.copy()

    # ------------------------------------------------------------------ PathTracer surface
    def Compute(self, want_stats=True):
        if self._frame is None:
            raise IdkPtError("SetFrame() has not been called")
        stats = capi.IdkPtStats() if want_stats else None
        rc = self._lib.idkpt_compute(self._ctx, self._frame.ctypes.data, ctypes.byref(self._settings),
                                     ctypes.byref(stats) if want_stats else None)
        self._check(rc, "idkpt_compute")
        self.last_stats = stats
        return stats

    def ComputeAsync(self):
        """Queue one Compute() without waiting (stats == NULL): several samples stay in flight. Sync() waits."""
        if self._frame is None:
            raise IdkPtError("SetFrame() has not been called")
        self._check(self._lib.idkpt_compute(self._ctx, self._frame.ctypes.data, ctypes.byref(self._settings), None), "idkpt_compute")

    def StreamHandle(self):
        """cudaStream_t of the main (image) stream, e.g. for torch.cuda.ExternalStream."""
        h = ctypes.c_void_p()
        self._check(self._lib.idkpt_stream_handle(self._ctx, ctypes.byref(h)), "idkpt_stream_handle")
        return h.value

    def Sync(self):
        self._check(self._lib.idkpt_sync(self._ctx), "idkpt_sync")

    def SetSize(self, width, height):
        self._check(self._lib.idkpt_resize(self._ctx, width, height), "idkpt_resize")
        self.width, self.height = width, height

    def ResetAccumulation(self):
        self._check(self._lib.idkpt_reset_accumulation(self._ctx), "idkpt_reset_accumulation")

    @property
    def AccumulatedSamples(self):
        return int(self._lib.idkpt_accumulated_samples(self._ctx))

    def _read(self, which):
        img = np.zeros((self.height, self.width, 4), np.float32)
        self._check(self._lib.idkpt_read_result(self._ctx, which, img.ctypes.data, img.nbytes), "idkpt_read_result")
        return img

    @property
    def Result(self):
        return self._read(capi.IDKPT_IMAGE_RESULT)

    @property
    def AlbedoTexture(self):
        return self._read(capi.IDKPT_IMAGE_ALBEDO)

    @property
    def NormalTexture(self):
        return self._read(capi.IDKPT_IMAGE_NORMAL)

    def WriteResult(self, img, which=capi.IDKPT_IMAGE_RESULT, accumulated=None):
        img = np.ascontiguousarray(img, np.float32)
        self._check(self._lib.idkpt_write_result(self._ctx, which, img.ctypes.data, img.nbytes), "idkpt_write_result")
        if accumulated is not None:
            self._check(self._lib.idkpt_set_accumulated_samples(self._ctx, accumulated), "idkpt_set_accumulated_samples")

    def PresentAsync(self, host_ptr, nbytes, which=capi.IDKPT_IMAGE_RESULT):
        """Start copying the image of the last Compute() into host memory (pinned for full overlap) on a second stream;
        the next Compute() overlaps the transfer. PresentWait() blocks until it has landed."""
        self._check(self._lib.idkpt_present_async(self._ctx, which, host_ptr, nbytes), "idkpt_present_async")

    def PresentWait(self):
        self._check(self._lib.idkpt_present_wait(self._ctx), "idkpt_present_wait")

    def RegisterHostBuffer(self, host_ptr, nbytes):
        """Page-lock an engine-owned host buffer (e.g. the shared-memory frame every rank presents its stripes into)."""
        self._check(self._lib.idkpt_register_host_buffer(self._ctx, host_ptr, nbytes), "idkpt_register_host_buffer")

    def UnregisterHostBuffer(self, host_ptr):
        self._check(self._lib.idkpt_unregister_host_buffer(self._ctx, host_ptr), "idkpt_unregister_host_buffer")

    def EnablePeerGather(self, rank, world, exchange):
        """Multi-GPU: fuse the tile all-gather into Compute() over NVLink peer memory. `exchange(bytes) -> list[bytes]`
        must return every rank's blob in rank order (e.g. torch.distributed.all_gather_object)."""
        buf = (ctypes.c_uint8 * capi.IDKPT_GATHER_HANDLE_BYTES)()
        self._check(self._lib.idkpt_gather_export(self._ctx, buf, len(buf)), "idkpt_gather_export")
        blobs = exchange(bytes(buf))
        assert len(blobs) == world and all(len(b) == capi.IDKPT_GATHER_HANDLE_BYTES for b in blobs)
        allh = (ctypes.c_uint8 * (world * capi.IDKPT_GATHER_HANDLE_BYTES)).from_buffer_copy(b"".join(blobs))
        self._check(self._lib.idkpt_gather_import(self._ctx, rank, world, allh, len(allh)), "idkpt_gather_import")

    @staticmethod
    def ConnectPeers(tracers):
        """Single-process multi-GPU: wire the tile contexts (in tile order) to each other without IPC (idkpt_gather_connect)."""
        arr = (ctypes.c_void_p * len(tracers))(*[t._ctx.value for t in tracers])
        rc = tracers[0]._lib.idkpt_gather_connect(arr, len(tracers))
        if rc != 0:
            msgs = [t._lib.idkpt_last_error(t._ctx) for t in tracers]
            raise IdkPtError("idkpt_gather_connect failed (%d): %s" % (rc, "; ".join(m.decode() for m in msgs if m)))

    def GatheredDevicePtr(self):
        p, n = ctypes.c_void_p(), ctypes.c_uint64()
        self._check(self._lib.idkpt_gather_device_ptr(self._ctx, ctypes.byref(p), ctypes.byref(n)), "idkpt_gather_device_ptr")
        return p.value, n.value

    def ResultDevicePtr(self, which=capi.IDKPT_IMAGE_RESULT):
        p, n = ctypes.c_void_p(), ctypes.c_uint64()
        self._check(self._lib.idkpt_result_device_ptr(self._ctx, which, ctypes.byref(p), ctypes.byref(n)), "idkpt_result_device_ptr")
        return p.value, n.value

    def TileRows(self):
        n = ctypes.c_int32()
        self._lib.idkpt_tile_rows(self._ctx, ctypes.byref(n), None, 0)
        rows = np.zeros(n.value, np.int32)
        self._lib.idkpt_tile_rows(self._ctx, ctypes.byref(n), rows.ctypes.data, n.value)
        return rows

    def EnableWavefrontExport(self, on=True):
        self._export = on
        self._check(self._lib.idkpt_read_wavefront_rays(self._ctx, None, 1 if on else 0), "idkpt_read_wavefront_rays")

    def ReadWavefrontRays(self):
        rays = np.zeros(self.width * self.height, gt.GpuWavefrontRay)
        self._check(self._lib.idkpt_read_wavefront_rays(self._ctx, rays.ctypes.data, len(rays)), "idkpt_read_wavefront_rays")
        return rays

    def TraceRays(self, rays, trace_lights=False):
        """Stand-alone closest-hit batch (GPU analogue of BVH.Intersect, SRC/Bvh/BVH.cs:162-193)."""
        rays = np.ascontiguousarray(rays)
        assert rays.dtype == gt.IdkPtRay
        hits = np.zeros(len(rays), gt.IdkPtHit)
        ms = ctypes.c_float()
        self._check(self._lib.idkpt_trace_rays(self._ctx, rays.ctypes.data, len(rays), int(trace_lights),
                                               hits.ctypes.data, ctypes.byref(ms)), "idkpt_trace_rays")
        return hits, ms.value

    def TraceRaysAny(self, rays, trace_lights=False):
        """Any-hit / occlusion batch (TraceRayAny, BVHIntersect.glsl:299-411). hits["NodePairFetches"] == 1 where occluded."""
        rays = np.ascontiguousarray(rays)
        assert rays.dtype == gt.IdkPtRay
        hits = np.zeros(len(rays), gt.IdkPtHit)
        ms = ctypes.c_float()
        self._check(self._lib.idkpt_trace_rays_any(self._ctx, rays.ctypes.data, len(rays), int(trace_lights),
                                                   hits.ctypes.data, ctypes.byref(ms)), "idkpt_trace_rays_any")
        return hits, ms.value

    def ShadowsRayTraced(self, frame, depth, normal_rg, light_index, samples=1, noise_index=0, jitter=(0.0, 0.0), visibility=None):
        """PointShadowManager.ComputeRayTracedShadowMaps for one light: visibility image from a G-buffer (host arrays)."""
        h, w = depth.shape
        depth = np.ascontiguousarray(depth, np.float32)
        nrg = np.ascontiguousarray(normal_rg, np.float32)
        vis = np.zeros((h, w), np.float32) if visibility is None else np.ascontiguousarray(visibility, np.float32)
        jit = np.array(jitter, np.float32)
        frame = np.ascontiguousarray(frame)
        ms = ctypes.c_float()
        self._check(self._lib.idkpt_shadows_ray_traced(self._ctx, frame.ctypes.data, depth.ctypes.data, nrg.ctypes.data, w, h, light_index,
                                                       samples, noise_index, jit.ctypes.data, vis.ctypes.data, ctypes.byref(ms)), "idkpt_shadows_ray_traced")
        return vis, ms.value

    # ---- properties with the reference's reset-on-set behaviour
    def _reset_prop(name, sub=None):  # noqa: N805
        def get(self):
            return getattr(self._settings.Gpu if sub else self._settings, name)

        def set_(self, v):
            setattr(self._settings.Gpu if sub else self._settings, name, v)
            self.ResetAccumulation()
        return property(get, set_)

    def _plain_prop(name):  # noqa: N805
        def get(self):
            return getattr(self._settings, name)

        def set_(self, v):
            setattr(self._settings, name, v)
        return property(get, set_)

    RayDepth = _reset_prop("RayDepth")                          # PathTracer.cs:16-25
    FocalLength = _reset_prop("FocalLength", True)              # :39-48
    LenseRadius = _reset_prop("LenseRadius", True)              # :50-59
    DoDebugBVHTraversal = _reset_prop("DoDebugBVHTraversal", True)  # :61-71
    DoTraceLights = _reset_prop("DoTraceLights", True)          # :73-84
    DoRussianRoulette = _reset_prop("DoRussianRoulette", True)  # :86-97
    SamplesPerPixel = _plain_prop("SamplesPerPixel")            # :12
    DoRaySorting = _plain_prop("DoRaySorting")                  # :101-111
    OutputAOVs = _plain_prop("OutputAOVs")                      # :113-125
    CollectStats = _plain_prop("CollectStats")

    def GetGpuSettings(self):
        return self._settings.Gpu
