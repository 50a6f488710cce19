"""ctypes declarations of include/idkpt.h -- the stand-in for the C# [LibraryImport] stubs of INTEGRATION.md.
No compute lives here; this only marshals the engine's arrays across the C ABI."""
import ctypes
import os

import numpy as np

from . import build as _build

c_i32, c_u32, c_u64, c_f = ctypes.c_int32, ctypes.c_uint32, ctypes.c_uint64, ctypes.c_float
c_vp = ctypes.c_void_p

IDKPT_MAX_RAY_DEPTH = 64


class IdkPtGpuSettings(ctypes.Structure):
    _fields_ = [("FocalLength", c_f), ("LenseRadius", c_f), ("DoDebugBVHTraversal", c_i32),
                ("DoTraceLights", c_i32), ("DoRussianRoulette", c_i32)]


class IdkPtCreateInfo(ctypes.Structure):
    _fields_ = [("Device", c_i32), ("Width", c_i32), ("Height", c_i32), ("TileStripeHeight", c_i32),
                ("TileIndex", c_i32), ("TileCount", c_i32), ("Flags", c_u32)]


IDKPT_TEX_RGBA8_UNORM, IDKPT_TEX_RGBA8_SRGB = 0, 1
IDKPT_TEX_BC7_UNORM, IDKPT_TEX_BC7_SRGB, IDKPT_TEX_BC5_RG_UNORM, IDKPT_TEX_BC4_R_UNORM = 2, 3, 4, 5
IDKPT_TEX_RG32F, IDKPT_TEX_R32F, IDKPT_TEX_RGBA32F = 6, 7, 8
IDKPT_TEX_FLAG_R_FROM_B, IDKPT_TEX_FLAG_MAG_NEAREST = 1, 2
GL_REPEAT, GL_CLAMP_TO_EDGE, GL_MIRRORED_REPEAT = 10497, 33071, 33648


class IdkPtTextureDesc(ctypes.Structure):
    _fields_ = [("Pixels", c_vp), ("Width", c_i32), ("Height", c_i32), ("Format", c_i32), ("WrapS", c_i32), ("WrapT", c_i32), ("Flags", c_i32)]


class IdkPtSceneDesc(ctypes.Structure):
    _fields_ = [
        ("BlasNodes", c_vp), ("BlasNodeCount", c_u64),
        ("BlasTriangles", c_vp), ("BlasTriangleCount", c_u64),
        ("BlasDescs", c_vp), ("BlasDescCount", c_u64),
        ("BlasInstances", c_vp), ("BlasInstanceCount", c_u64),
        ("TlasNodes", c_vp), ("TlasNodeCount", c_u64),
        ("MeshTransforms", c_vp), ("MeshTransformCount", c_u64),
        ("Meshes", c_vp), ("MeshCount", c_u64),
        ("Materials", c_vp), ("MaterialCount", c_u64),
        ("Vertices", c_vp), ("VertexCount", c_u64),
        ("VertexPositions", c_vp), ("VertexPositionCount", c_u64),
        ("Lights", c_vp), ("LightCount", c_u64),
        ("UseTlas", c_i32), ("BlasStackSize", c_i32),
        ("Textures", c_vp), ("TextureCount", c_u64),
    ]


class IdkPtSkyDesc(ctypes.Structure):
    _fields_ = [("Color", c_f * 3), ("FaceSize", c_i32), ("Faces", c_vp * 6)]


class IdkPtSettings(ctypes.Structure):
    _fields_ = [("Gpu", IdkPtGpuSettings), ("RayDepth", c_i32), ("SamplesPerPixel", c_i32),
                ("DoRaySorting", c_i32), ("OutputAOVs", c_i32), ("CollectStats", c_i32)]


class IdkPtStats(ctypes.Structure):
    _fields_ = [("Rays", c_u64), ("BounceRays", c_u64 * IDKPT_MAX_RAY_DEPTH),
                ("NodePairFetches", c_u64), ("TriangleTests", c_u64), ("InstanceVisits", c_u64), ("Hits", c_u64),
                ("TotalMs", c_f), ("TraverseMs", c_f), ("ShadeMs", c_f), ("SortMs", c_f), ("OtherMs", c_f),
                ("KernelLaunches", c_u32), ("TraverseLaunches", c_u32),
                ("BounceTraverseMs", c_f * IDKPT_MAX_RAY_DEPTH), ("BounceShadeMs", c_f * IDKPT_MAX_RAY_DEPTH),
                ("BounceMaxSteps", c_u32 * IDKPT_MAX_RAY_DEPTH), ("CompactMs", c_f), ("AccumulateMs", c_f)]

    def as_dict(self):
        arrays = ("BounceRays", "BounceTraverseMs", "BounceShadeMs", "BounceMaxSteps")
        d = {n: getattr(self, n) for n, _ in self._fields_ if n not in arrays}
        d["BounceRays"] = [int(v) for v in self.BounceRays]
        d["BounceTraverseMs"] = [float(v) for v in self.BounceTraverseMs]
        d["BounceShadeMs"] = [float(v) for v in self.BounceShadeMs]
        d["BounceMaxSteps"] = [int(v) for v in self.BounceMaxSteps]
        return d


IDKPT_IMAGE_RESULT, IDKPT_IMAGE_ALBEDO, IDKPT_IMAGE_NORMAL, IDKPT_IMAGE_GATHERED, IDKPT_IMAGE_DENOISED = 0, 1, 2, 3, 4
IDKPT_GATHER_HANDLE_BYTES = 320
IDKPT_CREATE_GLOBAL_SLOTS = 1 << 12
IDKPT_ARRAY_MESH_TRANSFORMS, IDKPT_ARRAY_MESHES, IDKPT_ARRAY_MATERIALS, IDKPT_ARRAY_LIGHTS = 0, 1, 2, 3
IDKPT_ARRAY_TLAS_NODES, IDKPT_ARRAY_BLAS_NODES, IDKPT_ARRAY_VERTEX_POSITIONS, IDKPT_ARRAY_VERTICES = 4, 5, 6, 7

# every symbol include/idkpt.h declares
EXPORTS = [
    "idkpt_create", "idkpt_destroy", "idkpt_last_error", "idkpt_set_scene", "idkpt_update_range", "idkpt_set_sky", "idkpt_set_textures",
    "idkpt_resize", "idkpt_reset_accumulation", "idkpt_accumulated_samples", "idkpt_set_accumulated_samples",
    "idkpt_compute", "idkpt_sync", "idkpt_stream_handle", "idkpt_read_result", "idkpt_write_result", "idkpt_present_async", "idkpt_present_wait",
    "idkpt_register_host_buffer", "idkpt_unregister_host_buffer",
    "idkpt_gather_export", "idkpt_gather_import", "idkpt_gather_connect", "idkpt_gather_device_ptr",
    "idkpt_result_device_ptr", "idkpt_tile_rows",
    "idkpt_read_wavefront_rays", "idkpt_trace_rays", "idkpt_trace_rays_any", "idkpt_shadows_ray_traced",
    "idkpt_set_skinning_data", "idkpt_skin_vertices", "idkpt_blas_refit", "idkpt_read_range", "idkpt_post_process", "idkpt_ldr_device_ptr", "idkpt_abi_version",
    "idkpt_denoise", "idkpt_denoise_device_ptrs", "idkpt_denoise_import_output", "idkpt_tlas_build",
    "idkpt_blas_default_build_settings", "idkpt_blas_build", "idkpt_blas_build_read", "idkpt_blas_build_phase_ms",
]


class IdkPtBlasBuildSettings(ctypes.Structure):
    _fields_ = [("StopSplittingThreshold", c_i32), ("MaxLeafTriangleCount", c_i32), ("TriangleCost", c_f),
                ("StackOptThreshold", c_i32), ("StackOptSahIncreaseAcceptance", c_f), ("SplitFactor", c_f), ("DoPreSplit", c_i32)]


class IdkPtBlasBuildInfo(ctypes.Structure):
    _fields_ = [("NodeCount", c_u32), ("TriangleCount", c_u32), ("FragmentCount", c_u32), ("RequiredStackSize", c_i32),
                ("SahBits", c_u64)]


class IdkPtDenoiseSettings(ctypes.Structure):
    _fields_ = [("Iterations", c_i32), ("SigmaColor", c_f), ("SigmaNormal", c_f), ("SigmaAlbedo", c_f), ("Demodulate", c_i32)]


def default_denoise_settings():
    return IdkPtDenoiseSettings(5, 3.0, 0.35, 0.25, 1)


class IdkPtPostSettings(ctypes.Structure):
    _fields_ = [("Exposure", c_f), ("Saturation", c_f), ("Linear", c_f), ("Peak", c_f), ("Compression", c_f),
                ("DoTonemapAndSrgbTransform", c_i32), ("IsBloom", c_i32), ("BloomThreshold", c_f), ("BloomMaxColor", c_f),
                ("BloomMinusLods", c_i32)]


def default_post_settings():
    """TonemapAndGammaCorrect.GpuSettings + Bloom.GpuSettings defaults (TonemapAndGammaCorrecter.cs:10-22, Bloom.cs:10-19,46)."""
    return IdkPtPostSettings(0.45, 1.06, 0.18, 1.0, 0.1, 1, 1, 1.5, 3.8, 3)


def default_settings():
    """PathTracer defaults: GpuSettings (PathTracer.cs:127-138), RayDepth 7 (:211), SamplesPerPixel 1 (:12)."""
    s = IdkPtSettings()
    s.Gpu.FocalLength = 8.0
    s.Gpu.LenseRadius = 0.0
    s.Gpu.DoDebugBVHTraversal = 0
    s.Gpu.DoTraceLights = 0
    s.Gpu.DoRussianRoulette = 1
    s.RayDepth = 7
    s.SamplesPerPixel = 1
    s.DoRaySorting = 0
    s.OutputAOVs = 0
    s.CollectStats = 0
    return s


def scene_desc(scene):
    """IdkPtSceneDesc borrowing the numpy arrays of a host.Scene. Returns (desc, keepalive)."""
    keep = []

    def ptr(a):
        a = np.ascontiguousarray(a)
        keep.append(a)
        return a.ctypes.data if len(a) else None

    d = IdkPtSceneDesc()
    d.BlasNodes, d.BlasNodeCount = ptr(scene.blas_nodes), len(scene.blas_nodes)
    d.BlasTriangles, d.BlasTriangleCount = ptr(scene.blas_triangles), len(scene.blas_triangles)
    d.BlasDescs, d.BlasDescCount = ptr(scene.blas_descs), len(scene.blas_descs)
    d.BlasInstances, d.BlasInstanceCount = ptr(scene.blas_instances), len(scene.blas_instances)
    d.TlasNodes, d.TlasNodeCount = ptr(scene.tlas_nodes), len(scene.tlas_nodes)
    d.MeshTransforms, d.MeshTransformCount = ptr(scene.mesh_transforms), len(scene.mesh_transforms)
    d.Meshes, d.MeshCount = ptr(scene.meshes), len(scene.meshes)
    d.Materials, d.MaterialCount = ptr(scene.materials), len(scene.materials)
    d.Vertices, d.VertexCount = ptr(scene.vertices), len(scene.vertices)
    d.VertexPositions, d.VertexPositionCount = ptr(scene.positions), len(scene.positions)
    d.Lights, d.LightCount = ptr(scene.lights), len(scene.lights)
    d.UseTlas = int(scene.use_tlas)
    d.BlasStackSize = int(scene.blas_stack_size)
    textures = getattr(scene, "textures", [])
    if textures:
        arr, tkeep = texture_descs(textures)
        keep.extend(tkeep)
        d.Textures, d.TextureCount = ctypes.addressof(arr), len(textures)
    return d, keep


def texture_descs(textures):
    """IdkPtTextureDesc array for a list of texture dicts (host.Scene.textures). Returns (array, keepalive).
      uncompressed RGBA8:  dict(pixels [H, W, 4] uint8, srgb, wrap_s, wrap_t)
      any other format:    dict(format=IDKPT_TEX_*, width, height, data=<level-0 bytes: block stream or float texels>, wrap_s, wrap_t, flags)"""
    keep = []
    arr = (IdkPtTextureDesc * max(len(textures), 1))()
    for i, t in enumerate(textures):
        if "format" in t:
            data = np.ascontiguousarray(t["data"])
            keep.append(data)
            arr[i] = IdkPtTextureDesc(data.ctypes.data, int(t["width"]), int(t["height"]), int(t["format"]),
                                      t.get("wrap_s", GL_REPEAT), t.get("wrap_t", GL_REPEAT), int(t.get("flags", 0)))
            continue
        px = np.ascontiguousarray(t["pixels"], np.uint8)
        keep.append(px)
        arr[i] = IdkPtTextureDesc(px.ctypes.data, px.shape[1], px.shape[0], IDKPT_TEX_RGBA8_SRGB if t.get("srgb") else IDKPT_TEX_RGBA8_UNORM,
                                  t.get("wrap_s", GL_REPEAT), t.get("wrap_t", GL_REPEAT), int(t.get("flags", 0)))
    keep.append(arr)
    return arr, keep


def sky_desc(color=(0.6, 0.7, 0.9), faces=None):
    """Constant sky colour, or a cubemap: faces = float32 array [6, N, N, 4] (+X,-X,+Y,-Y,+Z,-Z)."""
    s = IdkPtSkyDesc()
    if isinstance(color, np.ndarray) and color.ndim == 4:
        faces, color = color, (0.0, 0.0, 0.0)
    s.Color[0], s.Color[1], s.Color[2] = color
    s.FaceSize = 0
    if faces is not None:
        faces = np.ascontiguousarray(faces, np.float32)
        assert faces.ndim == 4 and faces.shape[0] == 6 and faces.shape[1] == faces.shape[2] and faces.shape[3] == 4
        s.FaceSize = faces.shape[1]
        for i in range(6):
            s.Faces[i] = faces[i].ctypes.data
        s._keep = faces
    return s


_lib = None


def load(path=None):
    """dlopen libidkpt.so and declare signatures. Fails loudly if the library is missing: there is no fallback."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    path = path or os.environ.get("IDKPT_LIB") or _build.LIBIDKPT     # IDKPT_LIB: an experiment build (scripts/variant_probe.py)
    if not os.path.exists(path):
        raise RuntimeError(f"{path} is missing: build it with `python -m idkengine_b200.build` "
                           "(libidkpt has no CPU fallback)")
    L = ctypes.CDLL(path)
    P = ctypes.POINTER
    L.idkpt_create.restype = c_i32
    L.idkpt_create.argtypes = [P(IdkPtCreateInfo), P(c_vp)]
    L.idkpt_destroy.restype = None
    L.idkpt_destroy.argtypes = [c_vp]
    L.idkpt_last_error.restype = ctypes.c_char_p
    L.idkpt_last_error.argtypes = [c_vp]
    L.idkpt_set_scene.restype = c_i32
    L.idkpt_set_scene.argtypes = [c_vp, P(IdkPtSceneDesc)]
    L.idkpt_update_range.restype = c_i32
    L.idkpt_update_range.argtypes = [c_vp, c_i32, c_u64, c_u64, c_vp]
    L.idkpt_set_sky.restype = c_i32
    L.idkpt_set_sky.argtypes = [c_vp, P(IdkPtSkyDesc)]
    L.idkpt_resize.restype = c_i32
    L.idkpt_resize.argtypes = [c_vp, c_i32, c_i32]
    L.idkpt_reset_accumulation.restype = c_i32
    L.idkpt_reset_accumulation.argtypes = [c_vp]
    L.idkpt_accumulated_samples.restype = c_u32
    L.idkpt_accumulated_samples.argtypes = [c_vp]
    L.idkpt_set_accumulated_samples.restype = c_i32
    L.idkpt_set_accumulated_samples.argtypes = [c_vp, c_u32]
    L.idkpt_compute.restype = c_i32
    L.idkpt_compute.argtypes = [c_vp, c_vp, P(IdkPtSettings), P(IdkPtStats)]
    L.idkpt_read_result.restype = c_i32
    L.idkpt_read_result.argtypes = [c_vp, c_i32, c_vp, c_u64]
    L.idkpt_write_result.restype = c_i32
    L.idkpt_write_result.argtypes = [c_vp, c_i32, c_vp, c_u64]
    L.idkpt_present_async.restype = c_i32
    L.idkpt_present_async.argtypes = [c_vp, c_i32, c_vp, c_u64]
    L.idkpt_present_wait.restype = c_i32
    L.idkpt_present_wait.argtypes = [c_vp]
    L.idkpt_register_host_buffer.restype = c_i32
    L.idkpt_register_host_buffer.argtypes = [c_vp, c_vp, c_u64]
    L.idkpt_unregister_host_buffer.restype = c_i32
    L.idkpt_unregister_host_buffer.argtypes = [c_vp, c_vp]
    L.idkpt_gather_export.restype = c_i32
    L.idkpt_gather_export.argtypes = [c_vp, c_vp, c_u64]
    L.idkpt_gather_import.restype = c_i32
    L.idkpt_gather_import.argtypes = [c_vp, c_i32, c_i32, c_vp, c_u64]
    L.idkpt_gather_connect.restype = c_i32
    L.idkpt_gather_connect.argtypes = [c_vp, c_i32]
    L.idkpt_gather_device_ptr.restype = c_i32
    L.idkpt_gather_device_ptr.argtypes = [c_vp, P(c_vp), P(c_u64)]
    L.idkpt_result_device_ptr.restype = c_i32
    L.idkpt_result_device_ptr.argtypes = [c_vp, c_i32, P(c_vp), P(c_u64)]
    L.idkpt_tile_rows.restype = c_i32
    L.idkpt_tile_rows.argtypes = [c_vp, P(c_i32), c_vp, c_i32]
    L.idkpt_read_wavefront_rays.restype = c_i32
    L.idkpt_read_wavefront_rays.argtypes = [c_vp, c_vp, c_u64]
    L.idkpt_trace_rays.restype = c_i32
    L.idkpt_trace_rays.argtypes = [c_vp, c_vp, c_u64, c_i32, c_vp, P(c_f)]
    L.idkpt_trace_rays_any.restype = c_i32
    L.idkpt_trace_rays_any.argtypes = [c_vp, c_vp, c_u64, c_i32, c_vp, P(c_f)]
    L.idkpt_shadows_ray_traced.restype = c_i32
    L.idkpt_shadows_ray_traced.argtypes = [c_vp, c_vp, c_vp, c_vp, c_i32, c_i32, c_i32, c_i32, c_u32, c_vp, c_vp, P(c_f)]
    L.idkpt_set_skinning_data.restype = c_i32
    L.idkpt_set_skinning_data.argtypes = [c_vp, c_vp, c_u64]
    L.idkpt_skin_vertices.restype = c_i32
    L.idkpt_skin_vertices.argtypes = [c_vp, c_vp, c_u64, c_vp, c_u32, P(c_f)]
    L.idkpt_blas_refit.restype = c_i32
    L.idkpt_blas_refit.argtypes = [c_vp, c_u32, c_u32, P(c_f)]
    L.idkpt_read_range.restype = c_i32
    L.idkpt_read_range.argtypes = [c_vp, c_i32, c_u64, c_u64, c_vp]
    L.idkpt_post_process.restype = c_i32
    L.idkpt_post_process.argtypes = [c_vp, P(IdkPtPostSettings), c_i32, c_vp, P(c_f)]
    L.idkpt_ldr_device_ptr.restype = c_i32
    L.idkpt_ldr_device_ptr.argtypes = [c_vp, P(c_vp), P(c_u64)]
    L.idkpt_stream_handle.restype = c_i32
    L.idkpt_stream_handle.argtypes = [c_vp, P(c_vp)]
    L.idkpt_set_textures.restype = c_i32
    L.idkpt_set_textures.argtypes = [c_vp, c_vp, c_u64]
    L.idkpt_sync.restype = c_i32
    L.idkpt_sync.argtypes = [c_vp]
    L.idkpt_tlas_build.restype = c_i32
    L.idkpt_tlas_build.argtypes = [c_vp, c_i32, P(c_f)]
    L.idkpt_denoise.restype = c_i32
    L.idkpt_denoise.argtypes = [c_vp, P(IdkPtDenoiseSettings), P(c_f)]
    L.idkpt_denoise_device_ptrs.restype = c_i32
    L.idkpt_denoise_device_ptrs.argtypes = [c_vp, P(c_vp), P(c_vp), P(c_vp), P(c_vp), P(c_u64)]
    L.idkpt_denoise_import_output.restype = c_i32
    L.idkpt_denoise_import_output.argtypes = [c_vp]
    L.idkpt_blas_default_build_settings.restype = None
    L.idkpt_blas_default_build_settings.argtypes = [P(IdkPtBlasBuildSettings)]
    L.idkpt_blas_build.restype = c_i32
    L.idkpt_blas_build.argtypes = [c_vp, c_vp, c_u64, c_vp, c_u64, c_vp, c_u32, P(IdkPtBlasBuildSettings), c_vp, P(c_f)]
    L.idkpt_blas_build_read.restype = c_i32
    L.idkpt_blas_build_read.argtypes = [c_vp, c_u32, c_vp, c_vp]
    L.idkpt_blas_build_phase_ms.restype = c_i32
    L.idkpt_blas_build_phase_ms.argtypes = [c_vp, P(c_f), c_i32]
    L.idkpt_abi_version.restype = c_u32
    L.idkpt_abi_version.argtypes = []
    if path == _build.LIBIDKPT:
        _lib = L
    return L
