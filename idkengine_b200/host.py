"""Host side of the drop-in boundary: what the C# engine does *before* it calls the
path tracer, mirrored in Python/C++ because this image has no .NET.

  build_blas()   -> libidkhost.so, the C++ mirror of BLAS.Build + PreSplitting
                    (SRC/Bvh/BLAS.cs, SRC/Bvh/PreSplitting.cs)
  Scene          -> the global arrays ModelManager/BVH keep and upload
                    (SRC/ModelManager.cs:128-213, SRC/Bvh/BVH.cs:236-276,300-451)
  make_per_frame_data() -> GpuPerFrameData as Application.OnRender fills it
                    (SRC/Application.cs:144-159, SRC/Camera.cs:187-200)
"""
import ctypes
import os
import numpy as np

from . import gpu_types as gt
from . import build as _build


class IdkBlasBuildSettings(ctypes.Structure):
    _fields_ = [
        ("StopSplittingThreshold", ctypes.c_int32),
        ("MaxLeafTriangleCount", ctypes.c_int32),
        ("TriangleCost", ctypes.c_float),
        ("StackOptThreshold", ctypes.c_int32),
        ("StackOptSahIncreaseAcceptance", ctypes.c_float),
        ("SplitFactor", ctypes.c_float),
        ("DoPreSplit", ctypes.c_int32),
        ("Threads", ctypes.c_int32),
    ]


_lib = None


def lib():
    global _lib
    if _lib is None:
        path = _build.LIBIDKHOST
        if not os.path.exists(path):
            path = _build.build_host()
        L = ctypes.CDLL(path)
        L.idkhost_blas_build.restype = ctypes.c_void_p
        L.idkhost_blas_build.argtypes = [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_uint64,
                                         ctypes.POINTER(IdkBlasBuildSettings)]
        L.idkhost_blas_node_count.restype = ctypes.c_uint64
        L.idkhost_blas_node_count.argtypes = [ctypes.c_void_p]
        L.idkhost_blas_triangle_count.restype = ctypes.c_uint64
        L.idkhost_blas_triangle_count.argtypes = [ctypes.c_void_p]
        L.idkhost_blas_required_stack_size.restype = ctypes.c_int32
        L.idkhost_blas_required_stack_size.argtypes = [ctypes.c_void_p]
        L.idkhost_blas_fragment_count.restype = ctypes.c_int32
        L.idkhost_blas_fragment_count.argtypes = [ctypes.c_void_p]
        L.idkhost_blas_sah.restype = ctypes.c_double
        L.idkhost_blas_sah.argtypes = [ctypes.c_void_p]
        L.idkhost_blas_copy.restype = None
        L.idkhost_blas_copy.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
        L.idkhost_blas_free.restype = None
        L.idkhost_blas_free.argtypes = [ctypes.c_void_p]
        L.idkhost_hash64.restype = ctypes.c_uint64
        L.idkhost_hash64.argtypes = [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint64]
        L.idkhost_cache_save.restype = ctypes.c_int32
        L.idkhost_cache_save.argtypes = [ctypes.c_char_p, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_uint32]
        L.idkhost_cache_open.restype = ctypes.c_int32
        L.idkhost_cache_open.argtypes = [ctypes.c_char_p, ctypes.c_uint64, ctypes.POINTER(ctypes.c_void_p)]
        L.idkhost_cache_array.restype = ctypes.c_void_p
        L.idkhost_cache_array.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.POINTER(ctypes.c_uint32), ctypes.POINTER(ctypes.c_uint64)]
        L.idkhost_cache_close.restype = None
        L.idkhost_cache_close.argtypes = [ctypes.c_void_p]
        L.idkhost_transform_box.restype = None
        L.idkhost_transform_box.argtypes = [ctypes.c_void_p] * 5
        L.idkhost_tlas_build.restype = None
        L.idkhost_tlas_build.argtypes = [ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p, ctypes.c_int32]
        L.idkhost_default_build_settings.restype = None
        L.idkhost_default_build_settings.argtypes = [ctypes.POINTER(IdkBlasBuildSettings)]
        _lib = L
    return _lib


def default_build_settings():
    s = IdkBlasBuildSettings()
    lib().idkhost_default_build_settings(ctypes.byref(s))
    return s


def build_blas(positions, triangles, presplit=True, threads=None, settings=None):
    """positions: PackedVec3[V] (global array), triangles: GpuBlasTriangle[T] with global vertex ids.
    Returns dict(nodes, triangles, required_stack_size, fragment_count, sah)."""
    L = lib()
    s = settings or default_build_settings()
    s.DoPreSplit = 1 if presplit else 0
    s.Threads = threads if threads is not None else min(os.cpu_count() or 1, 32)
    positions = np.ascontiguousarray(positions)
    triangles = np.ascontiguousarray(triangles)
    assert positions.dtype == gt.PackedVec3 and triangles.dtype == gt.GpuBlasTriangle
    h = L.idkhost_blas_build(positions.ctypes.data, len(positions), triangles.ctypes.data, len(triangles), ctypes.byref(s))
    try:
        nodes = np.zeros(L.idkhost_blas_node_count(h), gt.GpuBlasNode)
        tris = np.zeros(L.idkhost_blas_triangle_count(h), gt.GpuBlasTriangle)
        L.idkhost_blas_copy(h, nodes.ctypes.data, tris.ctypes.data)
        return dict(nodes=nodes, triangles=tris,
                    required_stack_size=int(L.idkhost_blas_required_stack_size(h)),
                    fragment_count=int(L.idkhost_blas_fragment_count(h)),
                    sah=float(L.idkhost_blas_sah(h)))
    finally:
        L.idkhost_blas_free(h)


# --------------------------------------------------------------------------- on-disk BLAS cache (include/idkhost_cache.h)
BUILDER_VERSION = 1          # bump when host_mirror/bvh_build.cpp changes its output
CACHE_BLAS_NODES, CACHE_BLAS_TRIANGLES, CACHE_BUILD_INFO = 1, 2, 100
CACHE_OK, CACHE_ERR_IO, CACHE_ERR_FORMAT, CACHE_ERR_KEY, CACHE_ERR_CHECKSUM = 0, -1, -2, -3, -4


class IdkHostCacheArray(ctypes.Structure):
    _fields_ = [("Id", ctypes.c_uint32), ("ElemSize", ctypes.c_uint32), ("Count", ctypes.c_uint64), ("Data", ctypes.c_void_p)]


def hash64(arr, seed=0):
    arr = np.ascontiguousarray(arr)
    return int(lib().idkhost_hash64(arr.ctypes.data, arr.nbytes, seed))


def blas_source_key(model_positions, model_indices, tri_mesh, presplit, settings=None):
    """Hash of everything the builder's output depends on (not the thread count: the build is deterministic)."""
    s = settings or default_build_settings()
    blob = np.array([BUILDER_VERSION, s.StopSplittingThreshold, s.MaxLeafTriangleCount, s.StackOptThreshold, 1 if presplit else 0], np.int64)
    fl = np.array([s.TriangleCost, s.StackOptSahIncreaseAcceptance, s.SplitFactor], np.float32)
    h = hash64(blob)
    h = hash64(fl, h)
    h = hash64(np.ascontiguousarray(model_positions, np.float32), h)
    h = hash64(np.ascontiguousarray(model_indices, np.uint32), h)
    return hash64(np.ascontiguousarray(tri_mesh, np.int32), h)


def cache_save(path, key, b):
    """b: build_blas result with BLAS-local triangle vertex ids (relative to the model's first vertex) and mesh ids."""
    info = np.array([b["required_stack_size"], b["fragment_count"]], np.float64)
    info = np.concatenate([info, [b["sah"]]])
    keep = [np.ascontiguousarray(b["nodes"]), np.ascontiguousarray(b["triangles"]), info]
    arr = (IdkHostCacheArray * 3)(
        IdkHostCacheArray(CACHE_BLAS_NODES, 32, len(keep[0]), keep[0].ctypes.data),
        IdkHostCacheArray(CACHE_BLAS_TRIANGLES, 16, len(keep[1]), keep[1].ctypes.data),
        IdkHostCacheArray(CACHE_BUILD_INFO, 8, len(info), info.ctypes.data))
    return int(lib().idkhost_cache_save(os.fsencode(path), key, ctypes.addressof(arr), 3))


def cache_load(path, key):
    """Returns (rc, build-result dict or None); the arrays are copied out of the mapping."""
    L = lib()
    view = ctypes.c_void_p()
    rc = int(L.idkhost_cache_open(os.fsencode(path), key, ctypes.byref(view)))
    if rc != CACHE_OK:
        return rc, None
    try:
        def get(aid, dtype):
            es, n = ctypes.c_uint32(), ctypes.c_uint64()
            p = L.idkhost_cache_array(view, aid, ctypes.byref(es), ctypes.byref(n))
            if not p or es.value != np.dtype(dtype).itemsize:
                return None
            return np.frombuffer((ctypes.c_char * (n.value * es.value)).from_address(p), dtype=dtype).copy() if n.value else np.zeros(0, dtype)
        nodes, tris, info = get(CACHE_BLAS_NODES, gt.GpuBlasNode), get(CACHE_BLAS_TRIANGLES, gt.GpuBlasTriangle), get(CACHE_BUILD_INFO, np.float64)
        if nodes is None or tris is None or info is None or len(info) != 3:
            return CACHE_ERR_FORMAT, None
        return CACHE_OK, dict(nodes=nodes, triangles=tris, required_stack_size=int(info[0]), fragment_count=int(info[1]), sah=float(info[2]))
    finally:
        L.idkhost_cache_close(view)


# --------------------------------------------------------------------------- transforms
def trs_matrix(scale=1.0, rotation_deg_y=0.0, translation=(0.0, 0.0, 0.0)):
    """Column-vector 4x4 model matrix: T * Ry * S (the subset of `Transformation` the reference scene uses,
    SRC/Application.cs:448-471)."""
    s = np.diag([scale, scale, scale, 1.0]) if np.isscalar(scale) else np.diag(list(scale) + [1.0])
    a = np.deg2rad(rotation_deg_y)
    r = np.array([[np.cos(a), 0, np.sin(a), 0], [0, 1, 0, 0], [-np.sin(a), 0, np.cos(a), 0], [0, 0, 0, 1.0]])
    t = np.eye(4)
    t[:3, 3] = translation
    return t @ r @ s


def mesh_transform(model4x4):
    """GpuMeshTransform from a column-vector model matrix: rows of the upper 3x4 block
    (= MyMath.Matrix4x4ToTranposed3x4 of OpenTK's row-vector matrix, SRC/Utils/MyMath.cs:317-329)."""
    m = np.asarray(model4x4, np.float64)
    out = np.zeros(1, gt.GpuMeshTransform)
    m32 = m.astype(np.float32)
    out["ModelMatrix"][0] = m32[:3, :]
    out["InvModelMatrix"][0] = np.linalg.inv(m32.astype(np.float64)).astype(np.float32)[:3, :]
    out["PrevModelMatrix"][0] = m32[:3, :]
    return out


# --------------------------------------------------------------------------- Scene
class Model:
    """One glTF-like model after ModelLoader + HoistMeshPrimitives: local-space vertex data, an index
    buffer, a per-triangle local mesh id, per-mesh GpuMesh records, materials and one model matrix."""

    def __init__(self, positions, indices, tri_mesh=None, normals=None, texcoords=None, tangents=None,
                 meshes=None, materials=None, model_matrix=None, refittable=False, name="model"):
        self.positions = np.ascontiguousarray(positions, np.float32).reshape(-1, 3)
        self.indices = np.ascontiguousarray(indices, np.uint32).reshape(-1, 3)
        self.tri_mesh = np.zeros(len(self.indices), np.int32) if tri_mesh is None else np.ascontiguousarray(tri_mesh, np.int32)
        self.normals = compute_vertex_normals(self.positions, self.indices) if normals is None else np.asarray(normals, np.float32)
        self.texcoords = np.zeros((len(self.positions), 2), np.float32) if texcoords is None else np.asarray(texcoords, np.float32)
        self.tangents = default_tangents(self.normals) if tangents is None else np.asarray(tangents, np.float32)
        self.meshes = gt.default_mesh(int(self.tri_mesh.max()) + 1 if len(self.tri_mesh) else 1) if meshes is None else meshes
        self.materials = gt.default_material(1) if materials is None else materials
        self.model_matrix = np.eye(4) if model_matrix is None else np.asarray(model_matrix, np.float64)
        self.refittable = refittable
        self.name = name


def compute_vertex_normals(positions, indices):
    p = positions.astype(np.float64)
    e1 = p[indices[:, 1]] - p[indices[:, 0]]
    e2 = p[indices[:, 2]] - p[indices[:, 0]]
    fn = np.cross(e1, e2)
    n = np.zeros_like(p)
    for k in range(3):
        np.add.at(n, indices[:, k], fn)
    ln = np.linalg.norm(n, axis=1, keepdims=True)
    n = np.where(ln > 1e-20, n / np.maximum(ln, 1e-20), np.array([0.0, 1.0, 0.0]))
    return n.astype(np.float32)


def default_tangents(normals):
    n = normals.astype(np.float64)
    up = np.where(np.abs(n[:, 2:3]) < 0.999, np.array([[0.0, 0.0, 1.0]]), np.array([[1.0, 0.0, 0.0]]))
    t = np.cross(up, n)
    t /= np.maximum(np.linalg.norm(t, axis=1, keepdims=True), 1e-20)
    return t.astype(np.float32)


class Scene:
    """The global arrays of ModelManager + BVH after Add(): exactly what the engine binds to SSBO 1-27."""

    def __init__(self):
        self.positions = np.zeros(0, gt.PackedVec3)
        self.vertices = np.zeros(0, gt.GpuVertex)
        self.meshes = np.zeros(0, gt.GpuMesh)
        self.materials = np.zeros(0, gt.GpuMaterial)
        self.mesh_transforms = np.zeros(0, gt.GpuMeshTransform)
        self.blas_nodes = np.zeros(0, gt.GpuBlasNode)
        self.blas_triangles = np.zeros(0, gt.GpuBlasTriangle)
        self.blas_descs = np.zeros(0, gt.GpuBlasDesc)
        self.blas_instances = np.zeros(0, gt.GpuBlasInstance)
        self.tlas_nodes = np.zeros(0, gt.GpuTlasNode)
        self.lights = np.zeros(0, gt.GpuLight)
        self.textures = []             # dict(pixels [H, W, 4] uint8, srgb, wrap_s, wrap_t); material handle k = textures[k - 1]
        self.use_tlas = 0
        self.blas_stack_size = 1
        self.source_triangle_count = 0
        self.build_info = []

    def add(self, *models, threads=None, cache_dir=None, builder=None):
        """ModelManager.Add (SRC/ModelManager.cs:128-213) + BVH.Add/BlasesBuild (SRC/Bvh/BVH.cs:236-276,300-451):
        one BLAS + one instance per model. cache_dir (or $IDKHOST_BVH_CACHE): directory of the on-disk BLAS cache.
        builder: a callable with build_blas's signature (default: build_blas, the host builder); when it has a `batch`
        attribute (PathTracer.BlasBuilder), every model of this call that the cache does not hold is built in one batch."""
        cache_dir = cache_dir or os.environ.get("IDKHOST_BVH_CACHE") or None
        pending = []
        for m in models:
            v_off = len(self.positions)
            mesh_off = len(self.meshes)
            mat_off = len(self.materials)

            pos = np.zeros(len(m.positions), gt.PackedVec3)
            pos["x"], pos["y"], pos["z"] = m.positions[:, 0], m.positions[:, 1], m.positions[:, 2]
            self.positions = np.concatenate([self.positions, pos])

            vtx = np.zeros(len(m.positions), gt.GpuVertex)
            vtx["TexCoord"] = m.texcoords
            vtx["Normal"] = gt.compress_sr11g11b10(m.normals)
            vtx["Tangent"] = gt.compress_sr11g11b10(m.tangents)
            self.vertices = np.concatenate([self.vertices, vtx])

            meshes = m.meshes.copy()
            meshes["MaterialId"] += mat_off
            self.meshes = np.concatenate([self.meshes, meshes])
            self.materials = np.concatenate([self.materials, m.materials])

            transform_id = len(self.mesh_transforms)
            self.mesh_transforms = np.concatenate([self.mesh_transforms, mesh_transform(m.model_matrix)])

            # BVH.Add: vertex-offset rebased indices + MeshId (BVH.cs:255-272)
            src = np.zeros(len(m.indices), gt.GpuBlasTriangle)
            src["X"] = m.indices[:, 0].astype(np.int64) + v_off
            src["Y"] = m.indices[:, 1].astype(np.int64) + v_off
            src["Z"] = m.indices[:, 2].astype(np.int64) + v_off
            src["MeshId"] = m.tri_mesh + mesh_off
            self.source_triangle_count += len(src)

            b = None
            key = cache_path = None
            if cache_dir is not None:     # skip the SweepSAH build when this exact model was built before
                key = blas_source_key(m.positions, m.indices, m.tri_mesh, not m.refittable)
                cache_path = os.path.join(cache_dir, f"{key:016x}.idkbvh")
                rc, b = cache_load(cache_path, key) if os.path.exists(cache_path) else (CACHE_ERR_IO, None)
                if b is not None:         # stored model-relative: rebase onto this scene's vertex / mesh offsets
                    for f in ("X", "Y", "Z"):
                        b["triangles"][f] += v_off
                    b["triangles"]["MeshId"] += mesh_off
                    b["from_cache"] = True
            pending.append(dict(m=m, src=src, b=b, key=key, cache_path=cache_path, v_off=v_off, mesh_off=mesh_off,
                                transform_id=transform_id))

        todo = [p for p in pending if p["b"] is None]
        if todo and builder is not None and getattr(builder, "batch", None) is not None:
            for p, b in zip(todo, builder.batch(self.positions, [(p["src"], not p["m"].refittable) for p in todo])):
                p["b"] = b
        for p in todo:
            if p["b"] is None:
                p["b"] = (builder or build_blas)(self.positions, p["src"], presplit=not p["m"].refittable, threads=threads)
            if p["cache_path"] is not None:
                b = p["b"]
                rel = dict(b)
                rel["triangles"] = b["triangles"].copy()
                for f in ("X", "Y", "Z"):
                    rel["triangles"][f] -= p["v_off"]
                rel["triangles"]["MeshId"] -= p["mesh_off"]
                os.makedirs(cache_dir, exist_ok=True)
                cache_save(p["cache_path"], p["key"], rel)

        for p in pending:
            m, b, src = p["m"], p["b"], p["src"]
            desc = np.zeros(1, gt.GpuBlasDesc)
            desc["NodeOffset"] = len(self.blas_nodes)
            desc["NodeCount"] = len(b["nodes"])
            desc["TriangleOffset"] = len(self.blas_triangles)
            desc["TriangleCount"] = len(b["triangles"])
            desc["RequiredStackSize"] = b["required_stack_size"]
            desc["IsRefittable"] = 1 if m.refittable else 0
            blas_id = len(self.blas_descs)
            self.blas_descs = np.concatenate([self.blas_descs, desc])
            self.blas_nodes = np.concatenate([self.blas_nodes, b["nodes"]])
            self.blas_triangles = np.concatenate([self.blas_triangles, b["triangles"]])
            inst = np.zeros(1, gt.GpuBlasInstance)
            inst["BlasId"] = blas_id
            inst["MeshTransformId"] = p["transform_id"]
            self.blas_instances = np.concatenate([self.blas_instances, inst])
            self.build_info.append(dict(name=m.name, source_triangles=len(src), fragments=b["fragment_count"],
                                        triangles=len(b["triangles"]), nodes=len(b["nodes"]),
                                        required_stack_size=b["required_stack_size"], sah=b["sah"], from_cache=bool(b.get("from_cache", False))))
        # BVH.UpdateBlasStackSize (BVH.cs:559-567)
        self.blas_stack_size = max(1, int(self.blas_descs["RequiredStackSize"].max())) if len(self.blas_descs) else 1
        return self

    def build_tlas(self, use=True, search_radius=15):
        """BVH.TlasBuild (SRC/Bvh/BVH.cs:278-298) + TLAS.Build (SRC/Bvh/TLAS.cs:28-141): world-space bounds of every BLAS
        instance (Box.Transformed of the BLAS root by its ModelMatrix), serial PLOC; sets BVH.GpuUseTlas."""
        n = len(self.blas_instances)
        boxes = np.zeros((n, 6), np.float32)
        L = lib()
        for i, inst in enumerate(self.blas_instances):
            root = self.blas_nodes[self.blas_descs[inst["BlasId"]]["NodeOffset"] + 1]
            mn = np.ascontiguousarray(root["Min"], np.float32)
            mx = np.ascontiguousarray(root["Max"], np.float32)
            m = np.ascontiguousarray(self.mesh_transforms[inst["MeshTransformId"]]["ModelMatrix"], np.float32)
            L.idkhost_transform_box(mn.ctypes.data, mx.ctypes.data, m.ctypes.data, boxes[i, :3].ctypes.data, boxes[i, 3:].ctypes.data)
        self.tlas_nodes = np.zeros(max(2 * n - 1, 0), gt.GpuTlasNode)
        if n:
            L.idkhost_tlas_build(boxes.ctypes.data, n, self.tlas_nodes.ctypes.data, search_radius)
        self.use_tlas = 1 if use else 0
        return self

    def add_texture(self, pixels, srgb=False, wrap_s=10497, wrap_t=10497):
        """Registers an RGBA8 image and returns the handle to store in a GpuMaterial texture slot (ModelLoader's bindless
        handle, ModelLoader.cs:985-1000; here an index into IdkPtSceneDesc.Textures, 0 = 1x1 white)."""
        pixels = np.ascontiguousarray(pixels, np.uint8)
        assert pixels.ndim == 3 and pixels.shape[2] == 4
        self.textures.append(dict(pixels=pixels, srgb=bool(srgb), wrap_s=int(wrap_s), wrap_t=int(wrap_t)))
        return len(self.textures)

    def add_texture_raw(self, fmt, width, height, data, wrap_s=10497, wrap_t=10497, flags=0):
        """Registers a texture in one of the other IdkPtTextureFormat formats: the level-0 BC7 / BC5 / BC4 block stream of a
        KTX2 image as the loader hands it to GL (ModelLoader.cs:954-968), or R / RG / RGBA float texels. Returns the handle."""
        self.textures.append(dict(format=int(fmt), width=int(width), height=int(height), data=np.ascontiguousarray(data),
                                  wrap_s=int(wrap_s), wrap_t=int(wrap_t), flags=int(flags)))
        return len(self.textures)

    def add_light(self, position, color, radius):
        """LightManager.AddLight (SRC/Render/LightManager.cs) -> GpuLight in UBO 2."""
        l = np.zeros(1, gt.GpuLight)
        l["Position"] = position
        l["PrevPosition"] = position
        l["Color"] = color
        l["Radius"] = radius
        l["PointShadowIndex"] = -1
        self.lights = np.concatenate([self.lights, l])
        return self

    def bvh_bytes(self):
        return self.blas_nodes.nbytes + self.blas_triangles.nbytes + self.positions.nbytes


# --------------------------------------------------------------------------- camera
def look_at(eye, target, up):
    """OpenTK Matrix4.LookAt, row-vector convention (returned as a 4x4 whose ROWS are OpenTK rows)."""
    eye, target, up = (np.asarray(v, np.float64) for v in (eye, target, up))
    z = eye - target
    z /= np.linalg.norm(z)
    x = np.cross(up, z)
    x /= np.linalg.norm(x)
    y = np.cross(z, x)
    y /= np.linalg.norm(y)
    m = np.eye(4)
    m[0, :3] = [x[0], y[0], z[0]]
    m[1, :3] = [x[1], y[1], z[1]]
    m[2, :3] = [x[2], y[2], z[2]]
    m[3, :3] = [-x.dot(eye), -y.dot(eye), -z.dot(eye)]
    return m


def perspective_zero_to_one(fov_y, aspect, near, far):
    """MyMath.CreatePerspectiveFieldOfViewDepthZeroToOne (SRC/Utils/MyMath.cs:180-188), row-vector convention."""
    m = np.zeros((4, 4))
    f = 1.0 / np.tan(fov_y * 0.5)
    m[0, 0] = f / aspect
    m[1, 1] = f
    m[2, 2] = far / (near - far)
    m[2, 3] = -1.0
    m[3, 2] = -(far * near) / (far - near)
    return m


def view_dir_from_angles(yaw_deg, pitch_deg):
    """Camera.ViewDir = MyMath.PolarToCartesian(yaw, pitch) (SRC/Camera.cs, SRC/Utils/MyMath.cs:168-178)."""
    az, el = np.deg2rad(yaw_deg), np.deg2rad(pitch_deg)
    st = np.sin(el)
    return np.array([st * np.cos(az), np.cos(el), st * np.sin(az)])


def make_per_frame_data(position, view_dir, width, height, fov_y_deg=102.0, near=0.1, far=250.0, up=(0.0, 1.0, 0.0)):
    """Application.OnRender's GpuPerFrameData fill (SRC/Application.cs:144-159). Matrices are stored in OpenTK's
    row-major order, which GLSL (std140, column-major) reads as the transposed, column-vector matrix."""
    position = np.asarray(position, np.float64)
    view = look_at(position, position + np.asarray(view_dir, np.float64), up)
    proj = perspective_zero_to_one(np.deg2rad(fov_y_deg), width / float(height), near, far)
    projview = view @ proj
    pf = np.zeros(1, gt.GpuPerFrameData)
    pf["ProjView"][0] = projview.astype(np.float32).reshape(-1)
    pf["View"][0] = view.astype(np.float32).reshape(-1)
    pf["InvView"][0] = np.linalg.inv(view).astype(np.float32).reshape(-1)
    pf["PrevView"][0] = pf["View"][0]
    pf["ViewPos"][0] = position.astype(np.float32)
    pf["Projection"][0] = proj.astype(np.float32).reshape(-1)
    pf["InvProjection"][0] = np.linalg.inv(proj).astype(np.float32).reshape(-1)
    pf["InvProjView"][0] = np.linalg.inv(projview).astype(np.float32).reshape(-1)
    pf["PrevProjView"][0] = pf["ProjView"][0]
    pf["NearPlane"] = near
    pf["FarPlane"] = far
    return pf
