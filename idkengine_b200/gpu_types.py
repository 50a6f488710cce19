"""numpy dtypes byte-identical to include/idk_gpu_types.h (and therefore to the
reference's SRC/GpuTypes/*.cs / SH/include/GpuTypes.glsl). tests/test_contract.py
checks every itemsize/offset against the C header through the compiled library."""
import numpy as np

f4, i4, u4, u8 = np.float32, np.int32, np.uint32, np.uint64

GpuBlasNode = np.dtype([("Min", f4, 3), ("TriStartOrChild", i4), ("Max", f4, 3), ("TriCount", i4)])
GpuBlasTriangle = np.dtype([("X", i4), ("Y", i4), ("Z", i4), ("MeshId", i4)])
GpuBlasDesc = np.dtype([
    ("NodeOffset", i4), ("NodeCount", i4), ("TriangleOffset", i4), ("TriangleCount", i4),
    ("LeafIndicesOffset", i4), ("LeafIndicesCount", i4), ("ParentIndicesOffset", i4), ("ParentIndicesCount", i4),
    ("RequiredStackSize", i4), ("IsRefittable", i4)])
GpuBlasInstance = np.dtype([("BlasId", u4), ("MeshTransformId", u4)])
GpuTlasNode = np.dtype([("Min", f4, 3), ("IsLeafAndChildOrInstanceId", u4), ("Max", f4, 3), ("_pad0", f4)])
GpuMeshTransform = np.dtype([("ModelMatrix", f4, (3, 4)), ("InvModelMatrix", f4, (3, 4)), ("PrevModelMatrix", f4, (3, 4))])
GpuMesh = np.dtype([
    ("LocalBoundsMin", f4, 3), ("MaterialId", i4), ("LocalBoundsMax", f4, 3), ("NormalMapStrength", f4),
    ("AbsorbanceBias", f4, 3), ("MeshletsOffset", i4), ("MeshletCount", i4), ("EmissiveBias", f4),
    ("SpecularBias", f4), ("RoughnessBias", f4), ("TransmissionBias", f4), ("IORBias", f4),
    ("InstanceCount", i4), ("VertexCount", i4), ("_pad0", f4, 3), ("TintOnTransmissive", i4)])
GpuMaterial = np.dtype([
    ("EmissiveFactor", f4, 3), ("BaseColorFactor", u4), ("Absorbance", f4, 3), ("IOR", f4),
    ("TransmissionFactor", f4), ("RoughnessFactor", f4), ("MetallicFactor", f4), ("AlphaCutoff", f4),
    ("BaseColorTexture", u8), ("MetallicRoughnessTexture", u8), ("NormalTexture", u8),
    ("EmissiveTexture", u8), ("TransmissionTexture", u8), ("IsVolumetric", i4), ("IsDoubleSided", i4)])
GpuVertex = np.dtype([("TexCoord", f4, 2), ("Tangent", u4), ("Normal", u4)])
PackedVec3 = np.dtype([("x", f4), ("y", f4), ("z", f4)])
GpuUnskinnedVertex = np.dtype([("JointIndices", u4, 4), ("JointWeights", f4, 4), ("Position", f4, 3), ("Tangent", u4), ("Normal", u4)])
IdkPtSkinningCmd = np.dtype([("InputVertexOffset", u4), ("OutputVertexOffset", u4), ("JointMatricesOffset", u4), ("VertexCount", u4)])
GpuLight = np.dtype([("Position", f4, 3), ("Radius", f4), ("Color", f4, 3), ("PointShadowIndex", i4),
                     ("PrevPosition", f4, 3), ("_pad0", f4)])
GpuPerFrameData = np.dtype([
    ("ProjView", f4, 16), ("View", f4, 16), ("InvView", f4, 16), ("PrevView", f4, 16),
    ("ViewPos", f4, 3), ("Frame", u4),
    ("Projection", f4, 16), ("InvProjection", f4, 16), ("InvProjView", f4, 16), ("PrevProjView", f4, 16),
    ("NearPlane", f4), ("FarPlane", f4), ("DeltaRenderTime", f4), ("Time", f4)])
GpuWavefrontRay = np.dtype([("Origin", f4, 3), ("PreviousIOROrTraverseCost", f4), ("Throughput", f4, 3),
                            ("PackedDirectionX", f4), ("Radiance", f4, 3), ("PackedDirectionY", f4)])
GpuAovRay = np.dtype([("Albedo", f4, 3), ("NewWeight", f4), ("Normal", f4, 3), ("_pad0", f4)])
IdkPtGpuSettings = np.dtype([("FocalLength", f4), ("LenseRadius", f4), ("DoDebugBVHTraversal", i4),
                             ("DoTraceLights", i4), ("DoRussianRoulette", i4)])
IdkPtRay = np.dtype([("Origin", f4, 3), ("TMax", f4), ("Direction", f4, 3), ("_pad0", f4)])
IdkPtHit = np.dtype([("BaryX", f4), ("BaryY", f4), ("T", f4), ("TriangleId", u4), ("MeshTransformId", u4),
                     ("NodePairFetches", u4), ("TriangleTests", u4), ("_pad0", u4)])
IdkPtBlasBuildSettings = np.dtype([("StopSplittingThreshold", i4), ("MaxLeafTriangleCount", i4), ("TriangleCost", f4),
                                   ("StackOptThreshold", i4), ("StackOptSahIncreaseAcceptance", f4), ("SplitFactor", f4),
                                   ("DoPreSplit", i4)])
IdkPtBlasBuildDesc = np.dtype([("TriangleOffset", u4), ("TriangleCount", u4), ("IsRefittable", i4), ("_pad0", i4)])
IdkPtBlasBuildInfo = np.dtype([("NodeCount", u4), ("TriangleCount", u4), ("FragmentCount", u4), ("RequiredStackSize", i4),
                               ("SahBits", u8)])

EXPECTED_SIZES = {
    "GpuBlasNode": 32, "GpuBlasTriangle": 16, "GpuBlasDesc": 40, "GpuBlasInstance": 8, "GpuTlasNode": 32,
    "GpuMeshTransform": 144, "GpuMesh": 96, "GpuMaterial": 96, "GpuVertex": 16, "PackedVec3": 12,
    "GpuLight": 48, "GpuPerFrameData": 544, "GpuWavefrontRay": 48, "GpuAovRay": 32, "IdkPtGpuSettings": 20,
    "IdkPtRay": 32, "IdkPtHit": 32, "GpuUnskinnedVertex": 52, "IdkPtSkinningCmd": 16,
    "IdkPtBlasBuildSettings": 28, "IdkPtBlasBuildDesc": 16, "IdkPtBlasBuildInfo": 24,
}
for _name, _size in EXPECTED_SIZES.items():
    assert globals()[_name].itemsize == _size, (_name, globals()[_name].itemsize, _size)


def default_mesh(n=1):
    """new GpuMesh() defaults (SRC/GpuTypes/GpuMesh.cs:27-31)."""
    m = np.zeros(n, GpuMesh)
    m["InstanceCount"] = 1
    m["TintOnTransmissive"] = 1
    return m


def pack_unorm4x8(rgba):
    """packUnorm4x8: R in the low byte."""
    v = np.clip(np.asarray(rgba, np.float64), 0.0, 1.0)
    b = np.rint(v * 255.0).astype(np.uint32)
    return np.uint32(b[..., 0] | (b[..., 1] << 8) | (b[..., 2] << 16) | (b[..., 3] << 24))


def default_material(n=1):
    """Material defaults as the loader produces them for a factor-only glTF material
    (SRC/Utils/ModelLoader.cs:458-460,853-867): white base colour, IOR 1.5, opaque."""
    m = np.zeros(n, GpuMaterial)
    m["BaseColorFactor"] = 0xFFFFFFFF
    m["IOR"] = 1.5
    m["RoughnessFactor"] = 1.0
    m["MetallicFactor"] = 0.0
    return m


def compress_sr11g11b10(v):
    """Compression.CompressSR11G11B10 (SRC/Utils/Compression.cs:21-40): snorm -> unorm 11/11/10.
    MathF.Round is round-half-even like np.rint."""
    v = np.asarray(v, np.float32) * np.float32(0.5) + np.float32(0.5)
    r = np.rint(v[..., 0] * np.float32(2047)).astype(np.uint32)
    g = np.rint(v[..., 1] * np.float32(2047)).astype(np.uint32)
    b = np.rint(v[..., 2] * np.float32(1023)).astype(np.uint32)
    return (b << np.uint32(22)) | (g << np.uint32(11)) | r
