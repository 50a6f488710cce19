"""Tiny run of every kernel family for compute-sanitizer (memcheck): no torch, small sizes."""
import os, sys
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests"))
import numpy as np
from idkengine_b200 import capi, scenes, vxgi, gpu_types as gt
from idkengine_b200.pathtracer import PathTracer

scene, cam = scenes.textured_room(threads=1)
scene.build_tlas(use=False)
w, h = 96, 64
frame = scenes.camera_frame(cam, w, h)
s = capi.default_settings()
s.RayDepth, s.OutputAOVs, s.DoRaySorting = 6, 1, 1
s.Gpu.DoTraceLights = 1
with PathTracer(w, h, s, lanes=3) as pt:
    pt.SetScene(scene); pt.SetSky((0.6, 0.7, 0.9)); pt.SetFrame(frame)
    pt.CollectStats = 1
    st = pt.Compute()
    pt.CollectStats = 0
    for _ in range(5):
        pt.ComputeAsync()
    pt.Sync()
    ldr, _ = pt.PostProcess()
    rng = np.random.default_rng(1)
    rays = np.zeros(3000, gt.IdkPtRay)
    rays["Origin"] = rng.uniform(-2.5, 2.5, (3000, 3)).astype(np.float32)
    d = rng.normal(size=(3000, 3)); rays["Direction"] = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
    rays["TMax"] = np.float32(3.4028235e38)
    pt.TraceRays(rays, trace_lights=True); pt.TraceRaysAny(rays, trace_lights=True)
    depth = np.full((h, w), 0.97, np.float32); nrg = np.full((h, w, 2), 0.5, np.float32)
    pt.ShadowsRayTraced(frame, depth, nrg, 0, samples=2)
    pt.SetTextures(scene.textures)
    pt.ComputeAsync(); pt.Sync()
    pt.SetSize(64, 40); pt.SetFrame(scenes.camera_frame(cam, 64, 40))
    pt.ComputeAsync(); pt.ComputeAsync(); pt.Sync()
print("path tracer ok", st.Rays)

scene2, cam2 = scenes.multi_blas(threads=1)
scene2.build_tlas()
with PathTracer(64, 48) as pt:
    pt.SetScene(scene2); pt.SetSky((0.6, 0.7, 0.9)); pt.SetFrame(scenes.camera_frame(cam2, 64, 48))
    pt.Compute()
    dsc = scene2.blas_descs[2]
    tris = scene2.blas_triangles[dsc["TriangleOffset"]:dsc["TriangleOffset"] + dsc["TriangleCount"]]
    idx = np.concatenate([tris["X"], tris["Y"], tris["Z"]]); v0, v1 = int(idx.min()), int(idx.max()) + 1
    u = np.zeros(v1 - v0, gt.GpuUnskinnedVertex)
    u["JointWeights"][:, 0] = 1.0
    for k, c in enumerate("xyz"): u["Position"][:, k] = scene2.positions[c][v0:v1]
    u["Normal"], u["Tangent"] = scene2.vertices["Normal"][v0:v1], scene2.vertices["Tangent"][v0:v1]
    jm = np.zeros((1, 3, 4), np.float32); jm[0, 0, 0] = jm[0, 1, 1] = jm[0, 2, 2] = 1.1
    cmd = np.zeros(1, gt.IdkPtSkinningCmd); cmd["OutputVertexOffset"], cmd["VertexCount"] = v0, v1 - v0
    pt.SetSkinningData(u); pt.SkinVertices(jm, cmd); pt.BlasRefit(0, 3)
    pt.Compute()
print("dynamic ok")

# device BLAS build: a pre-split and a refittable BLAS in one batch, a single-triangle BLAS, read back
with PathTracer(16, 16) as pt:
    rng = np.random.default_rng(6)
    pts = np.zeros(900, gt.PackedVec3)
    for c in "xyz": pts[c] = rng.uniform(-1, 1, 900).astype(np.float32)
    t = np.zeros(300, gt.GpuBlasTriangle); t["X"], t["Y"], t["Z"] = np.arange(0, 900, 3), np.arange(1, 900, 3), np.arange(2, 900, 3)
    pt.BuildBlases(pts, [(t[:200], True), (t[200:299], False), (t[299:], True)])
print("blas build ok")

# round 2 additions: TLAS walk inside k_traverse2 (async lanes), BC7 / BC5 / BC4 decode at upload, float textures, cube-map sky
# with seamless filtering, denoise hand-off, point-shadowed lights in the voxeliser
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests"))
import copy
import bcn_ref
scene3, cam3 = scenes.instance_grid(2, threads=1)
with PathTracer(80, 56, lanes=3) as pt:
    pt.SetScene(scene3); pt.SetFrame(scenes.camera_frame(cam3, 80, 56))
    rng = np.random.default_rng(3)
    pt.SetSky((0, 0, 0), rng.uniform(0, 2, (6, 8, 8, 4)).astype(np.float32))
    pt.Compute()
    for _ in range(3):
        pt.ComputeAsync()
    pt.Sync()
    pt.TlasBuild(15); pt.TlasBuild(2)
    pt.Compute()
print("tlas phase + cube sky + device tlas build ok")
comp = copy.copy(scene)
comp.textures = []
rng = np.random.default_rng(4)
for k, t in enumerate(scene.textures):
    px = t["pixels"]; hh, ww = px.shape[:2]
    nb = ((hh + 3) // 4) * ((ww + 3) // 4)
    common = dict(wrap_s=t["wrap_s"], wrap_t=t["wrap_t"])
    if k % 3 == 0:
        comp.textures.append(dict(format=capi.IDKPT_TEX_BC7_SRGB, width=ww, height=hh, data=rng.integers(0, 256, (nb, 16), dtype=np.uint8), **common))
    elif k % 3 == 1:
        comp.textures.append(dict(format=capi.IDKPT_TEX_BC5_RG_UNORM, width=ww, height=hh, data=rng.integers(0, 256, (nb, 16), dtype=np.uint8), **common))
    else:
        comp.textures.append(dict(format=capi.IDKPT_TEX_BC4_R_UNORM, width=ww, height=hh, data=rng.integers(0, 256, (nb, 8), dtype=np.uint8), flags=0, **common))
comp.textures[1] = dict(format=capi.IDKPT_TEX_RGBA32F, width=5, height=3, data=rng.uniform(0, 1, (3, 5, 4)).astype(np.float32), wrap_s=33071, wrap_t=33648, flags=1)
s2 = capi.default_settings(); s2.OutputAOVs = 1
with PathTracer(w, h, s2) as pt:
    pt.SetScene(comp); pt.SetSky((0.6, 0.7, 0.9)); pt.SetFrame(frame)
    pt.Compute(); pt.Compute()
    pt.Denoise()
    pt.PostProcess(source=capi.IDKPT_IMAGE_DENOISED)
    pt.DenoiseDevicePtrs(); pt.DenoiseImportOutput()
    shadowed = copy.copy(comp)
    shadowed.lights = comp.lights.copy(); shadowed.lights["PointShadowIndex"][:] = 0
    with vxgi.Voxelizer((20, 16, 24), (-3.1, -0.1, -3.1), (3.1, 4.1, 3.1)) as vx:
        vx.SetScene(shadowed); vx.SetShadowTracer(pt); vx.Render()
        vx.SetSlab(5, 17); vx.Render(); vx.LevelDevicePtr(0); vx.Mipmap(); vx.SetSlab(0, 24)
        f3 = scenes.camera_frame(cam, 40, 24)
        vx.ConeTraceRows(f3, np.full((8, 40), 0.95, np.float32), np.full((8, 40, 2), 0.5, np.float32), np.full((8, 40, 2), 0.5, np.float32), 24, 8)
print("bcn + denoise + point shadows + slabs ok")

with vxgi.Voxelizer((24, 20, 28), (-3.1, -0.1, -3.1), (3.1, 4.1, 3.1)) as vx:
    vx.SetScene(scene)
    vx.Render()
    f2 = scenes.camera_frame(cam, 48, 32)
    vx.ConeTrace(f2, np.full((32, 48), 0.95, np.float32), np.full((32, 48, 2), 0.5, np.float32), np.full((32, 48, 2), 0.5, np.float32), vxgi.default_cone_settings())
print("vxgi ok")
