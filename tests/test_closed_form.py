"""Closed-form scenes: the path tracer against answers that do not come from the oracle.

Every other light-transport test compares the CUDA path with oracle/oracle.cpp, a second restatement of the same shaders;
a mistake made in both passes them. The scenes here have exact answers that follow from a handful of shading rules of
k_shade (csrc/idk_kernels.cuh) and oracle.cpp's ShadeTraceRay:
  * every branch has pdf == 1 and multiplies the throughput by `bsdf`, which is the albedo in the diffuse branch, the
    metallic branch and the tinted transmissive branch;
  * emission is added as rad += Emissive * thr before that multiplication, at every hit up to RayDepth, the last included;
  * Russian roulette starts after the first hit; a constant sky is returned as is; untextured meshes have
    NormalMapStrength == 0.
Expected values are float64 functions of the material as stored (BaseColorFactor is unorm8: albedo = k / 255). They do
not depend on tiles, lanes, ray sorting, the traversal variant, treelets or the TLAS, so each case runs on the CPU oracle
and, marked `gpu`, through PathTracer; test_production_paths_hit_the_closed_form runs two of them through every
production configuration at 1920x1080.

Known imprecision. Vertex normals are stored as SR11G11B10: an axis-aligned normal decodes ~5e-4 rad off the geometric
one, so a cosine-sampled direction can dip under a plane and re-hit it. A pixel so affected carries exactly one extra
factor of the albedo. Such pixels are accepted only at that exact value and only up to OUTLIER_BOUND.
"""
import os

import numpy as np
import pytest

import oracle_lib as ol
from idkengine_b200 import capi, scenes
from idkengine_b200.host import Model, Scene, make_per_frame_data, trs_matrix


def _has_cuda():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


BACKENDS = ["cpu", pytest.param("gpu", marks=[pytest.mark.gpu, pytest.mark.skipif(not _has_cuda(), reason="no CUDA device")])]
SKY = (0.6, 0.7, 0.9)
ULP = 4                     # one- or two-product closed forms: a few float32 roundings
M32 = np.uint64(0xFFFFFFFF)


def OUTLIER_BOUND(n_pixels):
    """Most pixels with one extra bounce accepted in an image of n_pixels (the SR11G11B10 dip, ~1e-6 per path)."""
    return 4 + n_pixels // 10000


# ------------------------------------------------------------------------------------------------ rendering
def settings(depth, rr=False, spp=1, aovs=False, sorting=False):
    s = capi.default_settings()
    s.RayDepth, s.SamplesPerPixel, s.OutputAOVs, s.DoRaySorting = depth, spp, int(aovs), int(sorting)
    s.Gpu.DoRussianRoulette = int(rr)
    return s


def render(backend, scene, frame, s, w, h, sky=SKY, calls=1, tile=(8, 0, 1), lanes=0, env=None):
    """(result, albedo, normal) rgba32f [h, w, 4] after `calls` Compute()s; a tile renders only its own rows."""
    if backend == "cpu":
        res, alb, nrm = (np.zeros((h, w, 4), np.float32) for _ in range(3))
        acc = 0
        for _ in range(calls):
            acc = ol.path_trace(scene, frame, s, w, h, sky=sky, tile=tile, accumulated=acc, result=res, albedo=alb,
                                normal=nrm, want_rays=False).accumulated
        return res, alb, nrm
    from idkengine_b200.pathtracer import PathTracer
    old = {k: os.environ.get(k) for k in (env or {})}
    os.environ.update(env or {})
    try:
        with PathTracer(w, h, s, tile=tile, lanes=lanes) as pt:
            pt.SetScene(scene); pt.SetSky(sky); pt.SetFrame(frame)
            for _ in range(calls):
                if lanes:
                    pt.ComputeAsync()
                else:
                    pt.Compute()
            pt.Sync()
            return pt.Result, pt.AlbedoTexture, pt.NormalTexture
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def tile_rows(h, tile):
    return np.array([y for y in range(h) if (y // tile[0]) % tile[2] == tile[1]])


# ------------------------------------------------------------------------------------------------ float64 references
def _pcg(state):
    state = (state * np.uint64(747796405) + np.uint64(2891336453)) & M32
    word = (((state >> ((state >> np.uint64(28)) + np.uint64(4))) ^ state) * np.uint64(277803737)) & M32
    return state, (word >> np.uint64(22)) ^ word


def primary_rays(frame, w, h, accumulated=0):
    """Origin and float64 direction [h, w, 3] of every pixel's jittered camera ray of sample `accumulated` (FirstHit: the
    sub-pixel offset is the first two PCG draws of seed (y * 4096 + x) * (n + 1), pinhole lens)."""
    y, x = np.mgrid[0:h, 0:w].astype(np.uint64)
    st = ((y * np.uint64(4096) + x) * np.uint64(accumulated + 1)) & M32
    st, h0 = _pcg(st)
    st, h1 = _pcg(st)
    sx = (h0.astype(np.float32) / np.float32(4294967296.0)).astype(np.float64)
    sy = (h1.astype(np.float32) / np.float32(4294967296.0)).astype(np.float64)
    nx = (x + sx) / w * 2.0 - 1.0
    ny = (y + sy) / h * 2.0 - 1.0
    ip = frame["InvProjection"][0].astype(np.float64)
    iv = frame["InvView"][0].astype(np.float64)
    vx, vy = ip[0] * nx + ip[4] * ny, ip[1] * nx + ip[5] * ny
    d = np.stack([iv[i] * vx + iv[4 + i] * vy - iv[8 + i] for i in range(3)], -1)
    return frame["ViewPos"][0].astype(np.float64), d / np.linalg.norm(d, axis=-1, keepdims=True)


def albedo_of(mat):
    c = int(mat["BaseColorFactor"])
    return np.array([(c >> s) & 255 for s in (0, 8, 16, 24)], np.float64) / 255.0


def ulps(got, want):
    """|got - want| in float32 ulps of want (per element)."""
    want = np.asarray(want, np.float64)
    return np.abs(got.astype(np.float64) - want) / np.spacing(np.abs(want).astype(np.float32)).astype(np.float64)


def match(img, want, tol=ULP):
    """Pixels [h, w] whose rgb is within tol ulp of want ([3] or [h, w, 3]) in every channel."""
    return (ulps(img[..., :3], np.broadcast_to(want, img[..., :3].shape)) <= tol).all(-1)


def classify(img, main, extra, tol=ULP):
    """main / extra: lists of (value [3] or [h, w, 3], mask [h, w]) -- the values a pixel may take where its mask is set.
    Returns (bad, outliers): pixels matching no candidate, and pixels matching only an extra-bounce candidate."""
    ok_main = np.zeros(img.shape[:2], bool)
    for v, m in main:
        ok_main |= match(img, v, tol) & m
    ok_extra = np.zeros(img.shape[:2], bool)
    for v, m in extra:
        ok_extra |= match(img, v, tol) & m
    return ~(ok_main | ok_extra), ok_extra & ~ok_main


def assert_closed_form(img, main, extra, what, tol=ULP):
    bad, out = classify(img, main, extra, tol)
    n = img.shape[0] * img.shape[1]
    assert bad.sum() == 0, f"{what}: {int(bad.sum())} of {n} pixels off the closed form, e.g. {img[bad][:3, :3].tolist()}"
    assert out.sum() <= OUTLIER_BOUND(n), f"{what}: {int(out.sum())} one-extra-bounce pixels"
    print(f"[closed-form] {what}: {int(out.sum())} one-extra-bounce pixels of {n}")
    return out


# ------------------------------------------------------------------------------------------------ scene builders
def flat_polyhedron(corners, faces):
    """Convex polyhedron with unshared vertices per face (so vertex normals are face normals), faces wound outward.
    Returns (positions, indices)."""
    corners = np.asarray(corners, np.float64)
    c = corners.mean(0)
    pos, idx = [], []
    for f in faces:
        p = corners[list(f)]
        if np.dot(np.cross(p[1] - p[0], p[2] - p[0]), p[0] - c) < 0:
            p = p[::-1]
        base = len(pos)
        pos.extend(p)
        idx.extend([base, base + k, base + k + 1] for k in range(1, len(p) - 1))
    return np.array(pos, np.float32), np.array(idx, np.uint32)


def world_planes(corners, faces, model):
    """Outward planes (n [F, 3], d [F]) of the polyhedron placed by `model`, from world-space vertices in float64."""
    p = (np.c_[np.asarray(corners, np.float64), np.ones(len(corners))] @ np.asarray(model, np.float64).T)[:, :3]
    c = p.mean(0)
    ns, ds = [], []
    for f in faces:
        q = p[list(f)]
        n = np.cross(q[1] - q[0], q[2] - q[0])
        n /= np.linalg.norm(n)
        n = n if np.dot(n, q[0] - c) > 0 else -n
        ns.append(n)
        ds.append(np.dot(n, q[0]))
    return np.array(ns), np.array(ds)


def ray_hits_convex(o, d, planes, margin):
    """Does o + t d (t > 0) meet {x : n.x <= dist + margin} for every plane? d [..., 3]."""
    n, dist = planes
    nd = d @ n.T
    no = o @ n.T
    lim = dist + margin - no                              # n.(o + t d) <= dist + margin  <=>  t nd <= lim
    with np.errstate(divide="ignore", invalid="ignore"):
        t = lim / nd
    t_near = np.where(nd < 0, t, -np.inf).max(-1)
    t_far = np.where(nd > 0, t, np.inf).min(-1)
    parallel_out = ((nd == 0) & (lim < 0)).any(-1)
    return (t_near <= t_far) & (t_far > 0) & ~parallel_out


def single_material_model(pos, idx, spec, model_matrix=None, name="m"):
    meshes, mats = scenes._materials([spec])
    return Model(pos, idx, np.zeros(len(idx), np.int32), meshes=meshes, materials=mats, model_matrix=model_matrix, name=name)


def camera(position, target, w, h, fov=60.0, up=(0.0, 1.0, 0.0)):
    d = np.asarray(target, np.float64) - np.asarray(position, np.float64)
    return make_per_frame_data(position, d / np.linalg.norm(d), w, h, fov, up=up)


PLANE_L = 100.0                 # the quad fills the view and catches rays that dip under it


def plane_scene(spec, facing=True):
    """One quad z = 0 with geometric normal +z (facing the camera at z > 0) or -z (seen from behind)."""
    p = [[-PLANE_L, -PLANE_L, 0], [PLANE_L, -PLANE_L, 0], [PLANE_L, PLANE_L, 0], [-PLANE_L, PLANE_L, 0]]
    if not facing:
        p = p[::-1]
    pos, idx = scenes.quad(*p)
    scene = Scene().add(single_material_model(pos, idx, spec, name="plane"), threads=1)
    return scene, scene.materials[0]


def _rotation(axis, deg):
    a = np.asarray(axis, np.float64) / np.linalg.norm(axis)
    k = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
    t = np.deg2rad(deg)
    return np.eye(3) + np.sin(t) * k + (1 - np.cos(t)) * (k @ k)


BOX_FACES = [(0, 1, 3, 2), (4, 6, 7, 5), (0, 4, 5, 1), (2, 3, 7, 6), (0, 2, 6, 4), (1, 5, 7, 3)]
# a unit cube turned off the axes in its own frame: a non-uniform instance scale then bends its normals (M^-T n is not
# parallel to M n), which an axis-aligned cube would hide
TILTED_BOX = np.array([[sx, sy, sz] for sx in (-0.5, 0.5) for sy in (-0.5, 0.5) for sz in (-0.5, 0.5)]) @ _rotation((1.0, 2.0, 0.5), 35.0).T
# an inverted frustum (top 2x2 at y = 0.5, bottom 1x1 at y = 0): from high above only its top is visible, and every
# top sees nothing but sky, so instances of it cannot light each other
MESA = np.array([[-0.5, 0, -0.5], [0.5, 0, -0.5], [0.5, 0, 0.5], [-0.5, 0, 0.5], [-1, 0.5, -1], [1, 0.5, -1], [1, 0.5, 1], [-1, 0.5, 1]], np.float64)
MESA_FACES = [(4, 5, 6, 7), (0, 1, 2, 3), (0, 1, 5, 4), (1, 2, 6, 5), (2, 3, 7, 6), (3, 0, 4, 7)]
POLY_SPEC = dict(color=(0.8, 0.5, 0.3), emissive=(0.5, 0.25, 1.0))


def polyhedron_scene(kind):
    """(scene, per-frame data, list of world planes, material) for the convex-object case rendered three ways."""
    w, h = 160, 120
    if kind == "identity":
        pos, idx = flat_polyhedron(TILTED_BOX, BOX_FACES)
        models = [single_material_model(pos, idx, POLY_SPEC)]
        planes = [world_planes(TILTED_BOX, BOX_FACES, np.eye(4))]
        frame = camera((0.4, 0.9, 2.6), (0, 0, 0), w, h, 45.0)
    elif kind == "instance":
        pos, idx = flat_polyhedron(TILTED_BOX, BOX_FACES)
        m = trs_matrix((4.0, 1.0, 0.5), 30.0, (0.3, -0.2, 0.1))
        models = [single_material_model(pos, idx, POLY_SPEC, model_matrix=m)]
        planes = [world_planes(TILTED_BOX, BOX_FACES, m)]
        frame = camera((1.0, 2.0, 5.5), (0, 0, 0), w, h, 50.0)
    else:
        pos, idx = flat_polyhedron(MESA, MESA_FACES)
        models, planes = [], []
        for k, (x, z) in enumerate([(-4.5, -2.5), (0.0, -2.5), (4.5, -2.5), (-4.5, 2.5), (0.0, 2.5), (4.5, 2.5)]):
            m = trs_matrix((1.0 + 0.1 * k, 1.0, 1.5 - 0.1 * k), 23.0 * k, (x, 0.0, z))
            models.append(single_material_model(pos, idx, POLY_SPEC, model_matrix=m, name=f"mesa{k}"))
            planes.append(world_planes(MESA, MESA_FACES, m))
        frame = camera((0.3, 20.0, 0.2), (0, 0, 0), w, h, 40.0, up=(0.0, 0.0, -1.0))
    scene = Scene().add(*models, threads=1)
    if kind == "tlas":
        scene.build_tlas()
        assert scene.use_tlas == 1 and len(scene.blas_instances) == 6
    return scene, frame, planes, scene.materials[0], (w, h)


def polyhedron_expectation(frame, w, h, planes, mat, sky, rows=None):
    """(main candidates, extra-bounce candidates) of the convex-object images: E + rho c where the camera ray surely
    hits, c where it surely misses, either within 1e-4 of the silhouette."""
    o, d = primary_rays(frame, w, h)
    sure = np.zeros((h, w), bool)
    maybe = np.zeros((h, w), bool)
    for pl in planes:
        sure |= ray_hits_convex(o, d, pl, -1e-4)
        maybe |= ray_hits_convex(o, d, pl, 1e-4)
    rho, E, c = albedo_of(mat)[:3], np.asarray(mat["EmissiveFactor"], np.float64), np.asarray(sky, np.float64)
    hit_v, miss_v, extra_v = E + rho * c, c, E + rho * E + rho * rho * c
    if rows is not None:
        sure, maybe = sure[rows], maybe[rows]
    return [(hit_v, maybe), (miss_v, ~sure)], [(extra_v, maybe)], sure, maybe


BOX_HALF = 1.0


def closed_box_scene(color, emissive):
    """Six walls of a 2x2x2 room, each extended 0.5 past the others so the room has no seams; one diffuse material."""
    a, b = BOX_HALF, BOX_HALF + 0.5
    walls = []
    for axis in range(3):
        for side in (-a, a):
            u, v = [k for k in range(3) if k != axis]
            pts = []
            for su, sv in ((-b, -b), (b, -b), (b, b), (-b, b)):
                q = [0.0, 0.0, 0.0]
                q[axis], q[u], q[v] = side, su, sv
                pts.append(q)
            walls.append(scenes.quad(*pts))
    pos = np.concatenate([p for p, _ in walls])
    idx = np.concatenate([i + 4 * k for k, (_, i) in enumerate(walls)])
    scene = Scene().add(single_material_model(pos, idx, dict(color=color, emissive=emissive, roughness=0.6), name="room"), threads=1)
    return scene, scene.materials[0]


def closed_box_value(mat, depth):
    rho, E = albedo_of(mat)[:3], np.asarray(mat["EmissiveFactor"], np.float64)
    return E * sum(rho ** k for k in range(depth))


BOX_FRAME_ARGS = ((0.13, -0.21, 0.3), (0.9, 0.3, -1.0))     # camera inside the room, looking into a corner


def box_tol(depth):
    return ULP + 2 * depth                               # a product and a sum per bounce


# ================================================================================================ case 1: one plane
PLANE_MATERIALS = {
    "diffuse": dict(color=(0.8, 0.5, 0.2)),
    "diffuse_emissive": dict(color=(0.8, 0.5, 0.2), emissive=(2.0, 1.0, 0.5)),
    "metal_r0": dict(color=(0.9, 0.6, 0.3), metallic=1.0, roughness=0.0),
    "metal_r0.5": dict(color=(0.9, 0.6, 0.3), metallic=1.0, roughness=0.5),
    "metal_r1": dict(color=(0.9, 0.6, 0.3), metallic=1.0, roughness=1.0),
    "glass_r0_ior1.5": dict(color=(0.7, 0.9, 0.4), transmission=1.0, roughness=0.0, ior=1.5),
    "glass_r0.7_ior1.5": dict(color=(0.7, 0.9, 0.4), transmission=1.0, roughness=0.7, ior=1.5),
    "glass_r0_ior1.1": dict(color=(0.7, 0.9, 0.4), transmission=1.0, roughness=0.0, ior=1.1),
    "glass_r0.7_ior2.4": dict(color=(0.7, 0.9, 0.4), transmission=1.0, roughness=0.7, ior=2.4),
    "cutout": dict(color=(0.8, 0.5, 0.2, 0.3), cutoff=0.5),
}


def surface_variance(mat):
    """GetSurfaceVariance of the stored (un-squared) material: the first-hit AOV weight w."""
    m, t, r = (float(np.float32(mat[k])) for k in ("MetallicFactor", "TransmissionFactor", "RoughnessFactor"))
    return (1.0 - m - t) + m * r + t * r


PLANE_W, PLANE_H = 96, 72


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("name", list(PLANE_MATERIALS))
def test_plane_under_constant_sky(backend, name):
    """Every pixel = rho c (E + rho c when emissive; c when cut out); first-hit AOVs: albedo = rho w + (1 - w) c, and
    for the diffuse material the normal is the plane's."""
    scene, mat = plane_scene(PLANE_MATERIALS[name])
    w, h = PLANE_W, PLANE_H
    frame = camera((0.2, 0.1, 2.0), (0.0, 0.0, 0.0), w, h)
    img, alb, nrm = render(backend, scene, frame, settings(3, aovs=True), w, h)
    rho, E, c = albedo_of(mat)[:3], np.asarray(mat["EmissiveFactor"], np.float64), np.asarray(SKY)
    everywhere = np.ones((h, w), bool)
    if name == "cutout":
        assert_closed_form(img, [(c, everywhere)], [], f"{backend} plane {name}")
        return
    out = assert_closed_form(img, [(E + rho * c, everywhere)], [(E + rho * E + rho * rho * c, everywhere)], f"{backend} plane {name}")
    wgt = surface_variance(mat)
    ok = ~out
    assert match(alb, rho * wgt + (1.0 - wgt) * c)[ok].all(), np.abs(alb[ok][:, :3] - (rho * wgt + (1.0 - wgt) * c)).max()
    if name.startswith("diffuse"):
        assert np.abs(nrm[ok][:, :3] - [0.0, 0.0, 1.0]).max() <= 2.0 / 1023     # one SR11G11B10 step


@pytest.mark.parametrize("backend", BACKENDS)
def test_plane_russian_roulette_starts_after_the_first_hit(backend):
    """With roulette on, a path that leaves the plane for the sky never meets it: the image equals the roulette-free one
    wherever the path took no extra bounce."""
    scene, mat = plane_scene(PLANE_MATERIALS["diffuse"])
    w, h = PLANE_W, PLANE_H
    frame = camera((0.2, 0.1, 2.0), (0.0, 0.0, 0.0), w, h)
    off, _, _ = render(backend, scene, frame, settings(3), w, h)
    on, _, _ = render(backend, scene, frame, settings(3, rr=True), w, h)
    rho, c = albedo_of(mat)[:3], np.asarray(SKY)
    ok = match(off, rho * c)
    assert ok.mean() > 0.99 and np.array_equal(on[ok], off[ok])


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("ior", [1.1, 1.5, 2.4])
def test_plane_back_facing_transmission(backend, ior):
    """A tinted, non-volumetric transmissive plane seen from behind: fromInside is true, so the transmitted path is
    untinted (bsdf = 1, pixel = c) and the first hit takes prevIor = IOR, which makes f0 = 0 and F = (1 - cos)^5 for the
    Fresnel reflection (bsdf = rho, pixel = rho c). Every pixel is one of the two; the share of reflected pixels is the
    mean of F within 5 standard deviations."""
    scene, mat = plane_scene(dict(color=(0.7, 0.9, 0.4), transmission=1.0, roughness=0.0, ior=ior), facing=False)
    w, h = PLANE_W, PLANE_H
    frame = camera((0.0, -1.0, 1.0), (0.0, 0.3, 0.0), w, h, 70.0)
    img, _, _ = render(backend, scene, frame, settings(3), w, h)
    rho, c = albedo_of(mat)[:3], np.asarray(SKY)
    everywhere = np.ones((h, w), bool)
    assert_closed_form(img, [(c, everywhere), (rho * c, everywhere)], [(rho * rho * c, everywhere)], f"{backend} back-facing ior {ior}")
    _, d = primary_rays(frame, w, h)
    F = (1.0 - (-d[..., 2])) ** 5
    reflected = match(img, rho * c) & ~match(img, c)
    n = w * h
    assert abs(reflected.mean() - F.mean()) <= 5.0 * np.sqrt((F * (1 - F)).sum()) / n + 1.0 / n


# ================================================================================================ case 2: convex object
@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("kind", ["identity", "instance", "tlas"])
def test_convex_polyhedron_under_constant_sky(backend, kind):
    """Flat-shaded convex object, diffuse with emission: hit pixels = E + rho c, missed pixels = c. A wrong normal
    transform (the non-uniformly scaled instance) sends bounce rays back into the object: E + rho E + rho^2 c."""
    scene, frame, planes, mat, (w, h) = polyhedron_scene(kind)
    img, _, _ = render(backend, scene, frame, settings(3), w, h)
    main, extra, sure, maybe = polyhedron_expectation(frame, w, h, planes, mat, SKY)
    assert sure.mean() > 0.1 and (~maybe).mean() > 0.1 and (maybe & ~sure).mean() < 0.01
    assert_closed_form(img, main, extra, f"{backend} polyhedron {kind}")


# ================================================================================================ case 3: closed room
ROOM_ALBEDOS = {"white": (1.0, 1.0, 1.0), "tinted": (0.8, 0.5, 0.3)}


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("albedo", list(ROOM_ALBEDOS))
@pytest.mark.parametrize("depth", [1, 2, 5, 9])
def test_closed_room_geometric_series(backend, albedo, depth):
    """Camera inside a seamless room, every wall diffuse with albedo rho and emission E, black sky, no roulette: every
    pixel = E (1 - rho^D) / (1 - rho) (E D for white). Rendering again under a bright sky changes no pixel: no path
    leaves the room."""
    scene, mat = closed_box_scene(ROOM_ALBEDOS[albedo], (0.7, 1.3, 0.4))
    w, h = 64, 48
    frame = camera(BOX_FRAME_ARGS[0], np.add(*BOX_FRAME_ARGS), w, h, 90.0)
    s = settings(depth)
    img, _, _ = render(backend, scene, frame, s, w, h, sky=(0.0, 0.0, 0.0))
    want = closed_box_value(mat, depth)
    err = ulps(img[..., :3], want)
    assert err.max() <= box_tol(depth), (err.max(), img[..., :3].reshape(-1, 3)[err.max(-1).reshape(-1).argmax()], want)
    sentinel, _, _ = render(backend, scene, frame, s, w, h, sky=(1.0e4, 2.0e4, 3.0e4))
    leaks = int((sentinel != img).any(-1).sum())
    assert leaks == 0, f"{leaks} paths left the room"


@pytest.mark.parametrize("backend", BACKENDS)
def test_accumulating_identical_samples(backend):
    """64 samples of a pixel whose every sample is identical (the roulette-free room) stay within 4 ulp of that value:
    the running mean mix(last, new, 1 / (n + 1)) does not drift."""
    scene, mat = closed_box_scene(ROOM_ALBEDOS["tinted"], (0.7, 1.3, 0.4))
    w, h = 32, 24
    frame = camera(BOX_FRAME_ARGS[0], np.add(*BOX_FRAME_ARGS), w, h, 90.0)
    one, _, _ = render(backend, scene, frame, settings(5), w, h, sky=(0.0, 0.0, 0.0))
    many, _, _ = render(backend, scene, frame, settings(5, spp=16), w, h, sky=(0.0, 0.0, 0.0), calls=4)
    assert ulps(one[..., :3], closed_box_value(mat, 5)).max() <= box_tol(5)
    drift = ulps(many[..., :3], one[..., :3].astype(np.float64))
    print(f"[closed-form] {backend} accumulation of 64 identical samples: max drift {drift.max():.0f} ulp")
    assert drift.max() <= 4


# ================================================================================================ statistical cases
def assert_unbiased(samples, expected, what):
    """Image mean vs expectation within 5 standard deviations of the estimate (empirical per-pixel variance)."""
    r = (samples.astype(np.float64) - expected).reshape(-1, samples.shape[-1])
    se = r.std(0, ddof=1) / np.sqrt(len(r))
    z = r.mean(0) / np.maximum(se, 1e-300)
    print(f"[closed-form] {what}: z = {np.round(z, 2).tolist()}")
    assert (np.abs(z) <= 5.0).all(), (what, z, r.mean(0), se)


@pytest.mark.parametrize("backend", BACKENDS)
def test_russian_roulette_is_unbiased(backend):
    """The closed room with roulette on (max albedo channel 0.8 < 1): 32 samples per pixel average to
    E (1 - rho^D) / (1 - rho); the roulette really ends paths early."""
    scene, mat = closed_box_scene(ROOM_ALBEDOS["tinted"], (0.7, 1.3, 0.4))
    w, h, depth = 64, 48, 9
    frame = camera(BOX_FRAME_ARGS[0], np.add(*BOX_FRAME_ARGS), w, h, 90.0)
    img, _, _ = render(backend, scene, frame, settings(depth, rr=True, spp=16), w, h, sky=(0.0, 0.0, 0.0), calls=2)
    want = closed_box_value(mat, depth)
    assert_unbiased(img[..., :3], want, f"{backend} roulette")
    assert ulps(img[..., :3], want).max() > 1000       # not the roulette-free image


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("ior", [1.3, 1.5, 2.0])
def test_fresnel_branch_selection(backend, ior):
    """Untinted (TintOnTransmissive = 0), non-volumetric transmissive plane seen at 15..75 degrees: the Fresnel
    reflection (probability F, bsdf = rho) or the untinted transmission (bsdf = 1). Every pixel is rho c or c, and the mean
    is c (F rho + 1 - F) with Schlick's F at each pixel's camera-ray cosine."""
    scene, mat = plane_scene(dict(color=(0.7, 0.9, 0.4), transmission=1.0, roughness=0.0, ior=ior, tint=False))
    w, h = 128, 96
    frame = camera((0.0, -1.0, 1.0), (0.0, 0.0, 0.0), w, h, 60.0)
    img, _, _ = render(backend, scene, frame, settings(3), w, h)
    rho, c = albedo_of(mat)[:3], np.asarray(SKY)
    everywhere = np.ones((h, w), bool)
    assert_closed_form(img, [(c, everywhere), (rho * c, everywhere)], [(rho * rho * c, everywhere)], f"{backend} fresnel ior {ior}")
    _, d = primary_rays(frame, w, h)
    cos = -d[..., 2]
    assert cos.min() > 0.1 and cos.max() < 0.99
    ior32 = float(np.float32(ior))
    f0 = ((1.0 - ior32) / (1.0 + ior32)) ** 2
    F = (f0 + (1.0 - f0) * (1.0 - cos) ** 5)[..., None]
    assert_unbiased(img[..., :3], c * (F * rho + 1.0 - F), f"{backend} fresnel ior {ior}")


@pytest.mark.parametrize("backend", BACKENDS)
def test_stochastic_alpha(backend):
    """AlphaCutoff == 2.0: the surface is kept with probability A (pixel = rho c) and passed through otherwise (c);
    the mean is c (A rho + 1 - A)."""
    scene, mat = plane_scene(dict(color=(0.8, 0.5, 0.2, 0.4), cutoff=2.0))
    w, h = 128, 96
    frame = camera((0.2, 0.1, 2.0), (0.0, 0.0, 0.0), w, h)
    img, _, _ = render(backend, scene, frame, settings(3), w, h)
    alb = albedo_of(mat)
    rho, A, c = alb[:3], alb[3], np.asarray(SKY)
    everywhere = np.ones((h, w), bool)
    assert_closed_form(img, [(c, everywhere), (rho * c, everywhere)], [(rho * rho * c, everywhere)], f"{backend} stochastic alpha")
    assert 0.3 < match(img, c).mean() < 0.9
    assert_unbiased(img[..., :3], c * (A * rho + 1.0 - A), f"{backend} stochastic alpha")


# ================================================================================================ every production path
PRODUCTION = [("sync", {}), ("lanes4_async", dict(lanes=4)), ("ray_sorting", dict(sorting=True)), ("aovs", dict(aovs=True)),
              ("traverse_variant_1", dict(env={"IDKPT_TRAVERSE_VARIANT": "1"})),
              ("traverse_variant_2", dict(env={"IDKPT_TRAVERSE_VARIANT": "2"})),
              ("treelet_pairs", dict(env={"IDKPT_TREELET_PAIRS": "256"}))] + \
             [(f"tile_{t}_of_8", dict(tile=(8, t, 8))) for t in range(8)]


@pytest.mark.gpu
@pytest.mark.skipif(not _has_cuda(), reason="no CUDA device")
@pytest.mark.parametrize("config", [p[0] for p in PRODUCTION])
def test_production_paths_hit_the_closed_form(config):
    """The closed room (D = 5) and the TLAS of convex objects at 1920x1080 through one production configuration:
    pipelined lanes, ray sorting, AOVs, each traversal variant, treelets, or one of the 8 stripe tiles on its own rows."""
    opt = dict(PRODUCTION)[config]
    w, h = 1920, 1080
    tile = opt.get("tile", (8, 0, 1))
    rows = tile_rows(h, tile)
    kw = dict(tile=tile, lanes=opt.get("lanes", 0), env=opt.get("env"))

    scene, mat = closed_box_scene(ROOM_ALBEDOS["tinted"], (0.7, 1.3, 0.4))
    frame = camera(BOX_FRAME_ARGS[0], np.add(*BOX_FRAME_ARGS), w, h, 90.0)
    s = settings(5, aovs=opt.get("aovs", False), sorting=opt.get("sorting", False))
    img, _, _ = render("gpu", scene, frame, s, w, h, sky=(0.0, 0.0, 0.0), calls=3 if kw["lanes"] else 1, **kw)
    err = ulps(img[rows][..., :3], closed_box_value(mat, 5))
    assert err.max() <= box_tol(5), (config, err.max())

    scene, _, planes, mat, _ = polyhedron_scene("tlas")
    frame = camera((0.3, 20.0, 0.2), (0, 0, 0), w, h, 40.0, up=(0.0, 0.0, -1.0))
    s = settings(3, aovs=opt.get("aovs", False), sorting=opt.get("sorting", False))
    img, _, _ = render("gpu", scene, frame, s, w, h, **kw)
    main, extra, _, _ = polyhedron_expectation(frame, w, h, planes, mat, SKY, rows=rows)
    assert_closed_form(img[rows], main, extra, f"gpu 1080p {config} tlas")
