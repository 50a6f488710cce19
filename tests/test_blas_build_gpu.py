"""Device BLAS build (idkpt_blas_build): every BLAS equals the host builder's (host_mirror/bvh_build.cpp) byte for byte --
nodes, unindexed triangles, fragment count, required stack size and the bits of the SAH."""
import importlib.util
import json
import os

import numpy as np
import pytest

from idkengine_b200 import capi, host, scenes, gpu_types as gt
from idkengine_b200.pathtracer import PathTracer, IdkPtError

pytestmark = pytest.mark.gpu

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
_spec = importlib.util.spec_from_file_location("make_sponza_golden", os.path.join(GOLDEN_DIR, "make_sponza_golden.py"))
sponza_golden = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(sponza_golden)
SPONZA = json.load(open(os.path.join(GOLDEN_DIR, "sponza_golden.json")))


@pytest.fixture(scope="module")
def pt():
    with PathTracer(64, 48) as p:
        yield p


def assert_same(dev, ref, what=""):
    assert dev["fragment_count"] == ref["fragment_count"], what
    assert dev["required_stack_size"] == ref["required_stack_size"], what
    assert len(dev["nodes"]) == len(ref["nodes"]), what
    assert dev["nodes"].tobytes() == ref["nodes"].tobytes(), what
    assert len(dev["triangles"]) == len(ref["triangles"]), what
    assert dev["triangles"].tobytes() == ref["triangles"].tobytes(), what
    assert np.float64(dev["sah"]).tobytes() == np.float64(ref["sah"]).tobytes(), what


def packed(p):
    p = np.asarray(p, np.float32).reshape(-1, 3)
    out = np.zeros(len(p), gt.PackedVec3)
    out["x"], out["y"], out["z"] = p[:, 0], p[:, 1], p[:, 2]
    return out


def blas_tris(idx, mesh=None, v_off=0):
    idx = np.asarray(idx, np.int64).reshape(-1, 3)
    t = np.zeros(len(idx), gt.GpuBlasTriangle)
    t["X"], t["Y"], t["Z"] = idx[:, 0] + v_off, idx[:, 1] + v_off, idx[:, 2] + v_off
    t["MeshId"] = np.arange(len(idx)) % 7 if mesh is None else mesh
    return t


def check(pt, positions, tris, presplit=True, settings=None, what=""):
    ref = host.build_blas(positions, tris, presplit=presplit, settings=settings)
    dev = pt.BuildBlas(positions, tris, presplit=presplit, settings=settings)
    assert_same(dev, ref, what)
    return dev, ref


def captured_build_inputs(make):
    """Runs make() (which builds a host.Scene) and returns (scene, [(positions, triangles, presplit)]): the inputs that
    Scene.add handed to the host builder, one per model."""
    jobs = []
    orig = host.build_blas

    def capture(positions, triangles, presplit=True, threads=None, settings=None):
        jobs.append((positions, triangles.copy(), presplit))
        return orig(positions, triangles, presplit, threads, settings)
    host.build_blas = capture
    try:
        scene = make()
    finally:
        host.build_blas = orig
    return scene, jobs


# ---------------------------------------------------------------------------------------------------------------- Sponza
def sponza_input():
    P, I, M = sponza_golden.load_sample()
    return packed(P), blas_tris(I, M)


def test_sponza_sample_default_build(pt):
    pv, tris = sponza_input()
    dev, _ = check(pt, pv, tris)
    g = SPONZA["default_build"]
    assert dev["fragment_count"] == g["fragments"] and len(dev["triangles"]) == g["triangles"]
    assert dev["required_stack_size"] == g["required_stack_size"]


@pytest.mark.parametrize("sf", sponza_golden.SPLIT_FACTORS)
def test_sponza_sample_settings_sweep(pt, sf):
    pv, tris = sponza_input()
    st = host.default_build_settings()
    st.MaxLeafTriangleCount = 8
    st.StackOptThreshold = 1 << 30
    st.SplitFactor = sf
    dev, _ = check(pt, pv, tris, presplit=sf > 0, settings=st)
    g = SPONZA["settings_sweep"][str(sf)]
    assert dev["fragment_count"] - len(tris) == g["new_fragments"] and len(dev["triangles"]) - len(tris) == g["new_triangles"]
    assert dev["sah"] == g["sah"] and dev["required_stack_size"] == g["stack_size"]


def test_stack_optimisation_collapses(pt):
    """The default build runs OptimizeStackSize's collapse passes: its stack size is below the unoptimised build's."""
    pv, tris = sponza_input()
    st = host.default_build_settings()
    st.StackOptThreshold = 1 << 30
    plain, _ = check(pt, pv, tris, settings=st)
    opt, _ = check(pt, pv, tris)
    assert opt["required_stack_size"] < plain["required_stack_size"]


# ---------------------------------------------------------------------------------------------------------------- atrium
@pytest.fixture(scope="module")
def atrium_inputs():
    out = {}
    for n in (262144, 1 << 20):
        _, jobs = captured_build_inputs(lambda: scenes.atrium(n, threads=os.cpu_count()))
        out[n] = jobs[0][:2]
    return out


@pytest.mark.parametrize("n", [262144, 1 << 20])
@pytest.mark.parametrize("presplit", [True, False])
def test_atrium(pt, atrium_inputs, n, presplit):
    pv, tris = atrium_inputs[n]
    check(pt, pv, tris, presplit=presplit, what=f"atrium {n} presplit={presplit}")


# ---------------------------------------------------------------------------------------------------------------- edges
@pytest.mark.parametrize("presplit", [True, False])
@pytest.mark.parametrize("count", [1, 2, 3])
def test_tiny_blases(pt, presplit, count):
    rng = np.random.default_rng(count)
    pv = packed(rng.uniform(-1, 1, (3 * count, 3)))
    tris = blas_tris(np.arange(3 * count))
    dev, _ = check(pt, pv, tris, presplit=presplit)
    if count == 1:
        assert dev["nodes"][2].tobytes() == dev["nodes"][3].tobytes() or not presplit


@pytest.mark.parametrize("presplit", [True, False])
def test_identical_triangles(pt, presplit):
    """All centroid keys equal: the stable order alone decides."""
    pv = packed([[0, 0, 0], [1, 0, 0], [0, 1, 0]])
    tris = blas_tris(np.tile([0, 1, 2], 700))
    check(pt, pv, tris, presplit=presplit)


@pytest.mark.parametrize("presplit", [True, False])
def test_zero_area_and_flat(pt, presplit):
    rng = np.random.default_rng(5)
    p = rng.uniform(-3, 3, (3000, 3))
    p[:, 1] = 0.25                                   # flat mesh: no extent on y
    idx = rng.integers(0, 3000, (2500, 3))
    idx[::5, 1] = idx[::5, 0]                        # zero-area triangles (repeated vertex)
    q = rng.uniform(-3, 3, (300, 3))                 # collinear triangles
    col = np.stack([q[:, 0], np.full(300, 0.25), q[:, 2]], 1)
    pts = np.concatenate([p, col, col * 0.5, col * 0.25])
    idx2 = np.stack([3000 + np.arange(300), 3300 + np.arange(300), 3600 + np.arange(300)], 1)
    check(pt, packed(pts), blas_tris(np.concatenate([idx, idx2])), presplit=presplit)


def test_huge_triangles_split_thousands_of_times(pt):
    rng = np.random.default_rng(9)
    small = rng.uniform(-0.5, 0.5, (20000, 3, 3)) * 0.01 + rng.uniform(-1, 1, (20000, 1, 3))
    big = np.array([[[-500, -1, -500], [500, -1, -500], [0, 300, 500]],
                    [[-400, 200, 400], [400, -50, 400], [0, 10, -400]],
                    [[-450, 3, -450], [450, 3, 450], [-450, 3, 450]]], np.float32)
    pts = np.concatenate([small, big]).reshape(-1, 3)
    tris = blas_tris(np.arange(len(pts)))
    dev, ref = check(pt, packed(pts), tris)
    assert dev["fragment_count"] - len(tris) > 3000


# ---------------------------------------------------------------------------------------------------------------- batch
def test_batched_build_equals_per_model_builds(pt):
    models = scenes.multi_blas_models()
    rng = np.random.default_rng(11)
    for k, (n, refit) in enumerate([(1, False), (57, True), (3000, False), (129, False), (12000, True)]):
        p = rng.uniform(-1, 1, (n, 3, 3)) * rng.uniform(0.01, 0.5) + rng.uniform(-2, 2, (n, 1, 3))
        m = host.Model(p.reshape(-1, 3), np.arange(3 * n).reshape(-1, 3), name=f"r{k}")
        m.refittable = refit
        models.append(m)
    scene, captured = captured_build_inputs(lambda: host.Scene().add(*models))
    jobs = [(t, presplit) for _, t, presplit in captured]
    assert [p for _, p in jobs] == [not m.refittable for m in models]
    devs = pt.BuildBlases(scene.positions, jobs)
    assert len(devs) == len(models)
    for b, ((src, presplit), dev) in enumerate(zip(jobs, devs)):
        assert_same(dev, host.build_blas(scene.positions, src, presplit=presplit), f"blas {b}")


# ---------------------------------------------------------------------------------------------------------------- plumbing
def test_device_built_scene_renders_identically(pt):
    ref_scene, cam = scenes.multi_blas()
    dev_scene = host.Scene().add(*scenes.multi_blas_models(), builder=pt.BlasBuilder)
    dev_scene.add_light((-1.0, 2.5, 1.0), (30.0, 28.0, 20.0), 0.3)
    assert dev_scene.blas_nodes.tobytes() == ref_scene.blas_nodes.tobytes()
    assert dev_scene.blas_triangles.tobytes() == ref_scene.blas_triangles.tobytes()
    imgs = []
    for sc in (ref_scene, dev_scene):
        with PathTracer(96, 64) as r:
            r.SetScene(sc); r.SetSky((0.6, 0.7, 0.9)); r.SetFrame(scenes.camera_frame(cam, 96, 64))
            r.Compute()
            imgs.append(r.Result)
    assert imgs[0].tobytes() == imgs[1].tobytes()


def test_device_built_blas_refits_like_host_built(pt):
    """Skin the refittable crate (scale 1.1) and refit its BLAS: same nodes whether the BLAS was built on the host or here."""
    ref_scene, cam = scenes.multi_blas()
    dev_scene = host.Scene().add(*scenes.multi_blas_models(), builder=pt.BlasBuilder)
    out = []
    for sc in (ref_scene, dev_scene):
        with PathTracer(64, 48) as r:
            r.SetScene(sc)
            d = sc.blas_descs[2]
            assert d["IsRefittable"] == 1
            tris = sc.blas_triangles[d["TriangleOffset"]: d["TriangleOffset"] + d["TriangleCount"]]
            idx = np.concatenate([tris["X"], tris["Y"], tris["Z"]]); v0, v1 = int(idx.min()), int(idx.max()) + 1
            u = np.zeros(v1 - v0, gt.GpuUnskinnedVertex)
            u["JointWeights"][:, 0] = 1.0
            for k, c in enumerate("xyz"):
                u["Position"][:, k] = sc.positions[c][v0:v1]
            u["Normal"], u["Tangent"] = sc.vertices["Normal"][v0:v1], sc.vertices["Tangent"][v0:v1]
            jm = np.zeros((1, 3, 4), np.float32); jm[0, 0, 0] = jm[0, 1, 1] = jm[0, 2, 2] = 1.1
            cmd = np.zeros(1, gt.IdkPtSkinningCmd); cmd["OutputVertexOffset"], cmd["VertexCount"] = v0, v1 - v0
            r.SetSkinningData(u); r.SkinVertices(jm, cmd); r.BlasRefit(2, 1)
            out.append(r.ReadRange(capi.IDKPT_ARRAY_BLAS_NODES, int(d["NodeOffset"]), int(d["NodeCount"])))
    assert out[0].tobytes() == out[1].tobytes()


def test_build_between_async_computes_leaves_the_image(pt):
    scene, cam = scenes.multi_blas()
    pv, tris = sponza_input()
    imgs = []
    for build in (False, True):
        with PathTracer(96, 64) as r:
            r.SetScene(scene); r.SetSky((0.6, 0.7, 0.9)); r.SetFrame(scenes.camera_frame(cam, 96, 64))
            r.ComputeAsync()
            if build:
                r.BuildBlas(pv, tris)
            r.ComputeAsync()
            r.Sync()
            imgs.append((r.Result, r.AccumulatedSamples))
    assert imgs[0][0].tobytes() == imgs[1][0].tobytes() and imgs[0][1] == imgs[1][1]


# ---------------------------------------------------------------------------------------------------------------- errors
def _raw_build(pt, positions, tris, descs):
    infos = np.zeros(max(len(descs), 1), gt.IdkPtBlasBuildInfo)
    return pt._lib.idkpt_blas_build(pt._ctx, positions.ctypes.data if len(positions) else None, len(positions),
                                    tris.ctypes.data if len(tris) else None, len(tris), descs.ctypes.data, len(descs), None,
                                    infos.ctypes.data, None)


def _descs(*rows):
    d = np.zeros(len(rows), gt.IdkPtBlasBuildDesc)
    for i, (off, cnt, refit) in enumerate(rows):
        d[i]["TriangleOffset"], d[i]["TriangleCount"], d[i]["IsRefittable"] = off, cnt, refit
    return d


def test_bad_inputs_are_refused_and_the_context_stays_usable(pt):
    pv = packed(np.random.default_rng(2).uniform(-1, 1, (30, 3)))
    tris = blas_tris(np.arange(30))
    INV, UNS = -1, -6                                  # IDKPT_ERR_INVALID_ARGUMENT, IDKPT_ERR_UNSUPPORTED
    bad_idx = tris.copy(); bad_idx[3]["Y"] = 30
    neg_idx = tris.copy(); neg_idx[4]["Z"] = -1
    assert _raw_build(pt, pv, bad_idx, _descs((0, 10, 0))) == INV
    assert _raw_build(pt, pv, neg_idx, _descs((0, 10, 1))) == INV
    assert _raw_build(pt, pv, tris, _descs((0, 10, 0), (10, 0, 0))) == INV            # empty BLAS
    assert _raw_build(pt, pv, tris, _descs((5, 6, 0))) == INV                          # past the end
    assert _raw_build(pt, pv, tris, _descs((0xFFFFFFFF, 2, 0))) == INV                 # offset overflow
    nan = pv.copy(); nan[7]["y"] = np.nan
    assert _raw_build(pt, nan, tris, _descs((0, 10, 0))) == INV
    inf = pv.copy(); inf[7]["x"] = np.inf
    assert _raw_build(pt, inf, tris, _descs((0, 10, 0))) == INV
    huge = pv.copy(); huge[0]["x"], huge[1]["x"], huge[1]["y"], huge[1]["z"] = -3e38, 3e38, 3e38, 3e38   # finite, half-area is not
    assert _raw_build(pt, huge, tris, _descs((0, 10, 0))) == INV
    st = host.default_build_settings()
    st.SplitFactor = 1e9                                                               # pre-splits far past 2^24 fragments
    with pytest.raises(IdkPtError) as e:
        pt.BuildBlas(pv, tris, settings=st)
    assert f"({UNS})" in str(e.value)
    check(pt, pv, tris)
