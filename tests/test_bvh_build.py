"""Host-side BLAS builder (mirror of SRC/Bvh/BLAS.cs + PreSplitting.cs): structural invariants of the
BLAS.cs:16-22 doc comment, and BVH traversal == brute force over all triangles (config 1 of BASELINE.json)."""
import importlib.util
import json
import os

import numpy as np

import oracle_lib as ol
from idkengine_b200 import scenes, host

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
_spec = importlib.util.spec_from_file_location("make_sponza_golden", os.path.join(GOLDEN_DIR, "make_sponza_golden.py"))
sponza_golden = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(sponza_golden)
SPONZA = json.load(open(os.path.join(GOLDEN_DIR, "sponza_golden.json")))


def check_invariants(scene):
    tris_seen = np.zeros(len(scene.blas_triangles), bool)
    for desc in scene.blas_descs:
        nodes = scene.blas_nodes[desc["NodeOffset"]: desc["NodeOffset"] + desc["NodeCount"]]
        assert desc["NodeCount"] % 2 == 0 and desc["NodeOffset"] % 2 == 0       # child pairs stay 64-byte aligned
        assert np.all(nodes[0]["Min"] == 0) and nodes[0]["TriCount"] == 0        # 32-byte pad
        root = nodes[1]
        assert root["TriCount"] == 0 and root["TriStartOrChild"] == 2            # root never a leaf, left child at 2
        visited = np.zeros(len(nodes), bool)
        visited[:2] = True
        stack = [(2, 0)]
        max_depth_pairs = 0
        tri_cursor = 0
        while stack:
            top, sdepth = stack.pop()
            l, r = nodes[top], nodes[top + 1]
            visited[top] = visited[top + 1] = True
            ll, rl = l["TriCount"] > 0, r["TriCount"] > 0
            if ll and rl:
                # leaf pair: one continuous range starting left; straddling part shared
                assert l["TriStartOrChild"] <= r["TriStartOrChild"] <= l["TriStartOrChild"] + l["TriCount"]
                assert r["TriStartOrChild"] + r["TriCount"] >= l["TriStartOrChild"] + l["TriCount"]
            for n in (l, r):
                if n["TriCount"] > 0:
                    a, b = n["TriStartOrChild"], n["TriStartOrChild"] + n["TriCount"]
                    assert 0 <= a and b <= desc["TriangleCount"]
                    tris_seen[desc["TriangleOffset"] + a: desc["TriangleOffset"] + b] = True
                    # leaf bounds contain their triangles
                    t = scene.blas_triangles[desc["TriangleOffset"] + a: desc["TriangleOffset"] + b]
                    for k in ("X", "Y", "Z"):
                        p = scene.positions[t[k]]
                        pts = np.stack([p["x"], p["y"], p["z"]], 1)
                        # presplit fragments may clip a triangle: the union of the leaves holding a triangle covers it,
                        # a single leaf need not. Only check against the root here.
                        assert np.all(pts >= root["Min"] - 1e-4) and np.all(pts <= root["Max"] + 1e-4)
                else:
                    c = n["TriStartOrChild"]
                    assert c > top and c % 2 == 0                              # DFS order, pairs at even ids
                    assert np.all(nodes[c]["Min"] >= n["Min"] - 1e-5) and np.all(nodes[c + 1]["Max"] <= n["Max"] + 1e-5)
            both = (not ll) and (not rl)
            if not rl:
                stack.append((r["TriStartOrChild"], sdepth + (1 if both else 0)))
            if not ll:
                stack.append((l["TriStartOrChild"], sdepth + (1 if both else 0)))
            max_depth_pairs = max(max_depth_pairs, sdepth)
        assert visited.all()                                                     # no empty subtrees left
        assert desc["RequiredStackSize"] <= 64
    assert tris_seen.all()


def test_invariants_cornell(cornell):
    check_invariants(cornell[0])
    info = cornell[0].build_info[0]
    assert info["source_triangles"] == 1006
    assert info["fragments"] >= info["triangles"] >= info["source_triangles"]


def test_invariants_multi_blas(multi_blas):
    check_invariants(multi_blas[0])
    assert len(multi_blas[0].blas_descs) == 3
    # refittable BLAS (crate) is not presplit: triangle count unchanged
    assert multi_blas[0].build_info[2]["triangles"] == multi_blas[0].build_info[2]["source_triangles"]


def test_invariants_atrium(atrium_small):
    check_invariants(atrium_small[0])


def _compare_to_brute_force(scene, rays):
    # A ray with an exactly-zero direction component whose origin lies on a box plane evaluates 0*inf = NaN in the
    # reference's slab test (IntersectionRoutines.glsl:29-31) and is culled there; that artefact is part of the
    # reference algorithm (and reproduced by oracle and kernel alike) but not of the brute-force intersector.
    rays = rays[np.all(rays["Direction"] != 0.0, axis=1)]
    bvh = ol.trace_rays(scene, rays)
    bf = ol.brute_force(scene, rays)
    # same closest distance for every ray, bit for bit (identical triangle arithmetic on both sides)
    assert np.array_equal(bvh["T"], bf["T"])
    hit = bf["TriangleId"] != 0xFFFFFFFF
    assert hit.sum() > 0.3 * len(rays)
    # ids agree except where two triangles are hit at the identical distance (shared edges / presplit duplicates)
    diff = bvh["TriangleId"] != bf["TriangleId"]
    if diff.any():
        ta = scene.blas_triangles[bvh["TriangleId"][diff]]
        tb = scene.blas_triangles[bf["TriangleId"][diff]]
        same_source = (ta["X"] == tb["X"]) & (ta["Y"] == tb["Y"]) & (ta["Z"] == tb["Z"])
        # remaining differences are exact-distance ties between coplanar neighbours (quad diagonals)
        assert diff.sum() - same_source.sum() <= 1e-2 * len(rays)
    assert np.array_equal(bvh["MeshTransformId"][~diff], bf["MeshTransformId"][~diff])


def test_bvh_equals_brute_force_cornell_256(cornell):
    """BASELINE.json configs[0]: 1k-tri Cornell box, 256x256, all 65,536 primary rays, CPU only."""
    scene, cam = cornell
    frame = scenes.camera_frame(cam, 256, 256)
    rays = ol.primary_rays(frame, 256, 256)
    assert len(rays) == 65536
    _compare_to_brute_force(scene, rays)


def test_bvh_equals_brute_force_multi_blas_random(multi_blas):
    scene, cam = multi_blas
    rng = np.random.RandomState(7)
    o = rng.uniform(-2.5, 2.5, (4000, 3)).astype(np.float32)
    o[:, 1] = np.abs(o[:, 1]) + 0.2
    d = rng.normal(size=(4000, 3)).astype(np.float32)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    _compare_to_brute_force(scene, ol.make_rays(o, d))


def test_cpu_collision_path_matches_glsl_path(cornell):
    """The C#-semantics traversal (division slab test, t > 0) finds the same closest hits as the GLSL-semantics one."""
    scene, cam = cornell
    frame = scenes.camera_frame(cam, 64, 64)
    rays = ol.gui_test_rays(frame, 64, 64)
    rays = rays[np.all(rays["Direction"] != 0.0, axis=1)]   # see _compare_to_brute_force
    a = ol.trace_rays(scene, rays)
    b, secs = ol.cpu_intersect(scene, rays, threads=2)
    assert secs > 0
    # the two intersectors differ in rounding (x*inv vs x/det, t>=0 vs t>0): rays exactly through an edge may slip
    # through one of them (neither is watertight), everything else agrees
    close = np.isclose(a["T"], b["T"], rtol=1e-5)
    assert (~close).mean() < 0.005
    assert (a["TriangleId"][close] != b["TriangleId"][close]).mean() < 0.01   # exact-distance ties only


def test_build_deterministic_and_threads_agree():
    s1, _ = scenes.atrium(40000, threads=1)
    s2, _ = scenes.atrium(40000, threads=4)
    assert np.array_equal(s1.blas_nodes, s2.blas_nodes)
    assert np.array_equal(s1.blas_triangles, s2.blas_triangles)


def test_real_sponza_sample_builds_and_traces_like_brute_force():
    """The architecture of IDKEngine's Sponza (tests/golden/sponza_architecture.npz, 11,105 of its triangles) placed like
    scenes.sponza_reference(): presplit build pinned to tests/golden/sponza_golden.json, and the primary rays of the
    reference's camera find the same closest hits as brute force."""
    P, I, M = sponza_golden.load_sample()
    scene = sponza_golden.sample_scene(P, I, M)
    assert sponza_golden.default_build(scene) == SPONZA["default_build"]
    info = scene.build_info[0]
    assert info["source_triangles"] == len(I) == SPONZA["sample"]["triangles"]
    assert info["source_triangles"] < info["triangles"] <= info["fragments"]       # presplit adds fragments, dedup drops some
    frame = scenes.camera_frame(scenes.SPONZA_CAMERA, 96, 54)
    rays = ol.primary_rays(frame, 96, 54)
    _compare_to_brute_force(scene, rays)


def test_build_settings_sweep_on_real_sponza_sample():
    """The builder settings of the README's table (Readme.md:812-824: `TRAVERSAL_COST=1.0`, `TriangleCost=1.1`, max 8
    primitives per leaf, OptimizeStackSize disabled, SplitFactor 0.0 / 0.3 / 1.0) on the Sponza sample. The README's
    figures are for the whole 262k-triangle model; the sample is pinned to this builder's values in sponza_golden.json:
    fragment and triangle counts and stack sizes exactly, SAH to 1e-9."""
    got = sponza_golden.settings_sweep(*sponza_golden.load_sample())
    exp = SPONZA["settings_sweep"]
    assert sorted(got) == sorted(exp)
    for sf in exp:
        for k in ("new_fragments", "new_triangles", "stack_size"):
            assert got[sf][k] == exp[sf][k], (sf, k)
        assert abs(got[sf]["sah"] - exp[sf]["sah"]) <= 1e-9 * exp[sf]["sah"], sf
    assert got["0.0"]["new_fragments"] == 0 and got["0.0"]["new_triangles"] == 0
    assert 0 < got["0.3"]["new_triangles"] <= got["0.3"]["new_fragments"] < got["1.0"]["new_fragments"]


def test_tlas_ploc_structure_and_equivalence(multi_blas):
    """TLAS.Build mirror (SRC/Bvh/TLAS.cs:28-141): 2n-1 nodes, root at 0, children adjacent, every instance in exactly
    one leaf, parents bound their children; the TLAS walk finds the same closest distances as the instance loop."""
    scene, cam = scenes.multi_blas(threads=1)
    scene.build_tlas()
    t = scene.tlas_nodes
    n = len(scene.blas_instances)
    assert len(t) == 2 * n - 1
    leaf = (t["IsLeafAndChildOrInstanceId"] >> 31) == 1
    ids = t["IsLeafAndChildOrInstanceId"] & 0x7FFFFFFF
    assert sorted(ids[leaf].tolist()) == list(range(n)) and not leaf[0]
    for i in np.nonzero(~leaf)[0]:
        c = ids[i]
        assert i < c < len(t) - 1
        assert np.all(t["Min"][i] <= np.minimum(t["Min"][c], t["Min"][c + 1]) + 1e-6)
        assert np.all(t["Max"][i] >= np.maximum(t["Max"][c], t["Max"][c + 1]) - 1e-6)
    rng = np.random.RandomState(2)
    o = rng.uniform(-2.5, 2.5, (3000, 3)).astype(np.float32)
    o[:, 1] = np.abs(o[:, 1]) + 0.2
    d = rng.normal(size=(3000, 3)).astype(np.float32)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    rays = ol.make_rays(o, d)
    a = ol.trace_rays(multi_blas[0], rays)
    b = ol.trace_rays(scene, rays)
    assert np.array_equal(a["T"], b["T"])
    # a bigger forest of instances: 40 copies of a small BLAS scattered around
    from idkengine_b200.host import Scene, Model, trs_matrix
    pos, idx = scenes.uv_sphere([0, 0, 0], 0.5, 8, 12)
    sc = Scene()
    for k in range(40):
        sc.add(Model(pos, idx, model_matrix=trs_matrix(0.5 + 0.02 * k, 7.0 * k, (rng.uniform(-6, 6), rng.uniform(0, 3), rng.uniform(-6, 6))), name=f"s{k}"), threads=1)
    flat = ol.trace_rays(sc, rays)
    sc.build_tlas()
    assert len(sc.tlas_nodes) == 79
    tl = ol.trace_rays(sc, rays)
    assert np.array_equal(flat["T"], tl["T"])
    assert np.array_equal(flat["TriangleId"], tl["TriangleId"])


# ---- on-disk BLAS cache (SURVEY 8f.4, include/idkhost_cache.h) ------------------------------------------------------
def test_blas_cache_round_trip_and_rejects(tmp_path):
    import time
    from idkengine_b200 import host, scenes
    cache = str(tmp_path / "bvh")
    t0 = time.perf_counter()
    a, _ = scenes.multi_blas(threads=1)
    fresh = host.Scene().add(*_models_of_multi_blas(), threads=1, cache_dir=cache)
    assert not any(i["from_cache"] for i in fresh.build_info)
    again = host.Scene().add(*_models_of_multi_blas(), threads=1, cache_dir=cache)
    assert all(i["from_cache"] for i in again.build_info)
    for f in ("blas_nodes", "blas_triangles", "blas_descs", "positions", "vertices"):
        assert getattr(fresh, f).tobytes() == getattr(again, f).tobytes() == getattr(a, f).tobytes(), f
    assert fresh.blas_stack_size == again.blas_stack_size
    # a different order in the scene rebases the cached triangle ids
    models = _models_of_multi_blas()
    swapped = host.Scene().add(models[2], models[0], models[1], threads=1, cache_dir=cache)
    direct = host.Scene().add(models[2], models[0], models[1], threads=1)
    assert all(i["from_cache"] for i in swapped.build_info)
    assert swapped.blas_triangles.tobytes() == direct.blas_triangles.tobytes() and swapped.blas_nodes.tobytes() == direct.blas_nodes.tobytes()
    # corruption / wrong key / truncation are detected
    import glob, os
    files = sorted(glob.glob(os.path.join(cache, "*.idkbvh")))
    assert len(files) == 3
    key = int(os.path.basename(files[0]).split(".")[0], 16)
    assert host.cache_load(files[0], key)[0] == host.CACHE_OK
    assert host.cache_load(files[0], key ^ 1)[0] == host.CACHE_ERR_KEY
    raw = bytearray(open(files[0], "rb").read())
    raw[len(raw) // 2] ^= 0x40
    bad = str(tmp_path / "bad.idkbvh")
    open(bad, "wb").write(raw)
    assert host.cache_load(bad, key)[0] == host.CACHE_ERR_CHECKSUM
    open(bad, "wb").write(raw[: len(raw) - 64])
    assert host.cache_load(bad, key)[0] == host.CACHE_ERR_FORMAT
    open(bad, "wb").write(b"not a cache")
    assert host.cache_load(bad, key)[0] == host.CACHE_ERR_FORMAT
    # a corrupt file in the cache directory falls back to a rebuild (and is overwritten)
    open(files[0], "wb").write(bytes(raw))
    healed = host.Scene().add(*_models_of_multi_blas(), threads=1, cache_dir=cache)
    assert sum(i["from_cache"] for i in healed.build_info) == 2
    assert healed.blas_nodes.tobytes() == a.blas_nodes.tobytes()
    assert host.cache_load(files[0], key)[0] == host.CACHE_OK


def _models_of_multi_blas():
    """The three models scenes.multi_blas() assembles (room, ball, crate)."""
    from idkengine_b200 import scenes
    return scenes.multi_blas_models()


def test_threaded_build_is_deterministic():
    """The task pool and the wide top-of-tree split must reproduce the serial builder bit for bit."""
    from idkengine_b200 import scenes
    a, _ = scenes.atrium(120000, threads=1)
    for th in (3, 8):
        b, _ = scenes.atrium(120000, threads=th)
        assert a.blas_nodes.tobytes() == b.blas_nodes.tobytes() and a.blas_triangles.tobytes() == b.blas_triangles.tobytes(), th
