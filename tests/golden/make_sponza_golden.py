"""Regenerate tests/golden/sponza_architecture.npz and tests/golden/sponza_golden.json from IDKEngine's Sponza model:

    python tests/golden/make_sponza_golden.py <IDKEngine>/Resource/Models/SponzaCompressed/Sponza.gltf

The whole model (262,267 triangles, ~750 KB even compressed) is too large for a test fixture, so the sample keeps its
architecture: every glTF primitive whose bounding box spans at least 10 units and that has at most 2,500 triangles (floor,
walls, arches, roof; the props and the dense ornaments are left out), with the original float32 positions and the
original triangles. The expected values are this builder's own results on the sample: they pin the host BLAS builder
against regressions. The README's published builder table is for the whole model."""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from idkengine_b200 import host, scenes  # noqa: E402
from idkengine_b200 import gpu_types as gt  # noqa: E402

SAMPLE = os.path.join(HERE, "sponza_architecture.npz")
GOLDEN = os.path.join(HERE, "sponza_golden.json")
MIN_EXTENT, MAX_TRIANGLES = 10.0, 2500
SPLIT_FACTORS = (0.0, 0.3, 1.0)


def take_sample(gltf_path):
    _, pos, _, _, idx, _, _ = scenes.load_gltf_geometry(gltf_path)
    first = np.cumsum([0] + [len(p) for p in pos])           # vertex offset of each primitive in the loader's indices
    keep = [k for k in range(len(pos))
            if np.linalg.norm(pos[k].max(0) - pos[k].min(0)) >= MIN_EXTENT and len(idx[k]) <= MAX_TRIANGLES]
    base = np.cumsum([0] + [len(pos[k]) for k in keep])
    positions = np.concatenate([pos[k] for k in keep]).astype(np.float32)
    indices = np.concatenate([idx[k] - first[k] + base[j] for j, k in enumerate(keep)]).astype(np.uint32)
    mesh_ids = np.concatenate([np.full(len(idx[k]), j, np.int32) for j, k in enumerate(keep)])
    return keep, positions, indices, mesh_ids


def load_sample():
    d = np.load(SAMPLE)
    return d["positions"], d["indices"], d["mesh_ids"]


def sample_scene(positions, indices, mesh_ids, threads=4):
    """The sample placed like scenes.sponza_reference() places the whole model (default build settings)."""
    model = host.Model(positions, indices, mesh_ids, model_matrix=host.trs_matrix(*scenes.SPONZA_PLACEMENT), name="sponza_architecture")
    return host.Scene().add(model, threads=threads)


def default_build(scene):
    info = scene.build_info[0]
    return dict(source_triangles=int(info["source_triangles"]), fragments=int(info["fragments"]),
                triangles=int(info["triangles"]), required_stack_size=int(info["required_stack_size"]))


def settings_sweep(positions, indices, mesh_ids):
    """The settings of the README's builder table (Readme.md:812-824): TRAVERSAL_COST 1.0, TriangleCost 1.1 (the
    defaults), at most 8 triangles per leaf, OptimizeStackSize disabled, SplitFactor 0.0 / 0.3 / 1.0."""
    pv = np.zeros(len(positions), gt.PackedVec3)
    pv["x"], pv["y"], pv["z"] = positions[:, 0], positions[:, 1], positions[:, 2]
    tris = np.zeros(len(indices), gt.GpuBlasTriangle)
    tris["X"], tris["Y"], tris["Z"], tris["MeshId"] = indices[:, 0], indices[:, 1], indices[:, 2], mesh_ids
    out = {}
    for sf in SPLIT_FACTORS:
        st = host.default_build_settings()
        st.MaxLeafTriangleCount = 8
        st.StackOptThreshold = 1 << 30
        st.SplitFactor = sf
        b = host.build_blas(pv, tris, presplit=sf > 0, threads=4, settings=st)
        out[str(sf)] = dict(new_fragments=int(b["fragment_count"]) - len(indices), new_triangles=len(b["triangles"]) - len(indices),
                            sah=float(b["sah"]), stack_size=int(b["required_stack_size"]))
    return out


if __name__ == "__main__":
    keep, positions, indices, mesh_ids = take_sample(sys.argv[1])
    np.savez_compressed(SAMPLE, positions=positions, indices=indices, mesh_ids=mesh_ids)
    positions, indices, mesh_ids = load_sample()
    out = dict(sample=dict(gltf_primitives=keep, vertices=len(positions), triangles=len(indices)),
               default_build=default_build(sample_scene(positions, indices, mesh_ids)),
               settings_sweep=settings_sweep(positions, indices, mesh_ids))
    json.dump(out, open(GOLDEN, "w"), indent=1)
    print(json.dumps(out, indent=1))
