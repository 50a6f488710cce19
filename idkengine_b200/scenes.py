"""Synthetic scene generators for the configs of BASELINE.json (SURVEY.md section 8d) plus a loader for
the reference's own Sponza geometry (tests/golden/ keeps a sample of it for the tests).

All generators are seeded and deterministic; all materials use constant (1x1) textures, i.e. factors only
(the reference's own fallback for missing maps, SRC/Utils/ModelLoader.cs:877-885).
"""
import json
import os
import numpy as np

from . import gpu_types as gt
from .host import Model, Scene, trs_matrix, make_per_frame_data, view_dir_from_angles

SEED = 0x1D4E


# --------------------------------------------------------------------------- primitives
def quad(p0, p1, p2, p3):
    """Two triangles p0-p1-p2, p0-p2-p3."""
    pos = np.array([p0, p1, p2, p3], np.float32)
    idx = np.array([[0, 1, 2], [0, 2, 3]], np.uint32)
    return pos, idx


def grid(origin, du, dv, nu, nv, displace=None):
    """(nu x nv) quads spanning origin + u*du + v*dv, optionally displaced by displace(u, v) -> (N,3)."""
    u, v = np.meshgrid(np.linspace(0, 1, nu + 1), np.linspace(0, 1, nv + 1), indexing="ij")
    u, v = u.reshape(-1), v.reshape(-1)
    pos = np.asarray(origin, np.float64)[None, :] + u[:, None] * np.asarray(du, np.float64)[None, :] + v[:, None] * np.asarray(dv, np.float64)[None, :]
    if displace is not None:
        pos = pos + displace(u, v)
    i, j = np.meshgrid(np.arange(nu), np.arange(nv), indexing="ij")
    a = (i * (nv + 1) + j).reshape(-1)
    b = a + (nv + 1)
    idx = np.concatenate([np.stack([a, b, b + 1], 1), np.stack([a, b + 1, a + 1], 1)]).astype(np.uint32)
    return pos.astype(np.float32), idx


def box(mn, mx, rot_y_deg=0.0):
    mn, mx = np.asarray(mn, np.float64), np.asarray(mx, np.float64)
    c = (mn + mx) * 0.5
    h = (mx - mn) * 0.5
    corners = np.array([[sx, sy, sz] for sx in (-1, 1) for sy in (-1, 1) for sz in (-1, 1)], np.float64) * h
    a = np.deg2rad(rot_y_deg)
    r = np.array([[np.cos(a), 0, np.sin(a)], [0, 1, 0], [-np.sin(a), 0, np.cos(a)]])
    pos = corners @ r.T + c
    # corner index = 4*ix + 2*iy + iz
    faces = [(0, 1, 3, 2), (4, 6, 7, 5), (0, 4, 5, 1), (2, 3, 7, 6), (0, 2, 6, 4), (1, 5, 7, 3)]
    idx = []
    for f in faces:
        idx += [[f[0], f[1], f[2]], [f[0], f[2], f[3]]]
    return pos.astype(np.float32), np.array(idx, np.uint32)


def uv_sphere(center, radius, stacks, slices):
    """stacks x slices UV sphere: 2*slices cap triangles + 2*slices*(stacks-2) band triangles."""
    center = np.asarray(center, np.float64)
    th = np.linspace(0, np.pi, stacks + 1)[1:-1]
    ph = np.linspace(0, 2 * np.pi, slices, endpoint=False)
    ring = np.stack([np.outer(np.sin(th), np.cos(ph)), np.outer(np.cos(th), np.ones_like(ph)), np.outer(np.sin(th), np.sin(ph))], -1)
    pos = np.concatenate([[[0, 1, 0]], ring.reshape(-1, 3), [[0, -1, 0]]]) * radius + center
    idx = []
    top, bottom = 0, 1 + (stacks - 1) * slices
    for s in range(slices):
        idx.append([top, 1 + (s + 1) % slices, 1 + s])
    for r in range(stacks - 2):
        for s in range(slices):
            a = 1 + r * slices + s
            b = 1 + r * slices + (s + 1) % slices
            c, d = a + slices, b + slices
            idx += [[a, b, d], [a, d, c]]
    base = 1 + (stacks - 2) * slices
    for s in range(slices):
        idx.append([bottom, base + s, base + (s + 1) % slices])
    return pos.astype(np.float32), np.array(idx, np.uint32)


def cylinder(base, radius, height, seg, rings, taper=0.0):
    """Open-ended tessellated column with 2*seg*rings triangles."""
    base = np.asarray(base, np.float64)
    t = np.linspace(0, 1, rings + 1)
    ph = np.linspace(0, 2 * np.pi, seg, endpoint=False)
    r = radius * (1.0 - taper * t) * (1.0 + 0.04 * np.sin(t * 40.0))
    pos = np.stack([np.outer(r, np.cos(ph)), np.outer(t * height, np.ones_like(ph)), np.outer(r, np.sin(ph))], -1).reshape(-1, 3) + base
    i, j = np.meshgrid(np.arange(rings), np.arange(seg), indexing="ij")
    a = (i * seg + j).reshape(-1)
    b = (i * seg + (j + 1) % seg).reshape(-1)
    c, d = a + seg, b + seg
    idx = np.concatenate([np.stack([a, d, b], 1), np.stack([a, c, d], 1)]).astype(np.uint32)
    return pos.astype(np.float32), idx


class _Assembler:
    def __init__(self):
        self.pos, self.idx, self.mesh, self.nv = [], [], [], 0

    def add(self, pi, mesh_id):
        p, i = pi
        self.pos.append(p)
        self.idx.append(i + self.nv)
        self.mesh.append(np.full(len(i), mesh_id, np.int32))
        self.nv += len(p)

    def tri_count(self):
        return sum(len(i) for i in self.idx)

    def model(self, meshes, materials, model_matrix=None, name="model"):
        return Model(np.concatenate(self.pos), np.concatenate(self.idx), np.concatenate(self.mesh),
                     meshes=meshes, materials=materials, model_matrix=model_matrix, name=name)


def _materials(specs):
    """specs: list of dict(color=(r,g,b[,a]), emissive=(..), metallic, roughness, transmission, ior, cutoff,
    volumetric, absorbance)."""
    mats = gt.default_material(len(specs))
    meshes = gt.default_mesh(len(specs))
    for k, s in enumerate(specs):
        col = list(s.get("color", (1, 1, 1)))
        if len(col) == 3:
            col.append(1.0)
        mats["BaseColorFactor"][k] = gt.pack_unorm4x8(np.array(col))
        mats["EmissiveFactor"][k] = s.get("emissive", (0, 0, 0))
        mats["MetallicFactor"][k] = s.get("metallic", 0.0)
        mats["RoughnessFactor"][k] = s.get("roughness", 0.8)
        mats["TransmissionFactor"][k] = s.get("transmission", 0.0)
        mats["IOR"][k] = s.get("ior", 1.5)
        mats["AlphaCutoff"][k] = s.get("cutoff", 0.0)
        mats["IsVolumetric"][k] = 1 if s.get("volumetric", False) else 0
        mats["Absorbance"][k] = s.get("absorbance", (0, 0, 0))
        meshes["MaterialId"][k] = k
        meshes["EmissiveBias"][k] = s.get("emissive_bias", 0.0)
        meshes["TintOnTransmissive"][k] = 1 if s.get("tint", True) else 0
    return meshes, mats


# --------------------------------------------------------------------------- config 1: Cornell-1k
def cornell_1k(threads=None):
    """SURVEY 8d config 1: 5 walls + ceiling emitter + tall box + 16x30 UV sphere (metal) + small glass sphere
    + one alpha-blended card ~= 1k triangles, single BLAS, identity transform."""
    specs = [
        dict(color=(0.73, 0.73, 0.73)),                           # 0 white
        dict(color=(0.65, 0.05, 0.05)),                           # 1 red
        dict(color=(0.12, 0.45, 0.15)),                           # 2 green
        dict(color=(1, 1, 1), emissive=(15, 15, 15)),             # 3 emitter
        dict(color=(0.9, 0.8, 0.6), metallic=1.0, roughness=0.2),  # 4 metal sphere
        dict(color=(0.9, 0.95, 1.0), transmission=1.0, roughness=0.0, ior=1.5, volumetric=True,
             absorbance=(0.3, 0.1, 0.05)),                        # 5 glass sphere
        dict(color=(0.2, 0.3, 0.9, 0.5), cutoff=2.0),             # 6 blended card
    ]
    meshes, mats = _materials(specs)
    a = _Assembler()
    a.add(quad([-1, 0, -1], [-1, 0, 1], [1, 0, 1], [1, 0, -1]), 0)      # floor
    a.add(quad([-1, 2, -1], [1, 2, -1], [1, 2, 1], [-1, 2, 1]), 0)      # ceiling
    a.add(quad([-1, 0, -1], [1, 0, -1], [1, 2, -1], [-1, 2, -1]), 0)    # back
    a.add(quad([-1, 0, -1], [-1, 2, -1], [-1, 2, 1], [-1, 0, 1]), 1)    # left (red)
    a.add(quad([1, 0, -1], [1, 0, 1], [1, 2, 1], [1, 2, -1]), 2)        # right (green)
    a.add(quad([-0.3, 1.995, -0.3], [0.3, 1.995, -0.3], [0.3, 1.995, 0.3], [-0.3, 1.995, 0.3]), 3)
    a.add(box([-0.65, 0, -0.6], [-0.15, 1.2, -0.1], rot_y_deg=18.0), 0)
    a.add(uv_sphere([0.42, 0.4, 0.25], 0.4, 16, 30), 4)
    a.add(uv_sphere([-0.35, 0.25, 0.55], 0.25, 6, 8), 5)
    a.add(quad([0.1, 0.0, 0.75], [0.9, 0.0, 0.75], [0.9, 0.9, 0.75], [0.1, 0.9, 0.75]), 6)
    scene = Scene().add(a.model(meshes, mats, name="cornell"), threads=threads)
    cam = dict(position=(0.0, 1.0, 3.4), view_dir=(0.0, 0.0, -1.0), fov_y_deg=40.0)
    return scene, cam


# --------------------------------------------------------------------------- config 2/3: atrium
def atrium(target_tris=262144, seed=SEED, rotate_deg=0.0, instances=False, threads=None, transform=True):
    """'Sponza-sized synthetic mesh' (north_star): a colonnaded two-storey atrium -- big 2-triangle walls/floor
    (exercise PreSplitting), arcades of tessellated columns, draped cloth grids, foliage cards with alpha-mask and
    alpha-blend materials, emissive lamps -- scaled by tessellation to target_tris +- 1 %.
    transform=True keeps geometry in a smaller local space and places it with scale 1.815 / translate (0,-1,0)
    like the reference places Sponza (SRC/Application.cs:448)."""
    rng = np.random.RandomState(seed & 0x7FFFFFFF)
    specs = [
        dict(color=(0.72, 0.70, 0.66), roughness=0.9),                       # 0 stone walls
        dict(color=(0.55, 0.52, 0.50), roughness=0.6, metallic=0.05),        # 1 floor
        dict(color=(0.70, 0.68, 0.62), roughness=0.8),                       # 2 columns
        dict(color=(0.75, 0.08, 0.06), roughness=0.95),                      # 3 cloth red
        dict(color=(0.08, 0.35, 0.10), roughness=0.95),                      # 4 cloth green
        dict(color=(0.10, 0.15, 0.60), roughness=0.95),                      # 5 cloth blue
        dict(color=(0.95, 0.80, 0.45), metallic=1.0, roughness=0.25),        # 6 brass trim
        dict(color=(1.0, 0.9, 0.7), emissive=(1, 0.9, 0.7), emissive_bias=14.0),  # 7 lamps
        dict(color=(0.25, 0.55, 0.20, 1.0), cutoff=0.5),                     # 8 foliage (mask, visible)
        dict(color=(0.25, 0.55, 0.20, 0.3), cutoff=0.5),                     # 9 foliage (mask, cut away)
        dict(color=(0.6, 0.8, 0.9, 0.4), cutoff=2.0),                        # 10 glass panes (blend)
        dict(color=(0.85, 0.95, 1.0), transmission=0.95, roughness=0.02, ior=1.45, volumetric=True,
             absorbance=(0.4, 0.1, 0.05)),                                   # 11 crystal orbs
    ]
    meshes, mats = _materials(specs)

    n_cols_side, floors = 12, 2
    n_columns = n_cols_side * 2 * floors
    n_cloth, n_orbs, n_cards = 40, 6, 160
    fixed = 2 * 9 + 12 * 10 + 2 * n_cards + 2 * 8 + 12 * 6
    budget = max(target_tris - fixed, 2000)
    # ~45 % columns, ~45 % cloth, ~10 % orbs
    col_tris = budget * 0.45 / n_columns
    seg = int(np.clip(np.sqrt(col_tris / 2 / 3.0), 6, 4096))
    rings = max(2, int(col_tris / (2 * seg)))
    cloth_tris = budget * 0.45 / n_cloth
    g = max(2, int(np.sqrt(cloth_tris / 2)))
    orb_tris = budget * 0.10 / n_orbs
    osl = int(np.clip(np.sqrt(orb_tris / 2), 6, 4096))
    ost = max(4, int(orb_tris / (2 * osl)) + 1)

    a = _Assembler()
    X, Z, H = 14.0, 7.5, 11.0
    a.add(quad([-X, 0, -Z], [-X, 0, Z], [X, 0, Z], [X, 0, -Z]), 1)                       # floor
    a.add(quad([-X, 0, -Z], [X, 0, -Z], [X, H, -Z], [-X, H, -Z]), 0)                       # walls
    a.add(quad([-X, 0, Z], [-X, H, Z], [X, H, Z], [X, 0, Z]), 0)
    a.add(quad([-X, 0, -Z], [-X, H, -Z], [-X, H, Z], [-X, 0, Z]), 0)
    a.add(quad([X, 0, -Z], [X, 0, Z], [X, H, Z], [X, H, -Z]), 0)
    a.add(quad([-X, H, -Z], [X, H, -Z], [X, H, -Z * 0.45], [-X, H, -Z * 0.45]), 0)         # roof strips, open centre
    a.add(quad([-X, H, Z * 0.45], [X, H, Z * 0.45], [X, H, Z], [-X, H, Z]), 0)
    a.add(quad([-X, H * 0.5, -Z], [-X, H * 0.5, -Z * 0.62], [X, H * 0.5, -Z * 0.62], [X, H * 0.5, -Z]), 1)  # gallery floors
    a.add(quad([-X, H * 0.5, Z * 0.62], [-X, H * 0.5, Z], [X, H * 0.5, Z], [X, H * 0.5, Z * 0.62]), 1)
    for k in range(10):                                                                    # unaligned blocks
        cx, cz = rng.uniform(-X * 0.8, X * 0.8), rng.uniform(-Z * 0.3, Z * 0.3)
        s = rng.uniform(0.3, 0.9)
        a.add(box([cx - s, 0, cz - s * 0.6], [cx + s, rng.uniform(0.4, 1.6), cz + s * 0.6], rot_y_deg=rng.uniform(0, 90)), 0 if k % 3 else 6)
    for f in range(floors):
        for side in (-1, 1):
            for c in range(n_cols_side):
                x = -X + (c + 0.5) * (2 * X / n_cols_side)
                a.add(cylinder([x, f * H * 0.5, side * Z * 0.62], 0.38, H * 0.5, seg, rings, taper=0.12), 2)
    for c in range(n_cloth):
        x = -X * 0.92 + (c % 20) * (2 * X * 0.92 / 19)
        side = -1 if c < 20 else 1
        ph = rng.uniform(0, 6.28)
        amp = rng.uniform(0.10, 0.30)

        def drape(u, v, ph=ph, amp=amp, side=side):
            d = np.zeros((len(u), 3))
            d[:, 2] = side * amp * np.sin(u * 9.0 + ph) * (0.3 + v) + side * 0.05 * np.sin(v * 23.0 + u * 31.0)
            d[:, 0] = 0.04 * np.sin(v * 17.0 + ph)
            return d
        a.add(grid([x - 0.55, H * 0.5 - 0.2, side * Z * 0.60], [1.1, 0, 0], [0, -3.2, 0], g, g, drape), 3 + c % 3)
    for k in range(n_orbs):
        a.add(uv_sphere([-X * 0.7 + k * (1.4 * X / (n_orbs - 1)), 1.1, 0.0], 0.45, ost, osl), 11 if k % 2 == 0 else 6)
    for k in range(n_cards):
        cx, cz, cy = rng.uniform(-X * 0.9, X * 0.9), rng.uniform(-Z * 0.5, Z * 0.5), rng.uniform(0.0, 2.0)
        ang = rng.uniform(0, np.pi)
        dx, dz = 0.4 * np.cos(ang), 0.4 * np.sin(ang)
        a.add(quad([cx - dx, cy, cz - dz], [cx + dx, cy, cz + dz], [cx + dx, cy + 0.8, cz + dz], [cx - dx, cy + 0.8, cz - dz]),
              8 + (k % 3 if k % 3 < 2 else 2))
    for k in range(8):                                                                     # lamps
        x = -X * 0.8 + k * (1.6 * X / 7)
        a.add(quad([x - 0.35, H * 0.5 - 0.02, -0.35], [x + 0.35, H * 0.5 - 0.02, -0.35], [x + 0.35, H * 0.5 - 0.02, 0.35], [x - 0.35, H * 0.5 - 0.02, 0.35]), 7)
    for k in range(6):                                                                     # brass rails
        z = (-1 if k % 2 else 1) * Z * 0.62
        a.add(box([-X + k * 4.0, H * 0.5 + 0.9, z - 0.04], [-X + k * 4.0 + 3.6, H * 0.5 + 1.0, z + 0.04]), 6)

    # trim to target with an extra fine cloth
    missing = target_tris - a.tri_count()
    if missing > 8:
        gg = max(1, int(np.sqrt(missing / 2)))
        a.add(grid([-2.0, 0.02, -1.0], [4.0, 0, 0], [0, 0, 2.0], gg, max(1, missing // (2 * gg)),
                   lambda u, v: np.stack([0 * u, 0.03 * np.sin(u * 40) * np.sin(v * 40), 0 * u], 1)), 5)

    if transform:
        mm = trs_matrix(1.815, rotate_deg, (0.0, -1.0, 0.0))
        inv_s = 1.0 / 1.815
        for k in range(len(a.pos)):
            a.pos[k] = (a.pos[k] * np.float32(inv_s)).astype(np.float32)
        model_matrix = mm
    else:
        model_matrix = trs_matrix(1.0, rotate_deg)
    scene = Scene().add(a.model(meshes, mats, model_matrix=model_matrix, name="atrium"), threads=threads)
    # Reference camera (SRC/Application.cs:444): pos (7.63, 2.71, 0.8), yaw 194.6, pitch 82.6, fovY 102
    cam = dict(position=(7.63, 2.71, 0.8), view_dir=tuple(view_dir_from_angles(360.0 - 165.4, 90.0 - 7.4)), fov_y_deg=102.0)
    return scene, cam


def street_canyon(target_tris=3_900_000, seed=SEED + 1, threads=None):
    """Config 4 stand-in for Bistro: the atrium generator rotated 37 degrees so that nothing is axis aligned
    (stress for PreSplitting, cf. BLAS.cs:33-35)."""
    return atrium(target_tris, seed, rotate_deg=37.0, threads=threads)


# --------------------------------------------------------------------------- multi-BLAS test scene
def multi_blas_models():
    """room, ball (rotated / scaled instance), crate (refittable: the non-presplit builder path)."""
    specs_room = [dict(color=(0.7, 0.7, 0.7)), dict(color=(1, 1, 1), emissive=(12, 12, 12))]
    meshes, mats = _materials(specs_room)
    a = _Assembler()
    a.add(quad([-3, 0, -3], [-3, 0, 3], [3, 0, 3], [3, 0, -3]), 0)
    a.add(quad([-3, 0, -3], [3, 0, -3], [3, 4, -3], [-3, 4, -3]), 0)
    a.add(quad([-1, 3.99, -1], [1, 3.99, -1], [1, 3.99, 1], [-1, 3.99, 1]), 1)
    room = a.model(meshes, mats, name="room")
    m2, t2 = _materials([dict(color=(0.9, 0.3, 0.2), metallic=0.6, roughness=0.3)])
    b = _Assembler()
    b.add(uv_sphere([0, 0, 0], 1.0, 24, 32), 0)
    ball = b.model(m2, t2, model_matrix=trs_matrix(0.8, 90.0, (-1.2, 0.8, 0.0)), name="ball")
    m3, t3 = _materials([dict(color=(0.2, 0.4, 0.9), roughness=0.5)])
    c = _Assembler()
    c.add(box([-0.5, -0.5, -0.5], [0.5, 0.5, 0.5]), 0)
    c.add(cylinder([0, 0.5, 0], 0.3, 1.0, 24, 6), 0)
    crate = c.model(m3, t3, model_matrix=trs_matrix((1.0, 1.4, 0.7), 45.0, (1.3, 0.7, 0.4)), name="crate")
    crate.refittable = True  # exercises the non-presplit (BLAS.GetUnindexedTriangles) path
    return [room, ball, crate]


def multi_blas(threads=None):
    scene = Scene().add(*multi_blas_models(), threads=threads)
    scene.add_light((-1.0, 2.5, 1.0), (30.0, 28.0, 20.0), 0.3)
    cam = dict(position=(0.0, 1.6, 5.0), view_dir=(0.0, -0.1, -1.0), fov_y_deg=60.0)
    return scene, cam



def instance_grid(n=3, threads=None):
    """n^3 small models (spheres, boxes, cylinders; rotated / non-uniformly scaled instances) over a floor: a TLAS with
    2*(n^3+1)-1 nodes whose walk (BVHIntersect.glsl:205-272) is several levels deep, unlike multi_blas' three instances."""
    models = []
    meshes, mats = _materials([dict(color=(0.75, 0.75, 0.7))])
    a = _Assembler()
    a.add(quad([-6, 0, -6], [-6, 0, 6], [6, 0, 6], [6, 0, -6]), 0)
    models.append(a.model(meshes, mats, name="floor"))
    k = 0
    for ix in range(n):
        for iy in range(n):
            for iz in range(n):
                col = (0.25 + 0.25 * ix, 0.3 + 0.2 * iy, 0.35 + 0.2 * iz)
                spec = dict(color=col, metallic=0.5 if k % 3 == 0 else 0.0, roughness=0.2 + 0.1 * (k % 5))
                if k % 7 == 3:
                    spec = dict(color=(1.0, 0.9, 0.7), emissive=(6.0, 5.0, 3.0))
                m, t = _materials([spec])
                b = _Assembler()
                kind = k % 3
                if kind == 0:
                    b.add(uv_sphere([0, 0, 0], 0.45, 10, 14), 0)
                elif kind == 1:
                    b.add(box([-0.4, -0.4, -0.4], [0.4, 0.4, 0.4]), 0)
                else:
                    b.add(cylinder([0, -0.4, 0], 0.3, 0.8, 12, 3), 0)
                pos = (-2.4 + 2.4 * ix + 0.3 * iy, 0.7 + 1.5 * iy, -2.4 + 2.4 * iz - 0.2 * ix)
                scale = (0.8 + 0.15 * (k % 4), 0.9 + 0.2 * (k % 3), 1.0 + 0.1 * (k % 2))
                models.append(b.model(m, t, model_matrix=trs_matrix(scale, 17.0 * k, pos), name=f"obj{k}"))
                k += 1
    scene = Scene().add(*models, threads=threads)
    scene.add_light((0.0, 6.0, 0.0), (40.0, 38.0, 34.0), 0.4)
    scene.build_tlas()
    cam = dict(position=(0.5, 3.2, 8.5), view_dir=(-0.05, -0.28, -1.0), fov_y_deg=55.0)
    return scene, cam


# --------------------------------------------------------------------------- textured room (material textures)
def _checker(n, cells, a, b, alpha_a=255, alpha_b=255, seed=0):
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:n, 0:n]
    on = (((xx * cells) // n + (yy * cells) // n) % 2).astype(bool)
    img = np.zeros((n, n, 4), np.uint8)
    img[..., :3] = np.where(on[..., None], np.array(a, np.uint8), np.array(b, np.uint8))
    img[..., :3] = np.clip(img[..., :3].astype(np.int32) + rng.integers(-12, 13, (n, n, 3)), 0, 255)
    img[..., 3] = np.where(on, alpha_a, alpha_b)
    return img


def textured_room(threads=None):
    """A room whose materials use every texture slot of GpuMaterial (BaseColor sRGB with alpha, MetallicRoughness, Normal,
    Emissive, Transmission), all three wrap modes and non-square / non-power-of-two sizes; texcoords run outside [0, 1]."""
    scene = Scene()
    rng = np.random.default_rng(5)
    t_floor = scene.add_texture(_checker(64, 8, (200, 190, 170), (60, 50, 40), seed=1), srgb=True)
    t_wall = scene.add_texture(_checker(48, 6, (120, 140, 200), (200, 120, 90), seed=2)[:32], srgb=True, wrap_s=33648, wrap_t=33071)
    nrm = np.zeros((40, 56, 4), np.uint8)
    yy, xx = np.mgrid[0:40, 0:56]
    nrm[..., 0] = (127.5 + 90 * np.sin(xx * 0.6)).astype(np.uint8)
    nrm[..., 1] = (127.5 + 90 * np.cos(yy * 0.5)).astype(np.uint8)
    nrm[..., 2:] = 255
    t_normal = scene.add_texture(nrm)
    mr = rng.integers(0, 256, (16, 16, 4)).astype(np.uint8)
    t_mr = scene.add_texture(mr, wrap_s=33071, wrap_t=33648)
    t_cut = scene.add_texture(_checker(32, 4, (30, 160, 60), (30, 160, 60), alpha_a=255, alpha_b=20, seed=3), srgb=True)
    t_blend = scene.add_texture(_checker(32, 2, (220, 60, 200), (60, 200, 220), alpha_a=200, alpha_b=90, seed=4), srgb=True)
    t_emis = scene.add_texture(_checker(24, 3, (255, 220, 160), (10, 10, 10), seed=5), srgb=True)
    t_trans = scene.add_texture(_checker(20, 5, (255, 255, 255), (40, 40, 40), seed=6))
    specs = [
        dict(color=(1.0, 1.0, 1.0)),                                              # 0 floor: base colour texture
        dict(color=(0.9, 0.9, 0.9), metallic=1.0, roughness=1.0),                 # 1 wall: base + normal + metallic/roughness
        dict(color=(1.0, 1.0, 1.0), cutoff=0.5),                                  # 2 cutout card
        dict(color=(1.0, 1.0, 1.0, 0.9), cutoff=2.0),                             # 3 blended card
        dict(color=(0.2, 0.2, 0.2), emissive=(9.0, 8.0, 6.0)),                    # 4 emissive panel
        dict(color=(0.95, 0.95, 1.0), transmission=1.0, roughness=0.05, ior=1.45),  # 5 pane with a transmission texture
        dict(color=(0.75, 0.75, 0.75)),                                           # 6 untextured ceiling / side walls
        dict(color=(1, 1, 1), emissive=(14, 14, 14)),                             # 7 lamp
    ]
    meshes, mats = _materials(specs)
    mats["BaseColorTexture"][0] = t_floor
    mats["BaseColorTexture"][1], mats["NormalTexture"][1], mats["MetallicRoughnessTexture"][1] = t_wall, t_normal, t_mr
    mats["BaseColorTexture"][2] = t_cut
    mats["BaseColorTexture"][3] = t_blend
    mats["EmissiveTexture"][4] = t_emis
    mats["TransmissionTexture"][5] = t_trans
    meshes["NormalMapStrength"][1] = 0.8
    a = _Assembler()
    a.add(grid([-3, 0, -3], [6, 0, 0], [0, 0, 6], 6, 6), 0)
    a.add(grid([-3, 0, -3], [6, 0, 0], [0, 4, 0], 6, 4), 1)
    a.add(quad([-1.6, 0.2, -1.0], [-0.4, 0.2, -1.0], [-0.4, 1.8, -1.0], [-1.6, 1.8, -1.0]), 2)
    a.add(quad([0.3, 0.3, -0.4], [1.5, 0.3, -0.9], [1.5, 1.7, -0.9], [0.3, 1.7, -0.4]), 3)
    a.add(quad([-2.9, 1.0, -2.0], [-2.9, 1.0, 0.0], [-2.9, 2.2, 0.0], [-2.9, 2.2, -2.0]), 4)
    a.add(quad([-0.8, 0.1, 0.9], [0.8, 0.1, 0.9], [0.8, 1.5, 0.9], [-0.8, 1.5, 0.9]), 5)
    a.add(quad([-3, 4, -3], [3, 4, -3], [3, 4, 3], [-3, 4, 3]), 6)
    a.add(quad([-3, 0, -3], [-3, 0, 3], [-3, 4, 3], [-3, 4, -3]), 6)
    a.add(quad([3, 0, 3], [3, 0, -3], [3, 4, -3], [3, 4, 3]), 6)
    a.add(quad([-0.7, 3.98, -0.7], [0.7, 3.98, -0.7], [0.7, 3.98, 0.7], [-0.7, 3.98, 0.7]), 7)
    pos = np.concatenate(a.pos)
    uv = np.stack([pos[:, 0] * 0.61 + pos[:, 2] * 0.43 - 0.3, pos[:, 1] * 0.57 + pos[:, 2] * 0.29 - 0.7], 1).astype(np.float32)
    model = Model(pos, np.concatenate(a.idx), np.concatenate(a.mesh), texcoords=uv, meshes=meshes, materials=mats, name="textured_room")
    scene.add(model, threads=threads)
    scene.add_light((1.5, 2.6, 1.2), (25.0, 24.0, 22.0), 0.25)
    cam = dict(position=(0.2, 1.5, 4.6), view_dir=(-0.05, -0.08, -1.0), fov_y_deg=62.0)
    return scene, cam



def texturize(scene, size=512, count=8, seed=11):
    """Give every material of an already built scene a base-colour (sRGB) and a metallic-roughness texture out of `count`
    procedural size x size images and planar texcoords, e.g. to measure the textured shade path on the bench atrium."""
    rng = np.random.default_rng(seed)
    handles = []
    for k in range(count):
        img = _checker(size, 8 << (k % 3), rng.integers(60, 255, 3), rng.integers(20, 200, 3), seed=seed + k)
        handles.append((scene.add_texture(img, srgb=True), scene.add_texture(rng.integers(0, 256, (size // 4, size // 4, 4)).astype(np.uint8))))
    for m in range(len(scene.materials)):
        scene.materials["BaseColorTexture"][m], scene.materials["MetallicRoughnessTexture"][m] = handles[m % count]
    x, y, z = scene.positions["x"], scene.positions["y"], scene.positions["z"]
    scene.vertices["TexCoord"][:, 0] = x * 0.23 + z * 0.17
    scene.vertices["TexCoord"][:, 1] = y * 0.21 + z * 0.11 - x * 0.05
    return scene


# --------------------------------------------------------------------------- real Sponza (IDKEngine's Resource/Models/SponzaCompressed/Sponza.gltf)
SPONZA_PLACEMENT = (1.815, 0.0, (0.0, -1.0, 0.0))          # trs_matrix(scale, yaw, translation) of SRC/Application.cs:448
SPONZA_CAMERA = dict(position=(7.63, 2.71, 0.8), view_dir=tuple(view_dir_from_angles(360.0 - 165.4, 90.0 - 7.4)), fov_y_deg=102.0)


def load_gltf_geometry(path):
    """Minimal glTF reader: float32 POSITION/NORMAL/TEXCOORD_0 + integer indices, factor-only materials."""
    with open(path) as f:
        g = json.load(f)
    base = os.path.dirname(path)
    bufs = [np.fromfile(os.path.join(base, b["uri"]), np.uint8) for b in g["buffers"]]
    ctype = {5120: np.int8, 5121: np.uint8, 5122: np.int16, 5123: np.uint16, 5125: np.uint32, 5126: np.float32}
    ncomp = {"SCALAR": 1, "VEC2": 2, "VEC3": 3, "VEC4": 4}

    def acc(i):
        a = g["accessors"][i]
        bv = g["bufferViews"][a["bufferView"]]
        dt = np.dtype(ctype[a["componentType"]])
        n = ncomp[a["type"]]
        off = bv.get("byteOffset", 0) + a.get("byteOffset", 0)
        stride = bv.get("byteStride", 0) or dt.itemsize * n
        raw = bufs[bv["buffer"]]
        if stride == dt.itemsize * n:
            arr = raw[off:off + a["count"] * stride].view(dt).reshape(a["count"], n)
        else:
            arr = np.stack([raw[off + k * stride: off + k * stride + dt.itemsize * n].view(dt) for k in range(a["count"])])
        if a.get("normalized", False) and dt != np.float32:
            arr = arr.astype(np.float32) / np.iinfo(dt).max
        return arr

    pos, nrm, uv, idx, tri_mesh, mesh_mat = [], [], [], [], [], []
    nv = 0
    for mesh in g["meshes"]:
        for prim in mesh["primitives"]:
            p = acc(prim["attributes"]["POSITION"]).astype(np.float32)
            i = acc(prim["indices"]).astype(np.uint32).reshape(-1, 3)
            n = acc(prim["attributes"]["NORMAL"]).astype(np.float32) if "NORMAL" in prim["attributes"] else None
            t = acc(prim["attributes"]["TEXCOORD_0"]).astype(np.float32) if "TEXCOORD_0" in prim["attributes"] else np.zeros((len(p), 2), np.float32)
            pos.append(p)
            nrm.append(n)
            uv.append(t)
            idx.append(i + nv)
            tri_mesh.append(np.full(len(i), len(mesh_mat), np.int32))
            mesh_mat.append(prim.get("material", 0))
            nv += len(p)
    return g, pos, nrm, uv, idx, tri_mesh, mesh_mat


def sponza_reference(path, threads=None):
    """Config 2 with the reference's real Sponza.bin geometry (262,267 triangles), read from the Sponza.gltf at `path`.
    Materials from glTF factors with metallic=0, roughness=0.8 (SURVEY 8d 'constant-texture semantics'); emissive biases
    per SRC/Application.cs:449-457."""
    g, pos, nrm, uv, idx, tri_mesh, mesh_mat = load_gltf_geometry(path)
    gm = g.get("materials", [{}])
    mats = gt.default_material(len(gm))
    for k, m in enumerate(gm):
        pbr = m.get("pbrMetallicRoughness", {})
        mats["BaseColorFactor"][k] = gt.pack_unorm4x8(np.array(pbr.get("baseColorFactor", [1, 1, 1, 1])))
        mats["MetallicFactor"][k] = 0.0
        mats["RoughnessFactor"][k] = 0.8
        mats["EmissiveFactor"][k] = m.get("emissiveFactor", [0, 0, 0])
        mode = m.get("alphaMode", "OPAQUE")
        mats["AlphaCutoff"][k] = 0.0 if mode == "OPAQUE" else (m.get("alphaCutoff", 0.5) if mode == "MASK" else 2.0)
        mats["IsDoubleSided"][k] = 1 if m.get("doubleSided", False) else 0
    meshes = gt.default_mesh(len(mesh_mat))
    meshes["MaterialId"] = np.array(mesh_mat, np.int32)
    for mid, bias in {63: 10.0, 70: 20.0, 3: 12.0, 99: 15.0, 97: 9.0, 42: 20.0, 38: 20.0, 40: 20.0}.items():
        if mid < len(meshes):
            meshes["EmissiveBias"][mid] = bias
    normals = None if any(n is None for n in nrm) else np.concatenate(nrm)
    model = Model(np.concatenate(pos), np.concatenate(idx), np.concatenate(tri_mesh), normals=normals,
                  texcoords=np.concatenate(uv), meshes=meshes, materials=mats,
                  model_matrix=trs_matrix(*SPONZA_PLACEMENT), name="sponza")
    scene = Scene().add(model, threads=threads)
    return scene, dict(SPONZA_CAMERA)


def camera_frame(cam, width, height):
    return make_per_frame_data(cam["position"], cam["view_dir"], width, height, cam.get("fov_y_deg", 102.0))
