"""lgb_trace_rays (the round-1 BVH traversal: traverse / node_loop / leaf_prims) against the oracle's trace_rays, ray by ray, on
rays no camera makes: every direction octant, signed-zero and in-plane directions, extreme |d|, origins on and inside primitives,
rays grazing sphere silhouettes and cuboid / mesh edges to a few ulps, and origins on the faces and corners of the box the f32 error
bound is derived from (DESIGN.md §4) and up to one box extent outside it; origins 10^3 - 10^5 extents away are refused.

Every family is a seeded numpy generator in this file.  Each carries a non-vacuity check that runs on the oracle alone (the
`not gpu` tests below), so a generator that stops producing what it claims fails without a GPU.

Bars, per ray: same id and t bit-equal.  Never allowed: a device miss where the oracle hits, a device t greater than the oracle's,
the same id with a different t.  The one allowed difference (DESIGN.md §4, "What stays outside exact reproduction") is the
reference's own f64 node test dropping a box along its boundary: then the device may report a hit the oracle lacks, or another
equal-t primitive -- only for grazing (F3), in-plane (F4) and on-surface (F5) rays and rays aimed like F3 (F7, F7b), and only if the oracle's exact test of the device's primitive
gives the device's t bit for bit and that t is not beyond the oracle's.  Normals of equal ids agree to 1e-12 and face the same way
wherever |n.d| > 1e-9."""
import functools
import math
import zlib

import numpy as np
import pytest

from lasgun_b200 import scenes
from lasgun_b200.api import Aggregate, Material, ObjData, Scene

MISS = 0xFFFFFFFF
N = 2000                      # rays per family and scene (F1 / F2; the others are of the same order)
PARITY = ("F1", "F2", "F3", "F4", "F5", "F6", "F7b")   # origins inside the error box
FAMILIES = PARITY + ("F7n",)                           # F7n: origins outside it, less than one box extent away
# Where the reference's node test can drop a box along its boundary: grazing and in-plane rays, rays aimed like them (F7n, F7b),
# and rays that start exactly on a surface (F5), which lies on the boundary of its node box when the primitive is flat (a floor).
ALLOWED = ("F3", "F4", "F5", "F7n", "F7b")


# ------------------------------------------------------------------ scenes
def plain_scene(offset=(0.0, 0.0, 0.0), scale=1.0, seed=1):
    """Spheres, cuboids and a mesh in one plain space, built in numpy around `offset` at `scale` (so M and the error bound change)."""
    rng = np.random.default_rng(seed)
    off = np.array(offset, np.float64)
    sc = Scene()
    sc.set_perspective_camera(50.0).look_at((off + scale * np.array([0.3, 0.8, 4.0])).tolist(), off.tolist(), [0.0, 1.0, 0.0])
    sc.add_point_light((off + scale * np.array([2.0, 3.0, 3.0])).tolist(), [0.8, 0.8, 0.8], [1.0, 0.0, 0.0])
    pal = scenes._cube_palette()
    cen = off + scale * rng.uniform(-1.5, 1.5, (300, 3))
    sc.root.add_spheres(cen, scale * rng.uniform(0.03, 0.15, 300), pal, np.arange(300) % 8)
    for _ in range(40):
        lo = off + scale * rng.uniform(-1.5, 1.3, 3)
        sc.root.add_box(lo.tolist(), (lo + scale * rng.uniform(0.05, 0.3, 3)).tolist(), pal[3])
    m = scenes.mesh_grid(20, 0.6)
    pos = (m.positions.astype(np.float64) * scale + off + scale * np.array([0.2, -0.3, 0.1])).astype(np.float32)
    sc.root.add_obj_of(sc.add_obj(ObjData(pos, m.faces)), pal[5])
    sc.root.add_box((off + scale * np.array([-2.0, -1.8, -2.0])).tolist(), (off + scale * np.array([2.0, -1.6, 2.0])).tolist(), pal[6])
    return sc


def twins_scene():
    """test_device_built_bvh_degenerate's construction: 12 000 positions, each a sphere, the same sphere again and a cube inside
    them (36 000 primitives: the device-side builder, exact-t ties between the twins in every direction octant)."""
    rng = np.random.default_rng(0x5EED0C02)
    sc = Scene()
    sc.set_perspective_camera(45.0).look_at([0.0, 0.0, 160.0], [0.0, 0.0, 0.0], [0.0, 1.0, 0.0])
    sc.add_point_light([80.0, 120.0, 150.0], [0.8, 0.8, 0.8], [1.0, 0.0, 0.0])
    pos = -50.0 + 100.0 * rng.random((12000, 3)); rad = 0.6 + 0.6 * rng.random(12000)
    pal = [Material.plastic([0.8, 0.3, 0.2], [0.4, 0.4, 0.4], 0.2), Material.plastic([0.2, 0.7, 0.3], [0.3, 0.3, 0.3], 0.3)]
    sc.root.add_spheres(np.concatenate([pos, pos]), np.concatenate([rad, rad]), pal, np.arange(24000) % 2)
    for p, r in zip(pos, rad):
        sc.root.add_cube((p - 0.4 * r).tolist(), float(0.8 * r), pal[0])
    return sc


SCENES = {
    "mixed": lambda: scenes.mixed4k(mesh_n=48, nspheres=3000, res=(64, 36), supersampling=0)[0],
    "simple": lambda: scenes.simple("b", 0, 64)[0],
    "offset": lambda: plain_scene((3e4, -2e5, 1e3), 1.0, seed=2),
    "small": lambda: plain_scene((0.0, 0.0, 0.0), 1e-3, seed=3),
    "large": lambda: plain_scene((0.0, 0.0, 0.0), 1e3, seed=4),
    "coincident": lambda: scenes.coincident_planes(res=(64, 48))[0],
    "twins": twins_scene,
    "nested": lambda: scenes.nested_groups((64, 48))[0],
    "nested_root": lambda: scenes.nested_groups((64, 48), transformed_root=True)[0],
    "cornell_groups": lambda: scenes.cornell_groups((64, 64), 0)[0],
    "materials_grouped": lambda: scenes.materials((64, 48), 0, grouped=True)[0],
}
BIG = ("coincident", "twins")          # >= 32 768 primitives: device-built tree, compared with the host-built one too
FAR = ("mixed", "simple", "offset", "small", "large", "twins")


# ------------------------------------------------------------------ geometry of the scene's plain space (canonical ids as the oracle numbers them)
def plain_geometry(sc):
    """World-space spheres, cuboids and triangles of every level without a transform, with their canonical ids (depth-first in
    content order, as Accel::from numbers them), and the shared edges / vertices of the meshes among them."""
    g = {"sph": [], "sph_id": [], "box": [], "box_id": [], "tri": [], "tri_id": [], "edge": [], "vert": []}
    nid = 0

    def walk(agg, plain):
        nonlocal nid
        plain = plain and not agg.transforms
        for item in agg.contents:
            k = item[0]
            if k == "sphere":
                if plain:
                    g["sph"].append([*item[1], item[2]]); g["sph_id"].append(nid)
                nid += 1
            elif k == "spheres":
                n = len(item[2])
                if plain:
                    g["sph"] += np.concatenate([item[1], item[2][:, None]], axis=1).tolist(); g["sph_id"] += list(range(nid, nid + n))
                nid += n
            elif k in ("cube", "box"):
                a = np.array(item[1], np.float64)
                b = a + item[2] if k == "cube" else np.array(item[2], np.float64)
                if plain:
                    g["box"].append(np.concatenate([np.minimum(a, b), np.maximum(a, b)]).tolist()); g["box_id"].append(nid)
                nid += 1
            elif k == "mesh":
                m = sc.meshes[item[1].index]
                faces = np.asarray(m.faces, np.int64).reshape(-1, 3)
                if plain:
                    p = np.asarray(m.positions, np.float32).astype(np.float64)
                    tri = p[faces]
                    area = np.linalg.norm(np.cross(tri[:, 1] - tri[:, 0], tri[:, 2] - tri[:, 0]), axis=1)
                    g["tri"] += tri.reshape(-1, 9).tolist(); g["tri_id"] += list(range(nid, nid + len(faces)))
                    owners = {}
                    for f, (a, b, c) in enumerate(faces):
                        for e in ((a, b), (b, c), (c, a)):
                            owners.setdefault((min(e), max(e)), []).append(f)
                    for (a, b), fs in owners.items():
                        if len(fs) == 2 and area[fs[0]] > 0 and area[fs[1]] > 0 and set(faces[fs[0]]) != set(faces[fs[1]]):
                            ca, cb = (int(next(v for v in faces[f] if v not in (a, b))) for f in fs)
                            g["edge"].append([*p[a], *p[b], *p[ca], *p[cb], nid + fs[0], nid + fs[1]])
                    used = np.unique(faces[area > 0])
                    g["vert"] += p[used].tolist()
                nid += len(faces)
            elif k == "group":
                walk(item[1], plain)
    walk(sc.root, True)
    return {k: np.array(v, np.float64) for k, v in g.items()}


def error_box(flat):
    """The world box lgb_scene_create derives the f32 error bound from (lgb_api.cu): the reference root box, through the root
    transform, and the camera origin.  Same operations in the same order, so its faces are the library's to the bit."""
    d = flat.desc
    node = flat.nodes()[0]
    rlo, rhi = node["lo"].astype(np.float64), node["hi"].astype(np.float64)
    lo, hi = rlo.copy(), rhi.copy()
    if not d.root.identity:
        m = list(d.root.m)
        for r in range(3):
            l = h = m[12 + r]
            for c in range(3):
                a, b = m[4 * c + r] * rlo[c], m[4 * c + r] * rhi[c]
                l += min(a, b); h += max(a, b)
            lo[r], hi[r] = l, h
    slack = 2.5 * abs(d.camera.image_plane_height) * abs(d.camera.pixel_separation)
    for k in range(3):
        if math.isfinite(d.camera.origin[k]):
            lo[k] = min(lo[k], d.camera.origin[k] - slack); hi[k] = max(hi[k], d.camera.origin[k] + slack)
    return lo, hi


# ------------------------------------------------------------------ ray families
def unit(rng, n):
    v = rng.normal(size=(n, 3))
    return v / np.linalg.norm(v, axis=1, keepdims=True)


def in_box(rng, lo, hi, n):
    return lo + (hi - lo) * rng.random((n, 3))


def surface_points(rng, g, n, hits):
    """Points on random primitives: a sphere's surface, a cuboid's face, a triangle by barycentrics, and (for content inside
    transformed groups) hit points the oracle found."""
    pools = [k for k in ("sph", "box", "tri") if len(g[k])] + (["hit"] if len(hits) else [])
    kind = rng.integers(0, len(pools), n)
    out = np.zeros((n, 3))
    for j, pool in enumerate(pools):
        sel = np.nonzero(kind == j)[0]
        if pool == "sph":
            s = g["sph"][rng.integers(0, len(g["sph"]), len(sel))]
            out[sel] = s[:, :3] + s[:, 3:4] * unit(rng, len(sel))
        elif pool == "box":
            b = g["box"][rng.integers(0, len(g["box"]), len(sel))]
            p = b[:, :3] + (b[:, 3:] - b[:, :3]) * rng.random((len(sel), 3))
            ax = rng.integers(0, 3, len(sel)); side = rng.integers(0, 2, len(sel))
            p[np.arange(len(sel)), ax] = b[np.arange(len(sel)), ax + 3 * side]
            out[sel] = p
        elif pool == "tri":
            t = g["tri"][rng.integers(0, len(g["tri"]), len(sel))].reshape(-1, 3, 3)
            w = rng.random((len(sel), 3)); w /= w.sum(axis=1, keepdims=True)
            out[sel] = np.einsum("ni,nij->nj", w, t)
        else:
            out[sel] = hits[rng.integers(0, len(hits), len(sel))]
    return out


def grazing(rng, g, lo, hi, n, origins=None):
    """F3: towards sphere silhouettes at r (1 + k 2^-40), k in [-8, 8]; towards cuboid edges and corners; towards shared edges and
    vertices of meshes.  Returns rays, kind (0 sphere, 1 cuboid, 2 mesh edge, 3 mesh vertex) and the target's id / ids."""
    kinds = [k for k, key in ((0, "sph"), (1, "box"), (2, "edge"), (3, "vert")) if len(g[key])]
    if not kinds:                                     # (a transformed root: no world-space geometry to aim at)
        return np.zeros((0, 6)), np.zeros(0, np.int64), np.zeros((0, 2), np.int64), np.zeros(0, np.int64)
    kind = np.array(kinds)[rng.integers(0, len(kinds), n)]
    o = in_box(rng, lo, hi, n) if origins is None else origins
    tgt = np.zeros((n, 3)); ids = np.full((n, 2), -1, np.int64); ks = np.zeros(n, np.int64)
    for k in kinds:
        sel = np.nonzero(kind == k)[0]
        m = len(sel)
        if k == 0:
            j = rng.integers(0, len(g["sph"]), m); s = g["sph"][j]; c, r = s[:, :3], s[:, 3]
            e = o[sel] - c; L = np.linalg.norm(e, axis=1)
            ok = L > 1.05 * r
            e_hat = e / L[:, None]
            u = np.cross(e_hat, unit(rng, m)); u /= np.linalg.norm(u, axis=1, keepdims=True)
            with np.errstate(invalid="ignore"):
                T = c + (r * r / L)[:, None] * e_hat + (r * np.sqrt(np.maximum(1.0 - (r / L) ** 2, 0.0)))[:, None] * u
            kk = rng.integers(-8, 9, m)
            tgt[sel] = c + (T - c) * (1.0 + kk * 2.0 ** -40)[:, None]
            tgt[sel[~ok]] = np.nan
            ids[sel, 0] = g["sph_id"][j]; ks[sel] = kk
        elif k == 1:
            j = rng.integers(0, len(g["box"]), m); b = g["box"][j]
            p = b[:, :3] + (b[:, 3:] - b[:, :3]) * rng.random((m, 3))
            side = rng.integers(0, 2, (m, 3))
            fixed = np.ones((m, 3), bool)
            free = rng.integers(0, 4, m)                      # 0..2: an edge along that axis; 3: a corner
            fixed[free < 3, free[free < 3]] = False
            p = np.where(fixed, np.where(side == 1, b[:, 3:], b[:, :3]), p)
            kk = rng.integers(-8, 9, m)
            ext = np.max(b[:, 3:] - b[:, :3], axis=1)
            tgt[sel] = p + (kk * 2.0 ** -40 * ext)[:, None] * unit(rng, m) * (rng.random(m) < 0.5)[:, None]
            ids[sel, 0] = g["box_id"][j]
        elif k == 2:
            e = g["edge"][rng.integers(0, len(g["edge"]), m)]
            s = rng.uniform(0.05, 0.95, m)[:, None]
            tgt[sel] = e[:, 0:3] + s * (e[:, 3:6] - e[:, 0:3])
            ids[sel] = e[:, 12:14].astype(np.int64)
            # 1 where the ray crosses the surface at the edge (the third vertices lie on opposite sides of the plane of the edge
            # and d), 0 at a silhouette, where it passes both triangles or neither
            nrm = np.cross(e[:, 3:6] - e[:, 0:3], tgt[sel] - o[sel])
            ks[sel] = (np.sum(nrm * (e[:, 6:9] - e[:, 0:3]), axis=1) * np.sum(nrm * (e[:, 9:12] - e[:, 0:3]), axis=1) < 0)
        else:
            tgt[sel] = g["vert"][rng.integers(0, len(g["vert"]), m)]
    d = tgt - o
    keep = np.all(np.isfinite(d), axis=1) & (np.linalg.norm(d, axis=1) > 0)
    return np.concatenate([o, d], axis=1)[keep], kind[keep], ids[keep], ks[keep]


def signed_zero_rays(rng, g, lo, hi, base):
    """F4: aimed rays with one or two direction components set to exactly +0.0 or -0.0, and rays inside the face planes of cuboids
    and through mesh vertex coordinates (origin on the plane, the direction component across it a signed zero)."""
    n = len(base)
    r = base.copy()
    nz = rng.integers(1, 3, n)
    for i in range(n):
        axes = rng.choice(3, nz[i], replace=False)
        r[i, 3 + axes] = np.where(rng.random(len(axes)) < 0.5, 0.0, -0.0)
    extra = []
    if len(g["box"]):
        b = g["box"][rng.integers(0, len(g["box"]), n // 2)]
        ax = rng.integers(0, 3, n // 2); side = rng.integers(0, 2, n // 2)
        o = in_box(rng, lo, hi, n // 2); tgt = b[:, :3] + (b[:, 3:] - b[:, :3]) * rng.random((n // 2, 3))
        idx = np.arange(n // 2)
        o[idx, ax] = b[idx, ax + 3 * side]; tgt[idx, ax] = o[idx, ax]
        d = tgt - o
        d[idx, ax] = np.where(rng.random(n // 2) < 0.5, 0.0, -0.0)
        extra.append(np.concatenate([o, d], axis=1))
    if len(g["vert"]):
        v = g["vert"][rng.integers(0, len(g["vert"]), n // 2)]
        ax = rng.integers(0, 3, n // 2); idx = np.arange(n // 2)
        o = in_box(rng, lo, hi, n // 2); o[idx, ax] = v[idx, ax]
        d = v - o
        d[idx, ax] = np.where(rng.random(n // 2) < 0.5, 0.0, -0.0)
        extra.append(np.concatenate([o, d], axis=1))
    return np.concatenate([r] + extra)


def on_inside_rays(rng, g, hits, hit_dirs, hit_ng):
    """F5: origins at sphere centres, inside cuboids, and exactly at hit points with the incoming and the reflected direction."""
    out = []
    if len(g["sph"]):
        s = g["sph"][rng.integers(0, len(g["sph"]), N // 4)]
        out.append(np.concatenate([s[:, :3], unit(rng, len(s))], axis=1))
    if len(g["box"]):
        b = g["box"][rng.integers(0, len(g["box"]), N // 4)]
        out.append(np.concatenate([b[:, :3] + (b[:, 3:] - b[:, :3]) * rng.uniform(0.01, 0.99, (len(b), 3)), unit(rng, len(b))], axis=1))
    if len(hits):
        j = rng.integers(0, len(hits), N // 2)
        d, n = hit_dirs[j], hit_ng[j]
        refl = d - 2.0 * np.sum(d * n, axis=1, keepdims=True) * n
        out.append(np.concatenate([hits[j], d], axis=1)); out.append(np.concatenate([hits[j], refl], axis=1))
    return np.concatenate(out)


MAGNITUDES = (-40, -20, -12.01, -12, -11.99, 0, 11.99, 12, 12.01, 20, 40)


def magnitude_rays(rng, base):
    """F6: |d| = 10^k for every k of MAGNITUDES, and single direction components of f64-subnormal (1e-310) and f32-subnormal
    (1e-40) size."""
    dh = base[:, 3:] / np.linalg.norm(base[:, 3:], axis=1, keepdims=True)
    k = np.array(MAGNITUDES)[np.arange(len(base)) % len(MAGNITUDES)]
    r = np.concatenate([base[:, :3], dh * (10.0 ** k)[:, None]], axis=1)
    tiny = base.copy()[: len(base) // 2]
    idx = np.arange(len(tiny)); ax = rng.integers(0, 3, len(tiny))
    tiny[idx, 3 + ax] = np.where(rng.random(len(tiny)) < 0.5, 1.0, -1.0) * np.where(idx % 2 == 0, 1e-310, 1e-40)
    return np.concatenate([r, tiny])


def far_origins(rng, g, lo, hi, n):
    """F7: origins 10^3 - 10^5 scene extents away, with coordinates no f32 represents, aimed as F3."""
    ext = float(np.max(hi - lo)); ctr = 0.5 * (lo + hi)
    o = ctr + unit(rng, n) * (ext * 10.0 ** rng.uniform(3, 5, n))[:, None]
    o += ext * 1e-3 * rng.random((n, 3))              # (random f64 bits below the f32 mantissa)
    return grazing(rng, g, lo, hi, n, origins=o)[0]


def shell_extent(lo, hi):
    """E of lgb_trace_rays: origins up to E outside the error box are traced, farther ones refused (same operations)."""
    M = max(float(np.abs(lo).max()), float(np.abs(hi).max()))
    return float(np.max(hi - lo)) + M * 2.0 ** -10


def near_outside_origins(rng, lo, hi, n):
    """F7n: origins outside the error box but less than one box extent away."""
    E = 0.95 * shell_extent(lo, hi)
    o = in_box(rng, lo - E, hi + E, 4 * n)
    o = o[~np.all((o >= lo) & (o <= hi), axis=1)]
    return o[:n]


def box_face_origins(rng, lo, hi, n):
    """Origins exactly on the faces, edges and corners of the error box."""
    o = in_box(rng, lo, hi, n)
    snap = rng.random((n, 3)) < np.array([[0.6, 0.45, 0.45]])
    side = rng.integers(0, 2, (n, 3))
    return np.where(snap, np.where(side == 1, hi, lo), o)


# ------------------------------------------------------------------ one case: scene, oracle, rays of every family, oracle results
class Case:
    pass


@functools.lru_cache(maxsize=None)
def case(name):
    from lasgun_b200 import _native as native
    from oracle import pyoracle
    c = Case()
    c.name = name
    c.sc = SCENES[name]()
    c.o = pyoracle.OracleScene(c.sc)
    c.flat = native.FlatScene(c.sc)
    c.lo, c.hi = error_box(c.flat)
    c.g = plain_geometry(c.sc)
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    lo, hi = c.lo, c.hi
    fam = {}
    fam["F1"] = np.concatenate([in_box(rng, lo, hi, N), unit(rng, N)], axis=1)
    ids1, t1, ng1, _ = c.o.trace_rays(fam["F1"], normals=True)
    hit = ids1 != MISS
    hits = fam["F1"][hit, :3] + t1[hit, None] * fam["F1"][hit, 3:]
    o2 = in_box(rng, lo, hi, N)
    d2 = surface_points(rng, c.g, N, hits) - o2
    d2 = d2 / np.linalg.norm(d2, axis=1, keepdims=True) * (10.0 ** rng.uniform(-3, 3, N))[:, None]
    fam["F2"] = np.concatenate([o2, d2], axis=1)
    ids2, t2, ng2, _ = c.o.trace_rays(fam["F2"], normals=True)
    h2 = ids2 != MISS
    c.f2_hit_frac = float(h2.mean())
    hp = fam["F2"][h2, :3] + t2[h2, None] * fam["F2"][h2, 3:]
    fam["F3"], c.f3_kind, c.f3_ids, c.f3_k = grazing(rng, c.g, lo, hi, N)
    fam["F4"] = signed_zero_rays(rng, c.g, lo, hi, fam["F2"][: N // 2])
    fam["F5"] = on_inside_rays(rng, c.g, hp, fam["F2"][h2, 3:], ng2[h2])
    c.f5_src = ids2[h2]
    fam["F6"] = magnitude_rays(rng, fam["F2"][: N // 2])
    o7 = box_face_origins(rng, lo, hi, N // 2)
    r7 = grazing(rng, c.g, lo, hi, N // 2, origins=o7)[0]
    r7b = np.concatenate([o7, surface_points(rng, c.g, N // 2, hits) - o7], axis=1)
    fam["F7b"] = np.concatenate([r7, r7b])
    # every parity family stays inside the error box (a hit point on the scene's outer face can round one ulp outside it)
    for k in PARITY:
        r = fam[k]
        fam[k] = r[np.all((r[:, :3] >= lo) & (r[:, :3] <= hi), axis=1)]
    o7n = near_outside_origins(rng, lo, hi, N)
    fam["F7n"] = np.concatenate([grazing(rng, c.g, lo, hi, N // 2, origins=o7n[: N // 2])[0],
                                 np.concatenate([o7n[N // 2:], surface_points(rng, c.g, len(o7n) - N // 2, hits) - o7n[N // 2:]], axis=1)])
    fam["F7"] = far_origins(rng, c.g, lo, hi, N // 2) if name in FAR else np.zeros((0, 6))
    c.fam = fam
    c.ref = {k: c.o.trace_rays(v, normals=True) for k, v in fam.items()}
    return c


# ------------------------------------------------------------------ the classifier
def classify(c, family, rays, dev, ref):
    """Per-ray comparison of device and oracle results: counts of every outcome, and the first offending rays."""
    di, dt, dng, dns = dev
    ri, rt, rng_, rns = ref
    same = (di == ri) & (dt.view(np.uint64) == rt.view(np.uint64))
    cnt = {"rays": len(rays), "hits": int((ri != MISS).sum()), "diff": int((~same).sum()), "allowed": 0,
           "miss_where_oracle_hits": 0, "t_greater": 0, "same_id_t_differs": 0, "other": 0, "normal_diff": 0, "facing_flip": 0}
    bad = []
    for i in np.nonzero(~same)[0]:
        o, d = rays[i, :3], rays[i, 3:]
        if di[i] == MISS and ri[i] != MISS:
            why = "miss_where_oracle_hits"
        elif di[i] == ri[i]:
            why = "same_id_t_differs"
        elif ri[i] != MISS and dt[i] > rt[i]:
            why = "t_greater"
        else:
            rt_dev = c.o.retest(int(di[i]), o, d)
            ok = family in ALLOWED and np.float64(rt_dev).view(np.uint64) == dt[i].view(np.uint64) and dt[i] <= rt[i]
            why = "allowed" if ok else "other"
        cnt[why] += 1
        if why != "allowed" and len(bad) < 4:
            bad.append((why, rays[i].tolist(), int(di[i]), float(dt[i]), int(ri[i]), float(rt[i])))
    both = (di == ri) & (ri != MISS)
    if both.any():
        nd = np.maximum(np.abs(dng[both] - rng_[both]).max(axis=1), np.abs(dns[both] - rns[both]).max(axis=1))
        cnt["normal_diff"] = int((nd > 1e-12).sum())
        dh = rays[both, 3:] / np.linalg.norm(rays[both, 3:], axis=1, keepdims=True)
        flips = 0
        for dn, rn in ((dng[both], rng_[both]), (dns[both], rns[both])):
            a, b = np.sum(dn * dh, axis=1), np.sum(rn * dh, axis=1)
            flips += int(((np.abs(b) > 1e-9) & (np.sign(a) != np.sign(b))).sum())
        cnt["facing_flip"] = flips
        if cnt["normal_diff"] and len(bad) < 6:
            j = np.nonzero(both)[0][np.argmax(nd)]
            bad.append(("normal", rays[j].tolist(), dng[j].tolist(), rng_[j].tolist(), dns[j].tolist(), rns[j].tolist()))
    return cnt, bad


def violations(family, cnt):
    v = cnt["miss_where_oracle_hits"] + cnt["t_greater"] + cnt["same_id_t_differs"] + cnt["other"] + cnt["normal_diff"] + cnt["facing_flip"]
    return v + (cnt["allowed"] if family not in ALLOWED else 0)


def report(name, table, bad):
    lines = [f"scene {name}:"] + [f"  {k}: {v}" for k, v in table.items()] + [f"  e.g. {b}" for b in bad[:8]]
    return "\n".join(lines)


# ------------------------------------------------------------------ non-vacuity: the oracle alone (no GPU)
@pytest.mark.parametrize("name", sorted(SCENES))
def test_ray_families_are_not_vacuous(native, oracle, name):
    c = case(name)
    f = c.fam
    assert all(len(f[k]) >= N // 3 for k in PARITY if k != "F3" or len(c.g["sph"]) + len(c.g["box"])), {k: len(v) for k, v in f.items()}
    # F1: every direction octant carries >= 5 % of the rays
    octs = (np.signbit(f["F1"][:, 3]) * 1 + np.signbit(f["F1"][:, 4]) * 2 + np.signbit(f["F1"][:, 5]) * 4).astype(int)
    assert np.bincount(octs, minlength=8).min() >= 0.05 * len(f["F1"])
    # F2: aimed rays mostly hit
    assert c.f2_hit_frac >= 0.8, c.f2_hit_frac
    # F3: grazing sphere rays both hit and miss their sphere; rays through a shared mesh edge hit one of its two triangles
    sph = np.nonzero(c.f3_kind == 0)[0]
    if len(sph):
        r = f["F3"]
        hit = np.array([np.isfinite(c.o.retest(int(c.f3_ids[i, 0]), r[i, :3], r[i, 3:])) for i in sph])
        assert 0 < hit.sum() < len(hit), (hit.sum(), len(hit))
        assert hit[c.f3_k[sph] > 2].mean() < hit[c.f3_k[sph] < -2].mean()
    edge = np.nonzero(c.f3_kind == 2)[0]
    if len(edge):
        r = f["F3"]
        nh = np.array([sum(np.isfinite(c.o.retest(int(c.f3_ids[i, k]), r[i, :3], r[i, 3:])) for k in range(2)) for i in edge])
        cross = c.f3_k[edge] == 1
        assert cross.sum() >= 50 and (nh[cross] >= 1).all() and (nh[cross] == 1).mean() >= 0.9, np.bincount(nh[cross])   # watertight
    # F4: both signs of zero on each axis
    z = f["F4"][:, 3:]
    for a in range(3):
        assert ((z[:, a] == 0) & np.signbit(z[:, a])).sum() > 10 and ((z[:, a] == 0) & ~np.signbit(z[:, a])).sum() > 10, a
    # F5: some rays hit their own surface again at a tiny t
    ids5, t5 = c.ref["F5"][0], c.ref["F5"][1]
    assert ((ids5 != MISS) & (t5 < 1e-6)).sum() > 0
    # F7b: origins on every face of the error box
    o7 = f["F7b"][:, :3]
    for a in range(3):
        assert (o7[:, a] == c.lo[a]).sum() > 10 and (o7[:, a] == c.hi[a]).sum() > 10, a
    o7n, E = f["F7n"][:, :3], shell_extent(c.lo, c.hi)
    assert len(o7n) >= N // 2 and not np.all((o7n >= c.lo) & (o7n <= c.hi), axis=1).any()
    assert np.all((o7n >= c.lo - E) & (o7n <= c.hi + E))
    if name in FAR:
        assert len(f["F7"]) >= N // 4 and not np.all((f["F7"][:, :3] >= c.lo) & (f["F7"][:, :3] <= c.hi), axis=1).any()


@pytest.mark.parametrize("name", BIG)
def test_exact_ties_in_every_octant(native, oracle, name):
    """The >= 32 768-primitive scenes: >= 100 aimed rays per direction octant meet two primitives at bit-identical t (the twin
    sphere, or the floor triangle listed twice).  coincident_planes' floor is seen from above only: four octants there."""
    c = case(name)
    r = np.concatenate([c.fam["F2"], c.fam["F1"]])
    ids, t = np.concatenate([c.ref["F2"][0], c.ref["F1"][0]]), np.concatenate([c.ref["F2"][1], c.ref["F1"][1]])
    twin = {"twins": lambda i: i + 12000 if i < 12000 else (i - 12000 if i < 24000 else -1),
            "coincident": lambda i: {0: 2, 2: 0, 1: 3, 3: 1}.get(int(i), -1)}[name]
    tie = np.zeros(len(r), bool)
    for i in np.nonzero(ids != MISS)[0]:
        j = twin(int(ids[i]))
        tie[i] = j >= 0 and np.float64(c.o.retest(j, r[i, :3], r[i, 3:])).view(np.uint64) == t[i].view(np.uint64)
    octs = (np.signbit(r[:, 3]) * 1 + np.signbit(r[:, 4]) * 2 + np.signbit(r[:, 5]) * 4).astype(int)
    per = np.bincount(octs[tie], minlength=8)
    need = range(8) if name == "twins" else [o for o in range(8) if o & 2]     # d.y < 0
    assert all(per[o] >= 100 for o in need), per


# ------------------------------------------------------------------ device against oracle
@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(SCENES))
def test_trace_rays_parity(native, oracle, gpu_ctx, name):
    c = case(name)
    dev = native.DeviceScene(gpu_ctx, c.flat)
    table, bad = {}, []
    try:
        for k in FAMILIES:
            out = dev.trace_rays(c.fam[k])
            table[k], b = classify(c, k, c.fam[k], out, c.ref[k])
            bad += b
    finally:
        dev.destroy()
    print(report(name, table, []))
    assert all(violations(k, table[k]) == 0 for k in FAMILIES), report(name, table, bad)


@pytest.mark.gpu
@pytest.mark.parametrize("name", FAR)
def test_trace_rays_refuses_far_origins(native, oracle, gpu_ctx, name):
    """F7: origins 10^3 - 10^5 scene extents away.  There rounding the origin to f32 moves the ray by more than the node padding
    allows, and the reference's own f64 sphere test loses so much to cancellation that its hits stray from the surface by more than
    the conservative culls cover: lgb_trace_rays refuses the batch (LGB_ERR_UNSUPPORTED) instead of returning silent wrong misses.
    Origins up to one box extent outside the error box are traced (F7n in test_trace_rays_parity); one ulp beyond is refused."""
    c = case(name)
    E = shell_extent(c.lo, c.hi)
    dev = native.DeviceScene(gpu_ctx, c.flat)
    try:
        with pytest.raises(native.LasgunError) as e:
            dev.trace_rays(c.fam["F7"])
        assert e.value.status == native.LGB_ERR_UNSUPPORTED and "outside the box" in str(e.value), e.value
        lo, hi = c.lo - E, c.hi + E
        corners = np.array([list(lo) + list(hi - lo), list(hi) + list(lo - hi)])       # the shell's corners, along its diagonal
        ids, t, _, _ = dev.trace_rays(corners)
        ri, rt = c.o.trace_rays(corners)
        assert np.array_equal(ids, ri) and np.array_equal(t.view(np.uint64), rt.view(np.uint64))
        for k in range(3):
            for r, v in ((corners[:1].copy(), np.nextafter(lo[k], -np.inf)), (corners[1:].copy(), np.nextafter(hi[k], np.inf))):
                r[0, k] = v
                with pytest.raises(native.LasgunError):
                    dev.trace_rays(r)
        with pytest.raises(native.LasgunError):
            dev.trace_rays(np.array([[np.nan, 0.0, 0.0, 1.0, 0.0, 0.0]]))
    finally:
        dev.destroy()


@pytest.mark.gpu
@pytest.mark.parametrize("name", BIG)
def test_device_and_host_built_trees_trace_alike(native, oracle, gpu_ctx, monkeypatch, name):
    """The device-built tree and the host-built tree of the same scene give identical ids and t on every ray of every family."""
    c = case(name)
    rays = np.concatenate([c.fam[k] for k in PARITY])
    dev = native.DeviceScene(gpu_ctx, c.flat)
    assert dev.verify()["ranks_ok"] == 1, "expected the device-side builder for this many primitives"
    a = dev.trace_rays(rays)
    dev.destroy()
    monkeypatch.setenv("LGB_HOST_BUILD", "1")
    host = native.DeviceScene(gpu_ctx, c.flat)
    assert host.verify()["ranks_ok"] == 0
    b = host.trace_rays(rays)
    host.destroy()
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1].view(np.uint64), b[1].view(np.uint64))
