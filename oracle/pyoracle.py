"""ctypes front end of the CPU oracle (oracle/lasgun_oracle.cpp).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and the
cpu_baseline / --impl reference legs of bench.py.  Never imported by lasgun_b200/.
It replays a `lasgun_b200.api.Scene` description into the oracle's own scene.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "liblasgun_oracle.so")
_lib = None

MISS = 0xFFFFFFFF


class Counters(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("node_tests", "sphere_tests", "cuboid_tests", "tri_tests", "primary",
                                          "primary_hits", "shadow", "shadow_occluded", "exact_ties")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


def build(force=False):
    src = os.path.join(_HERE, "lasgun_oracle.cpp")
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-s"] + (["-B"] if force else []))
    return _SO


def lib():
    global _lib
    if _lib is not None:
        return _lib
    build()
    L = C.CDLL(_SO)
    dp, fp, u32p, u64p, u8p, ip = (C.POINTER(C.c_double), C.POINTER(C.c_float), C.POINTER(C.c_uint32),
                                   C.POINTER(C.c_uint64), C.POINTER(C.c_uint8), C.POINTER(C.c_int))
    vp = C.c_void_p
    sig = {
        "orc_scene_new": (vp, []), "orc_scene_free": (None, [vp]),
        "orc_set_perspective_camera": (None, [vp, C.c_double]), "orc_set_orthographic_camera": (None, [vp, C.c_double]),
        "orc_look_at": (None, [vp, dp, dp, dp]), "orc_set_supersampling": (None, [vp, C.c_int]),
        "orc_set_ambient_light": (None, [vp, dp]), "orc_set_radial_background": (None, [vp, dp, dp, C.c_double]),
        "orc_add_point_light": (None, [vp, dp, dp, dp]),
        "orc_add_mesh": (C.c_int, [vp, fp, C.c_uint64, u32p, C.c_uint64, fp, C.c_uint64, u32p]),
        "orc_agg_new": (C.c_int, [vp]),
        "orc_agg_add_sphere": (None, [vp, C.c_int, dp, C.c_double, C.c_int, dp, dp, C.c_double, C.c_double]),
        "orc_agg_add_spheres": (None, [vp, C.c_int, C.c_uint64, dp, dp, C.c_int, ip, dp, dp, dp, dp, ip]),
        "orc_agg_add_cube": (None, [vp, C.c_int, dp, C.c_double, C.c_int, dp, dp, C.c_double, C.c_double]),
        "orc_agg_add_box": (None, [vp, C.c_int, dp, dp, C.c_int, dp, dp, C.c_double, C.c_double]),
        "orc_agg_add_mesh": (None, [vp, C.c_int, C.c_int, C.c_int, C.c_int, dp, dp, C.c_double, C.c_double]),
        "orc_set_max_recursion_depth": (None, [vp, C.c_uint32]),
        "orc_test_fresnel": (None, [C.c_int, C.c_double, dp, dp]), "orc_test_bsdf": (None, [C.c_int, dp, dp, C.c_double, C.c_double, dp, dp, dp, dp, dp, dp]),
        "orc_agg_add_group": (None, [vp, C.c_int, C.c_int]), "orc_agg_swap_backface": (None, [vp, C.c_int]),
        "orc_agg_translate": (None, [vp, C.c_int, dp]), "orc_agg_scale": (None, [vp, C.c_int, C.c_double, C.c_double, C.c_double]),
        "orc_agg_rotate_axis": (None, [vp, C.c_int, C.c_int, C.c_double]), "orc_agg_rotate": (None, [vp, C.c_int, C.c_double, dp]),
        "orc_accel_build": (vp, [vp]), "orc_accel_free": (None, [vp]), "orc_accel_build_ms": (C.c_double, [vp]),
        "orc_accel_prim_count": (C.c_uint32, [vp]),
        "orc_bvh_node_count": (C.c_int64, [vp, ip, C.c_int]), "orc_bvh_prim_count": (C.c_int64, [vp, ip, C.c_int]),
        "orc_bvh_dump": (C.c_int, [vp, ip, C.c_int, dp, u32p, u64p]),
        "orc_capture": (C.c_int, [vp, C.c_uint32, C.c_uint32, C.c_int, C.c_uint64, C.c_uint64, C.c_uint64, u8p, u32p, dp,
                                  u32p, dp, C.POINTER(Counters), dp]),
        "orc_test_sphere": (C.c_int, [dp, C.c_double, dp, dp, dp]), "orc_test_cuboid": (C.c_int, [dp, dp, dp, dp, dp]),
        "orc_test_mesh": (C.c_int, [fp, C.c_uint64, u32p, C.c_uint64, fp, C.c_uint64, u32p, dp, dp, dp, C.POINTER(C.c_int64)]),
        "orc_test_surface": (None, [C.c_double, dp, dp, dp, dp, dp]),
        "orc_retest_prim": (C.c_double, [vp, C.c_uint32, dp, dp]),
        "orc_camera_sample": (None, [vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, dp]),
        "orc_hardware_threads": (C.c_int, []),
        "orc_trace_rays": (None, [vp, dp, C.c_uint64, u32p, dp, dp, dp]),
        "orc_debug_li": (C.c_uint64, [vp, dp, dp, dp, C.c_uint64]),
    }
    for name, (res, args) in sig.items():
        f = getattr(L, name)
        f.restype, f.argtypes = res, args
    _lib = L
    return L


def _d3(v):
    return (C.c_double * 3)(*[float(c) for c in v])


def _ptr(a, ty):
    return a.ctypes.data_as(C.POINTER(ty)) if a is not None and a.size else None


class OracleScene:
    """Oracle-side scene + BVH (`Accel::from`, bvh.rs:135) built from an api.Scene description."""

    def __init__(self, scene):
        L = lib()
        self.desc = scene
        self.h = L.orc_scene_new()
        self.accel = None
        cam = scene.camera
        (L.orc_set_perspective_camera if cam.perspective else L.orc_set_orthographic_camera)(self.h, cam.param)
        if cam.look is not None:
            L.orc_look_at(self.h, _d3(cam.look[0]), _d3(cam.look[1]), _d3(cam.look[2]))
        L.orc_set_supersampling(self.h, cam.supersampling)
        L.orc_set_ambient_light(self.h, _d3(scene.ambient))
        L.orc_set_max_recursion_depth(self.h, int(scene.recursion))
        L.orc_set_radial_background(self.h, _d3(scene.background[0]), _d3(scene.background[1]), scene.background[2])
        for p, i, f in scene.lights:
            L.orc_add_point_light(self.h, _d3(p), _d3(i), _d3(f))
        self._keep = []
        for m in scene.meshes:
            self._keep.append(m)
            L.orc_add_mesh(self.h, _ptr(m.positions, C.c_float), len(m.positions), _ptr(m.faces, C.c_uint32), len(m.faces),
                           _ptr(m.normals, C.c_float), len(m.normals), _ptr(m.normal_faces, C.c_uint32))
        self._fill(0, scene.root)
        self.accel = L.orc_accel_build(self.h)
        if not self.accel:
            raise RuntimeError("oracle: BVH build does not terminate in the reference (empty aggregate or degenerate SAH split)")
        self.spp = cam.num_samples()

    def _mat(self, m):
        return (m.kind, _d3(m.kd), _d3(m.ks), m.roughness, m.roughness2)

    def _fill(self, idx, agg):
        L = lib()
        for kind, *rest in agg.transforms:
            if kind == "translate":
                L.orc_agg_translate(self.h, idx, _d3(rest[0]))
            elif kind == "scale":
                L.orc_agg_scale(self.h, idx, *rest[0])
            elif kind == "rotate_axis":
                L.orc_agg_rotate_axis(self.h, idx, rest[0], rest[1])
            elif kind == "rotate":
                L.orc_agg_rotate(self.h, idx, rest[0], _d3(rest[1]))
        if agg._swap_backface:
            L.orc_agg_swap_backface(self.h, idx)
        for item in agg.contents:
            k = item[0]
            if k == "sphere":
                L.orc_agg_add_sphere(self.h, idx, _d3(item[1]), item[2], *self._mat(item[3]))
            elif k == "spheres":
                _, cen, rad, mats, midx = item
                kinds = np.array([m.kind for m in mats], np.int32)
                kd = np.array([m.kd for m in mats], np.float64); ks = np.array([m.ks for m in mats], np.float64)
                rough = np.array([m.roughness for m in mats], np.float64)
                rough2 = np.array([m.roughness2 for m in mats], np.float64)
                L.orc_agg_add_spheres(self.h, idx, len(rad), _ptr(cen, C.c_double), _ptr(rad, C.c_double), len(mats),
                                      _ptr(kinds, C.c_int), _ptr(kd, C.c_double), _ptr(ks, C.c_double),
                                      _ptr(rough, C.c_double), _ptr(rough2, C.c_double), _ptr(midx, C.c_int))
            elif k == "cube":
                L.orc_agg_add_cube(self.h, idx, _d3(item[1]), item[2], *self._mat(item[3]))
            elif k == "box":
                L.orc_agg_add_box(self.h, idx, _d3(item[1]), _d3(item[2]), *self._mat(item[3]))
            elif k == "mesh":
                from lasgun_b200.api import Material
                m = item[2] if item[2] is not None else Material.default()
                L.orc_agg_add_mesh(self.h, idx, item[1].index, 1 if item[2] is not None else 0, *self._mat(m))
            elif k == "group":
                child = L.orc_agg_new(self.h)
                self._fill(child, item[1])
                L.orc_agg_add_group(self.h, idx, child)

    def __del__(self):
        try:
            L = lib()
            if self.accel:
                L.orc_accel_free(self.accel)
            if self.h:
                L.orc_scene_free(self.h)
        except Exception:
            pass

    @property
    def build_ms(self):
        return lib().orc_accel_build_ms(self.accel)

    @property
    def prim_count(self):
        return lib().orc_accel_prim_count(self.accel)

    def capture(self, w, h, threads=0, aov=False, li=False, counters=False, subset=None):
        """Render.  subset=(n, k0, kcount) renders capture_subset(k, n) for k in [k0, k0+kcount)."""
        L = lib()
        spp = self.spp
        rgba = np.zeros((h, w, 4), np.uint8)
        out = {"rgba": rgba}
        ids = np.full((h * w * spp,), MISS, np.uint32) if aov else None
        ts = np.full((h * w * spp,), np.inf, np.float64) if aov else None
        occl = np.zeros((h * w * spp,), np.uint32) if aov else None
        lis = np.zeros((h * w * spp, 3), np.float64) if li else None
        cnt = Counters() if counters else None
        ms = C.c_double(0)
        n, k0, kc = subset if subset else (0, 0, 0)
        rc = L.orc_capture(self.accel, w, h, threads, n, k0, kc, _ptr(rgba, C.c_uint8), _ptr(ids, C.c_uint32) if aov else None,
                           _ptr(ts, C.c_double) if aov else None, _ptr(occl, C.c_uint32) if aov else None,
                           _ptr(lis, C.c_double) if li else None, C.byref(cnt) if counters else None, C.byref(ms))
        if rc == 1:
            raise RuntimeError("oracle: unknown material kind")
        if rc == 2:
            raise RuntimeError("oracle: traversal stack overflow (the reference would panic, bvh.rs:469)")
        out.update(render_ms=ms.value, prim_id=ids, t=ts, occl=occl, li=lis, counters=cnt.as_dict() if counters else None)
        return out

    def debug_li(self, ray, cap=4096):
        """li() of one ray and every ray cast below it: (radiance, array of {kind, depth, o, d, prim id or -1, t})."""
        r = np.ascontiguousarray(ray, np.float64); out = np.zeros(3); tr = np.zeros((cap, 10))
        n = lib().orc_debug_li(self.accel, _ptr(r, C.c_double), _ptr(out, C.c_double), _ptr(tr, C.c_double), cap)
        return out, tr[:min(n, cap)]

    def trace_rays(self, rays_od, normals=False):
        """Closest hit (canonical id, t) of rays given as (n, 6) origin + direction; normals=True also returns the world-space
        RayIntersection::ng() and ns() of each hit, (n, 3) each (zeros on a miss): (ids, t, ng, ns)."""
        rays = np.ascontiguousarray(rays_od, np.float64).reshape(-1, 6)
        ids = np.zeros((len(rays),), np.uint32); t = np.zeros((len(rays),), np.float64)
        ng = np.zeros((len(rays), 3)) if normals else None
        ns = np.zeros((len(rays), 3)) if normals else None
        lib().orc_trace_rays(self.accel, _ptr(rays, C.c_double), len(rays), _ptr(ids, C.c_uint32), _ptr(t, C.c_double),
                             _ptr(ng, C.c_double), _ptr(ns, C.c_double))
        return (ids, t, ng, ns) if normals else (ids, t)

    def camera_sample(self, x, y, w, h):
        out = np.zeros((self.spp, 6), np.float64)
        lib().orc_camera_sample(self.h, x, y, w, h, _ptr(out, C.c_double))
        return out

    def retest(self, prim_id, o, d):
        return lib().orc_retest_prim(self.accel, int(prim_id), _d3(o), _d3(d))

    def bvh_dump(self, path=()):
        L = lib()
        p = (C.c_int * max(1, len(path)))(*path)
        nn = L.orc_bvh_node_count(self.accel, p, len(path))
        npr = L.orc_bvh_prim_count(self.accel, p, len(path))
        if nn < 0:
            raise KeyError(path)
        b = np.zeros((nn, 6), np.float64); meta = np.zeros((nn, 3), np.uint32); order = np.zeros((npr,), np.uint64)
        L.orc_bvh_dump(self.accel, p, len(path), _ptr(b, C.c_double), _ptr(meta, C.c_uint32), _ptr(order, C.c_uint64))
        return b, meta, order


def test_sphere(c, r, o, d):
    out = (C.c_double * 7)()
    hit = lib().orc_test_sphere(_d3(c), r, _d3(o), _d3(d), out)
    return bool(hit), out[0], list(out[1:4]), list(out[4:7])


def test_cuboid(mn, mx, o, d):
    out = (C.c_double * 7)()
    hit = lib().orc_test_cuboid(_d3(mn), _d3(mx), _d3(o), _d3(d), out)
    return bool(hit), out[0], list(out[1:4]), list(out[4:7])


def test_mesh(obj, o, d):
    out = (C.c_double * 7)()
    which = C.c_int64(-1)
    hit = lib().orc_test_mesh(_ptr(obj.positions, C.c_float), len(obj.positions), _ptr(obj.faces, C.c_uint32), len(obj.faces),
                              _ptr(obj.normals, C.c_float), len(obj.normals), _ptr(obj.normal_faces, C.c_uint32),
                              _d3(o), _d3(d), out, C.byref(which))
    return bool(hit), out[0], list(out[1:4]), list(out[4:7]), which.value


def test_surface(t, dpdu, dpdv, o, d):
    out = (C.c_double * 3)()
    lib().orc_test_surface(t, _d3(dpdu), _d3(dpdv), _d3(o), _d3(d), out)
    return list(out)


def hardware_threads():
    return lib().orc_hardware_threads()
