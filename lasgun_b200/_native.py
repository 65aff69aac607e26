"""ctypes binding of liblasgun_b200.so: the lgb_* C ABI (include/lasgun_b200.h) and the lgh_* host
mirror (include/lasgun_host.hpp).  There is no fallback: if the library cannot be loaded, or no
sm_100 GPU is visible, every entry point raises."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import api

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("LASGUN_B200_SO") or os.path.join(_HERE, "liblasgun_b200.so")   # env override: kernel experiments only
_lib = None

LGB_OK, LGB_ERR_INVALID, LGB_ERR_CUDA, LGB_ERR_UNSUPPORTED, LGB_ERR_NOMEM, LGB_ERR_NO_DEVICE = 0, -1, -2, -3, -4, -5
LGB_MISS = 0xFFFFFFFF
CUDA_STREAM_LEGACY = 0x1                 # cudaStreamLegacy (driver_types.h): the legacy default stream as a stream handle
LGB_LEAF_FLAG = 0x80000000
LGB_SCENE_VIEW_BOX = 1

# Every symbol include/lasgun_b200.h declares (checked by tests/test_abi.py without a GPU).
ABI_SYMBOLS = [
    "lgb_build_probe", "lgb_device_count", "lgb_init", "lgb_init_devices", "lgb_context_devices", "lgb_set_option", "lgb_shutdown", "lgb_last_error", "lgb_status_string", "lgb_scene_create", "lgb_scene_set_camera", "lgb_scene_set_lights",
    "lgb_film_alloc_shared", "lgb_film_open_shared", "lgb_film_release_shared", "lgb_film_signal", "lgb_film_wait", "lgb_scene_destroy", "lgb_scene_layout_bytes", "lgb_scene_export", "lgb_scene_import", "lgb_scene_verify", "lgb_scene_device_bytes", "lgb_scene_build_ms", "lgb_scene_node_count", "lgb_capture", "lgb_capture_subset", "lgb_capture_aov",
    "lgb_capture_device", "lgb_capture_linear", "lgb_capture_guides", "lgb_capture_profile", "lgb_trace_rays", "lgb_debug_fastmath", "lgb_measure_l2_read_gbs", "lgb_measure_fp32_gops", "lgb_measure_fp64_gops",
]


class LasgunError(RuntimeError):
    def __init__(self, status, message):
        super().__init__(f"[{status}] {message}")
        self.status = status


class Node(C.Structure):
    _fields_ = [("lo", C.c_float * 3), ("a", C.c_uint32), ("hi", C.c_float * 3), ("b", C.c_uint32)]


class CameraDesc(C.Structure):
    _fields_ = [("origin", C.c_double * 3), ("view", C.c_double * 3), ("up", C.c_double * 3), ("aux", C.c_double * 3),
                ("image_plane_height", C.c_double), ("pixel_separation", C.c_double), ("sample_distance", C.c_double),
                ("supersampling_root", C.c_uint32), ("reserved", C.c_uint32)]


class LightDesc(C.Structure):
    """lgb_light (PointLight, src/light/point.rs:14-18)."""
    _fields_ = [("position", C.c_double * 3), ("intensity", C.c_double * 3), ("falloff", C.c_double * 3)]


class InstanceDesc(C.Structure):
    _fields_ = [("root_node", C.c_uint32), ("identity", C.c_uint32), ("swap_backface", C.c_uint32), ("reserved", C.c_uint32),
                ("m", C.c_double * 16), ("minv", C.c_double * 16)]


class SceneDesc(C.Structure):
    _fields_ = [
        ("abi_version", C.c_uint32), ("flags", C.c_uint32),
        ("nodes", C.c_void_p), ("n_nodes", C.c_uint64),
        ("prim_refs", C.c_void_p), ("n_prim_refs", C.c_uint64),
        ("spheres", C.c_void_p), ("n_spheres", C.c_uint64), ("sphere_material", C.c_void_p), ("sphere_id", C.c_void_p),
        ("cuboids", C.c_void_p), ("n_cuboids", C.c_uint64), ("cuboid_material", C.c_void_p), ("cuboid_id", C.c_void_p),
        ("triangles", C.c_void_p), ("n_triangles", C.c_uint64), ("triangle_material", C.c_void_p), ("triangle_id", C.c_void_p),
        ("tri_normals", C.c_void_p), ("tri_has_normals", C.c_void_p),
        ("instances", C.c_void_p), ("n_instances", C.c_uint64), ("root", InstanceDesc),
        ("materials", C.c_void_p), ("n_materials", C.c_uint64),
        ("lights", C.c_void_p), ("n_lights", C.c_uint64),
        ("camera", CameraDesc),
        ("ambient", C.c_double * 3), ("bg_inner", C.c_double * 3), ("bg_outer", C.c_double * 3), ("bg_scale", C.c_double),
        ("recursion", C.c_uint32), ("expected_film_pixels", C.c_uint32),
        ("reference_tree", C.c_void_p), ("reference_tree_user", C.c_void_p), ("bounds_lo", C.c_double * 3), ("bounds_hi", C.c_double * 3),
        ("view_lo", C.c_double * 3), ("view_hi", C.c_double * 3),
    ]


class BuildInfo(C.Structure):
    _fields_ = [("nodes", C.c_uint32), ("max_depth", C.c_uint32), ("leaves", C.c_uint32), ("max_leaf", C.c_uint32),
                ("prims", C.c_uint32), ("ranks_ok", C.c_uint32), ("boxes_ok", C.c_uint32), ("reserved", C.c_uint32),
                ("build_ms", C.c_double), ("rank_ms", C.c_double), ("sah_cost", C.c_double)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class Guides(C.Structure):
    """lgb_guides: the device buffers of lgb_capture_guides (NULL = not written)."""
    _fields_ = [("rgb", C.c_void_p), ("normal", C.c_void_p), ("depth", C.c_void_p), ("prim_id", C.c_void_p), ("coverage", C.c_void_p)]


class KernelTime(C.Structure):
    _fields_ = [("name", C.c_char * 40), ("ms", C.c_float), ("reserved", C.c_uint32), ("node_tests", C.c_uint64),
                ("filter_tests", C.c_uint64 * 3), ("exact_tests", C.c_uint64 * 3), ("primary_rays", C.c_uint64), ("primary_hits", C.c_uint64),
                ("shadow_rays", C.c_uint64), ("shadow_occluded", C.c_uint64)]


class Stats(C.Structure):
    _fields_ = [("primary_rays", C.c_uint64), ("primary_hits", C.c_uint64), ("shadow_rays", C.c_uint64),
                ("shadow_rays_traced", C.c_uint64), ("shadow_occluded", C.c_uint64), ("shadow_cache_hits", C.c_uint64), ("exact_tests", C.c_uint64 * 3),
                ("filter_tests", C.c_uint64 * 3), ("node_tests", C.c_uint64), ("primary_node_tests", C.c_uint64),
                ("primary_exact_tests", C.c_uint64 * 3), ("primary_filter_tests", C.c_uint64 * 3), ("kernel_ms", C.c_float * 6), ("render_ms", C.c_float), ("total_ms", C.c_float),
                ("kernel_launches", C.c_uint32), ("stack_overflow", C.c_uint32), ("beams", C.c_uint32), ("tie_retraces", C.c_uint32), ("secondary_rays", C.c_uint64),
                ("bands", C.c_uint32), ("reserved", C.c_uint32)]

    def as_dict(self):
        return {n: (list(getattr(self, n)) if n in ("exact_tests", "filter_tests", "primary_exact_tests", "primary_filter_tests", "kernel_ms") else getattr(self, n)) for n, _ in self._fields_}


def lib():
    """Loads the in-tree shared library; fails loudly if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise LasgunError(LGB_ERR_NO_DEVICE, f"{SO_PATH} is missing: run `python -m lasgun_b200.build` (no CPU fallback exists)")
    L = C.CDLL(SO_PATH)
    vp, dp, fp, u32p, u64p, u8p, ip = (C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_float), C.POINTER(C.c_uint32),
                                       C.POINTER(C.c_uint64), C.POINTER(C.c_uint8), C.POINTER(C.c_int))
    sig = {
        "lgb_device_count": (C.c_int, []), "lgb_init": (C.c_int, [C.c_int, C.POINTER(vp)]),
        "lgb_init_devices": (C.c_int, [C.c_int, ip, C.POINTER(vp)]), "lgb_context_devices": (C.c_int, [vp]), "lgb_shutdown": (None, [vp]),
        "lgb_set_option": (C.c_int, [vp, C.c_int, C.c_int]),
        "lgb_build_probe": (C.c_int, [C.POINTER(SceneDesc), C.POINTER(BuildInfo)]),
        "lgb_last_error": (C.c_char_p, [vp]), "lgb_status_string": (C.c_char_p, [C.c_int]),
        "lgb_scene_create": (C.c_int, [vp, C.POINTER(SceneDesc), C.POINTER(vp)]), "lgb_scene_destroy": (None, [vp]),
        "lgb_scene_set_camera": (C.c_int, [vp, vp, C.POINTER(CameraDesc)]),
        "lgb_scene_set_lights": (C.c_int, [vp, vp, C.POINTER(LightDesc), C.c_uint64, dp]),
        "lgb_film_alloc_shared": (C.c_int, [vp, C.c_uint64, C.POINTER(C.c_void_p), u8p]),
        "lgb_film_open_shared": (C.c_int, [vp, u8p, C.POINTER(C.c_void_p)]),
        "lgb_film_release_shared": (C.c_int, [vp, vp, C.c_int]),
        "lgb_film_signal": (C.c_int, [vp, vp, C.c_uint32, vp]),
        "lgb_film_wait": (C.c_int, [vp, vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, vp]),
        "lgb_scene_layout_bytes": (C.c_uint64, []),
        "lgb_scene_export": (C.c_int, [vp, vp, C.c_uint64, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]),
        "lgb_scene_import": (C.c_int, [vp, vp, C.c_uint64, vp, C.POINTER(C.c_void_p)]),
        "lgb_scene_verify": (C.c_int, [vp, vp, C.POINTER(BuildInfo)]),
        "lgb_scene_device_bytes": (C.c_uint64, [vp]), "lgb_scene_build_ms": (C.c_double, [vp]),
        "lgb_scene_node_count": (C.c_uint32, [vp]),
        "lgb_capture": (C.c_int, [vp, vp, C.c_uint32, C.c_uint32, u8p, C.POINTER(Stats)]),
        "lgb_capture_subset": (C.c_int, [vp, vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, u8p, C.POINTER(Stats)]),
        "lgb_capture_aov": (C.c_int, [vp, vp, C.c_uint32, C.c_uint32, u8p, u32p, dp, u32p, dp, C.POINTER(Stats)]),
        "lgb_capture_device": (C.c_int, [vp, vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, vp, vp, C.POINTER(Stats)]),
        "lgb_capture_linear": (C.c_int, [vp, vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, fp, vp, C.POINTER(Stats)]),
        "lgb_capture_guides": (C.c_int, [vp, vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(Guides), vp, C.POINTER(Stats)]),
        "lgb_capture_profile": (C.c_int, [vp, vp, C.c_uint32, C.c_uint32, vp, C.POINTER(KernelTime), C.c_uint32, u32p, C.POINTER(Stats)]),
        "lgb_trace_rays": (C.c_int, [vp, vp, dp, C.c_uint64, u32p, dp, dp, dp]),
        "lgb_debug_fastmath": (C.c_int, [vp, dp, C.c_uint64, dp, dp]),
        "lgb_measure_l2_read_gbs": (C.c_int, [vp, C.c_uint64, C.c_int, dp]),
        "lgb_measure_fp32_gops": (C.c_int, [vp, C.c_int, dp]), "lgb_measure_fp64_gops": (C.c_int, [vp, C.c_int, dp]),
        # host mirror
        "lgh_last_error": (C.c_char_p, []), "lgh_scene_new": (vp, []), "lgh_scene_free": (None, [vp]),
        "lgh_set_perspective_camera": (None, [vp, C.c_double]), "lgh_set_orthographic_camera": (None, [vp, C.c_double]),
        "lgh_look_at": (None, [vp, dp, dp, dp]), "lgh_set_supersampling": (C.c_int, [vp, C.c_int]),
        "lgh_camera_describe": (C.c_int, [C.c_int, C.c_double, dp, dp, dp, C.c_int, C.POINTER(CameraDesc)]),
        "lgh_set_ambient_light": (None, [vp, dp]), "lgh_set_radial_background": (None, [vp, dp, dp, C.c_double]),
        "lgh_set_mesh_smoothing": (None, [vp, C.c_int]), "lgh_add_point_light": (None, [vp, dp, dp, dp]),
        "lgh_add_mesh": (C.c_int, [vp, fp, C.c_uint64, u32p, C.c_uint64, fp, C.c_uint64, u32p, C.POINTER(C.c_int64)]),
        "lgh_agg_new": (C.c_int, [vp]),
        "lgh_agg_add_sphere": (None, [vp, C.c_int, dp, C.c_double, C.c_int, dp, dp, C.c_double, C.c_double]),
        "lgh_agg_add_spheres": (None, [vp, C.c_int, C.c_uint64, dp, dp, C.c_int, ip, dp, dp, dp, dp, ip]),
        "lgh_agg_add_cube": (None, [vp, C.c_int, dp, C.c_double, C.c_int, dp, dp, C.c_double, C.c_double]),
        "lgh_agg_add_box": (None, [vp, C.c_int, dp, dp, C.c_int, dp, dp, C.c_double, C.c_double]),
        "lgh_agg_add_mesh": (None, [vp, C.c_int, C.c_int64, C.c_int, C.c_int, dp, dp, C.c_double, C.c_double]),
        "lgh_set_max_recursion_depth": (None, [vp, C.c_uint32]),
        "lgh_agg_add_group": (None, [vp, C.c_int, C.c_int]), "lgh_agg_swap_backface": (None, [vp, C.c_int]),
        "lgh_agg_translate": (None, [vp, C.c_int, dp]), "lgh_agg_scale": (None, [vp, C.c_int, C.c_double, C.c_double, C.c_double]),
        "lgh_agg_rotate_axis": (None, [vp, C.c_int, C.c_int, C.c_double]), "lgh_agg_rotate": (None, [vp, C.c_int, C.c_double, dp]),
        "lgh_flatten": (vp, [vp, C.c_int, C.c_int]), "lgh_flat_tree_built": (C.c_int, [vp]), "lgh_flat_build_tree": (C.c_int, [vp]), "lgh_flat_free": (None, [vp]),
        "lgh_flat_describe": (None, [vp, C.POINTER(SceneDesc)]), "lgh_flat_build_ms": (C.c_double, [vp]),
        "lgh_flat_prim_count": (C.c_uint32, [vp]), "lgh_flat_level_count": (C.c_uint64, [vp]),
        "lgh_flat_level_dims": (C.c_int, [vp, C.c_uint64, u64p, u64p, u32p]),
        "lgh_flat_level_dump": (C.c_int, [vp, C.c_uint64, dp, u32p, u64p]),
        "lgh_capture": (C.c_int, [vp, C.c_uint32, C.c_uint32, u8p]),
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


def camera_desc(cam: api.Camera) -> CameraDesc:
    """The lgb_camera of an api.Camera, set up as HostScene sets up a scene's camera (constructor, look_at, set_supersampling):
    bit for bit the camera a scene built with `cam` carries in its desc."""
    out = CameraDesc()
    look = [_d3(v) for v in cam.look] if cam.look is not None else [None, None, None]
    rc = lib().lgh_camera_describe(1 if cam.perspective else 0, cam.param, *look, cam.supersampling, C.byref(out))
    if rc != LGB_OK:
        raise LasgunError(rc, lib().lgh_last_error().decode())
    return out


def light_descs(lights):
    """The lgb_light records of (position, intensity, falloff) triples, as api.Scene.lights holds them: the array FlatScene puts in
    the desc for a scene with these lights."""
    lights = [tuple(api._v3(v) for v in l) for l in lights]
    return (LightDesc * len(lights))(*[LightDesc(*(_d3(v) for v in l)) for l in lights])


class HostScene:
    """C++ `lasgun::Scene` built by replaying an api.Scene description (scene.rs / node.rs surface)."""

    def __init__(self, scene: api.Scene):
        L = lib()
        self.desc = scene
        self.h = L.lgh_scene_new()
        cam = scene.camera
        (L.lgh_set_perspective_camera if cam.perspective else L.lgh_set_orthographic_camera)(self.h, cam.param)
        if cam.look is not None:
            L.lgh_look_at(self.h, _d3(cam.look[0]), _d3(cam.look[1]), _d3(cam.look[2]))
        self._check(L.lgh_set_supersampling(self.h, cam.supersampling))
        L.lgh_set_ambient_light(self.h, _d3(scene.ambient))
        L.lgh_set_max_recursion_depth(self.h, int(scene.recursion))
        L.lgh_set_radial_background(self.h, _d3(scene.background[0]), _d3(scene.background[1]), scene.background[2])
        for p, i, f in scene.lights:
            L.lgh_add_point_light(self.h, _d3(p), _d3(i), _d3(f))
        for m in scene.meshes:
            ref = C.c_int64(-1)
            self._check(L.lgh_add_mesh(self.h, _ptr(m.positions, C.c_float), len(m.positions), _ptr(m.faces, C.c_uint32), len(m.faces),
                                       _ptr(m.normals, C.c_float), len(m.normals), _ptr(m.normal_faces, C.c_uint32), C.byref(ref)))
        self._fill(0, scene.root)

    def _check(self, rc):
        if rc != LGB_OK:
            raise LasgunError(rc, lib().lgh_last_error().decode())

    @staticmethod
    def _mat(m):
        return (m.kind, _d3(m.kd), _d3(m.ks), m.roughness, m.roughness2)

    def _fill(self, idx, agg):
        L = lib()
        for kind, *rest in agg.transforms:
            if kind == "translate":
                L.lgh_agg_translate(self.h, idx, _d3(rest[0]))
            elif kind == "scale":
                L.lgh_agg_scale(self.h, idx, *rest[0])
            elif kind == "rotate_axis":
                L.lgh_agg_rotate_axis(self.h, idx, rest[0], rest[1])
            elif kind == "rotate":
                L.lgh_agg_rotate(self.h, idx, rest[0], _d3(rest[1]))
        if agg._swap_backface:
            L.lgh_agg_swap_backface(self.h, idx)
        for item in agg.contents:
            k = item[0]
            if k == "sphere":
                L.lgh_agg_add_sphere(self.h, idx, _d3(item[1]), item[2], *self._mat(item[3]))
            elif k == "spheres":
                _, cen, rad, mats, midx = item
                kinds = np.array([m.kind for m in mats], np.int32)
                kd = np.array([m.kd for m in mats], np.float64); ks = np.array([m.ks for m in mats], np.float64)
                rough = np.array([m.roughness for m in mats], np.float64)
                rough2 = np.array([m.roughness2 for m in mats], np.float64)
                L.lgh_agg_add_spheres(self.h, idx, len(rad), _ptr(cen, C.c_double), _ptr(rad, C.c_double), len(mats),
                                      _ptr(kinds, C.c_int), _ptr(kd, C.c_double), _ptr(ks, C.c_double), _ptr(rough, C.c_double),
                                      _ptr(rough2, C.c_double), _ptr(midx, C.c_int))
            elif k == "cube":
                L.lgh_agg_add_cube(self.h, idx, _d3(item[1]), item[2], *self._mat(item[3]))
            elif k == "box":
                L.lgh_agg_add_box(self.h, idx, _d3(item[1]), _d3(item[2]), *self._mat(item[3]))
            elif k == "mesh":
                m = item[2] if item[2] is not None else api.Material.default()
                L.lgh_agg_add_mesh(self.h, idx, item[1].index, 1 if item[2] is not None else 0, *self._mat(m))
            elif k == "group":
                child = L.lgh_agg_new(self.h)
                self._fill(child, item[1])
                L.lgh_agg_add_group(self.h, idx, child)

    def __del__(self):
        try:
            if self.h:
                lib().lgh_scene_free(self.h)
                self.h = None
        except Exception:
            pass


class FlatScene:
    """Host-side flattened scene (Accel::from without the upload): owns the arrays of an lgb_scene_desc."""

    def __init__(self, scene, keep_levels=False, lazy=False, view_box=None):
        """lazy=True: the reference BVH is not built now; the device asks for it (reference_tree callback) only if a
        closest-hit ray meets two primitives at bit-identical t.  Accessors that need the tree build it.
        view_box=(lo, hi): world box of every camera origin DeviceScene.set_camera will be given (LGB_SCENE_VIEW_BOX); the scene's
        f32 error bound then covers it.  None: the scene and its own camera only."""
        L = lib()
        self.host = scene if isinstance(scene, HostScene) else HostScene(scene)
        self.h = L.lgh_flatten(self.host.h, 1 if keep_levels else 0, 1 if lazy else 0)
        if not self.h:
            msg = L.lgh_last_error().decode()
            raise LasgunError(LGB_ERR_UNSUPPORTED if "not on the device path" in msg or "outside the device" in msg else LGB_ERR_INVALID, msg)
        self.view_box = None if view_box is None else (_d3(view_box[0]), _d3(view_box[1]))
        self.desc = SceneDesc()
        self._describe()
        self.spp = self.desc.camera.supersampling_root ** 2

    def _describe(self):
        lib().lgh_flat_describe(self.h, C.byref(self.desc))
        if self.view_box is not None:
            self.desc.flags |= LGB_SCENE_VIEW_BOX
            self.desc.view_lo, self.desc.view_hi = self.view_box

    @property
    def tree_built(self):
        return bool(lib().lgh_flat_tree_built(self.h))

    def build_tree(self):
        """Builds the reference BVH now (no-op if it exists) and refreshes the desc."""
        L = lib()
        if L.lgh_flat_build_tree(self.h):
            raise LasgunError(LGB_ERR_INVALID, L.lgh_last_error().decode())
        self._describe()
        self.n_lights = self.desc.n_lights

    @property
    def build_ms(self):
        return lib().lgh_flat_build_ms(self.h)

    @property
    def prim_count(self):
        return lib().lgh_flat_prim_count(self.h)

    def nodes(self):
        self.build_tree()
        n = self.desc.n_nodes
        buf = (Node * n).from_address(self.desc.nodes)
        return np.frombuffer(buf, dtype=np.dtype([("lo", "<f4", 3), ("a", "<u4"), ("hi", "<f4", 3), ("b", "<u4")]), count=n)

    def prim_refs(self):
        self.build_tree()
        n = self.desc.n_prim_refs
        return np.frombuffer((C.c_uint32 * n).from_address(self.desc.prim_refs), dtype=np.uint32, count=n)

    def level(self, i):
        L = lib()
        nn, npr, off = C.c_uint64(), C.c_uint64(), C.c_uint32()
        if L.lgh_flat_level_dims(self.h, i, C.byref(nn), C.byref(npr), C.byref(off)):
            raise IndexError(i)
        b = np.zeros((nn.value, 6)); meta = np.zeros((nn.value, 3), np.uint32); order = np.zeros((npr.value,), np.uint64)
        L.lgh_flat_level_dump(self.h, i, _ptr(b, C.c_double), _ptr(meta, C.c_uint32), _ptr(order, C.c_uint64))
        return b, meta, order, off.value

    def level_count(self):
        return lib().lgh_flat_level_count(self.h)

    def build_probe(self):
        """Host-only run of lgb_scene_create's device-BVH + rank-table construction (no GPU needed)."""
        info = BuildInfo()
        rc = lib().lgb_build_probe(C.byref(self.desc), C.byref(info))
        if rc:
            raise LasgunError(rc, "lgb_build_probe failed")
        return info.as_dict()

    def __del__(self):
        try:
            if self.h:
                lib().lgh_flat_free(self.h)
                self.h = None
        except Exception:
            pass


class Context:
    """lgb_ctx: one GPU."""

    def __init__(self, device=0, devices=None):
        """One GPU (`device`), or a device group in this process (`devices`: the first one leads, lgb_init_devices)."""
        L = lib()
        h = C.c_void_p()
        if devices is not None:
            arr = (C.c_int * len(devices))(*devices)
            rc = L.lgb_init_devices(len(devices), arr, C.byref(h))
            device = devices[0] if len(devices) else 0
        else:
            rc = L.lgb_init(device, C.byref(h))
        if rc:
            raise LasgunError(rc, L.lgb_last_error(None).decode())
        self.h = h
        self.device = device
        self.n_devices = int(L.lgb_context_devices(h))

    def check(self, rc):
        if rc:
            raise LasgunError(rc, lib().lgb_last_error(self.h).decode())

    def close(self):
        if self.h:
            lib().lgb_shutdown(self.h)
            self.h = None

    def set_count_work(self, on: bool):
        self.check(lib().lgb_set_option(self.h, 1, 1 if on else 0))

    def set_beams(self, mode: int):
        """LGB_OPT_BEAMS: 1 on (whenever spp >= 4), 0 off, -1 automatic (the default)."""
        self.check(lib().lgb_set_option(self.h, 2, int(mode)))

    def set_light_grids(self, mode: int):
        """LGB_OPT_LIGHT_GRIDS (read at scene creation): 1 on, 0 off, -1 automatic (the default)."""
        self.check(lib().lgb_set_option(self.h, 5, int(mode)))

    def set_wave_budget_mb(self, mb: int):
        """LGB_OPT_WAVE_BUDGET_MB: per-sample buffers of one band of a frame (default 16384)."""
        self.check(lib().lgb_set_option(self.h, 7, int(mb)))

    def set_lazy_bvh(self, mode: int):
        """LGB_OPT_LAZY_BVH (read at scene creation): 0 build the device BVH with the scene, 1 / -1 only when something walks it."""
        self.check(lib().lgb_set_option(self.h, 8, int(mode)))

    def set_camera_grid(self, mode: int):
        """LGB_OPT_CAMERA_GRID: 1 on, 0 off, -1 automatic (the default)."""
        self.check(lib().lgb_set_option(self.h, 6, int(mode)))

    def set_side_streams(self, on: bool):
        """LGB_OPT_SIDE_STREAMS: overlap the shadow chains of different lights (default on)."""
        self.check(lib().lgb_set_option(self.h, 4, 1 if on else 0))

    def set_whitted(self, wavefront: bool):
        """LGB_OPT_WHITTED: the specular ray trees level by level (default) or one thread per tree."""
        self.check(lib().lgb_set_option(self.h, 3, 1 if wavefront else 0))

    def fastmath(self, x):
        """lgb_debug_fastmath: the shading kernel's reciprocal and reciprocal square root of every x (positive, normal f64)."""
        import numpy as np
        x = np.ascontiguousarray(x, dtype=np.float64)
        r, q = np.empty_like(x), np.empty_like(x)
        self.check(lib().lgb_debug_fastmath(self.h, _ptr(x, C.c_double), x.size, _ptr(r, C.c_double), _ptr(q, C.c_double)))
        return r, q

    def measure(self):
        L = lib()
        out = {}
        v = C.c_double()
        self.check(L.lgb_measure_l2_read_gbs(self.h, 32 << 20, 50, C.byref(v))); out["l2_read_gbs"] = v.value
        self.check(L.lgb_measure_fp32_gops(self.h, 20000, C.byref(v))); out["fp32_ffma_glanes"] = v.value
        self.check(L.lgb_measure_fp64_gops(self.h, 20000, C.byref(v))); out["fp64_dfma_glanes"] = v.value
        return out


_default_ctx = None


def default_context():
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = Context(int(os.environ.get("LOCAL_RANK", "0")) if lib().lgb_device_count() > 1 else 0)
    return _default_ctx


class DeviceScene:
    """lgb_scene: the flattened scene resident in HBM."""

    def __init__(self, ctx: Context, flat: FlatScene | None, _handle=None, _spp=None, _keep=None):
        L = lib()
        self.ctx, self.flat = ctx, flat
        self._keep = _keep                       # imported scenes: the object that owns the arena memory
        if _handle is not None:
            self.h, self.spp = _handle, _spp
            return
        h = C.c_void_p()
        ctx.check(L.lgb_scene_create(ctx.h, C.byref(flat.desc), C.byref(h)))
        self.h = h
        self.spp = flat.spp

    def set_camera(self, camera):
        """lgb_scene_set_camera: captures enqueued from now on render with `camera` (an api.Camera or a CameraDesc); captures already
        enqueued keep theirs.  A camera whose origin leaves the scene's world box (the scene, its creation camera and the view box of
        its FlatScene) raises LasgunError with LGB_ERR_UNSUPPORTED, and the scene keeps its camera.  Returns self."""
        desc = camera if isinstance(camera, CameraDesc) else camera_desc(camera)
        self.ctx.check(lib().lgb_scene_set_camera(self.ctx.h, self.h, C.byref(desc)))
        self.spp = desc.supersampling_root ** 2
        return self

    def set_lights(self, lights, ambient):
        """lgb_scene_set_lights: captures enqueued from now on render with `lights` ((position, intensity, falloff) triples, as
        api.Scene.lights; 0 to LGB_MAX_LIGHTS of them) and the ambient term `ambient`; captures already enqueued keep theirs.  A light
        with a coordinate beyond 4 M (M: the largest coordinate of the scene's world box) raises LasgunError with LGB_ERR_UNSUPPORTED,
        and the scene keeps its lights.  Returns self."""
        recs = light_descs(lights)
        self.ctx.check(lib().lgb_scene_set_lights(self.ctx.h, self.h, recs, len(recs), _d3(ambient)))
        return self

    def verify(self):
        """Structural check of the resident device BVH (lgb_scene_verify)."""
        info = BuildInfo()
        self.ctx.check(lib().lgb_scene_verify(self.ctx.h, self.h, C.byref(info)))
        return info.as_dict()

    def export(self):
        """(layout bytes, arena device pointer, arena bytes): what another rank needs to import this scene."""
        L = lib()
        n = L.lgb_scene_layout_bytes()
        buf = (C.c_uint8 * n)()
        ptr, nbytes = C.c_void_p(), C.c_uint64()
        self.ctx.check(L.lgb_scene_export(self.h, buf, n, C.byref(ptr), C.byref(nbytes)))
        return bytes(buf), ptr.value, nbytes.value

    @staticmethod
    def adopt(ctx: Context, layout: bytes, arena_ptr: int, spp: int, keep=None):
        """Scene over an arena this rank received from the rank that built it (lgb_scene_import)."""
        L = lib()
        h = C.c_void_p()
        buf = (C.c_uint8 * len(layout)).from_buffer_copy(layout)
        ctx.check(L.lgb_scene_import(ctx.h, buf, len(layout), C.c_void_p(arena_ptr), C.byref(h)))
        return DeviceScene(ctx, None, _handle=h, _spp=spp, _keep=keep)

    @property
    def device_bytes(self):
        return lib().lgb_scene_device_bytes(self.h)

    @property
    def build_ms(self):
        return lib().lgb_scene_build_ms(self.h)

    @property
    def node_count(self):
        return lib().lgb_scene_node_count(self.h)

    def capture(self, w, h, out=None):
        rgba = out if out is not None else np.zeros((h, w, 4), np.uint8)
        st = Stats()
        self.ctx.check(lib().lgb_capture(self.ctx.h, self.h, w, h, _ptr(rgba, C.c_uint8), C.byref(st)))
        return rgba, st.as_dict()

    def capture_subset(self, k, n, w, h, rgba):
        st = Stats()
        self.ctx.check(lib().lgb_capture_subset(self.ctx.h, self.h, k, n, w, h, _ptr(rgba, C.c_uint8), C.byref(st)))
        return st.as_dict()

    def capture_aov(self, w, h, li=False):
        ns = w * h * self.spp
        rgba = np.zeros((h, w, 4), np.uint8)
        ids = np.zeros((ns,), np.uint32); t = np.zeros((ns,), np.float64); occl = np.zeros((ns,), np.uint32)
        rad = np.zeros((ns, 3), np.float64) if li else None
        st = Stats()
        self.ctx.check(lib().lgb_capture_aov(self.ctx.h, self.h, w, h, _ptr(rgba, C.c_uint8), _ptr(ids, C.c_uint32),
                                             _ptr(t, C.c_double), _ptr(occl, C.c_uint32), _ptr(rad, C.c_double) if li else None, C.byref(st)))
        return {"rgba": rgba, "prim_id": ids, "t": t, "occl": occl, "li": rad, "stats": st.as_dict()}

    def capture_device(self, w, h, d_film_ptr, rank=0, ranks=1, stream=0, want_stats=False):
        st = Stats() if want_stats else None
        self.ctx.check(lib().lgb_capture_device(self.ctx.h, self.h, w, h, rank, ranks, C.c_void_p(d_film_ptr),
                                                C.c_void_p(stream) if stream else None, C.byref(st) if want_stats else None))
        return st.as_dict() if want_stats else None

    def capture_linear(self, w, h, out=None, rank=0, ranks=1, stream=None, want_stats=False):
        """lgb_capture_linear: the linear film (the colour the RGBA8 film quantises, as float32, neither clamped nor quantised) as a
        torch.float32 CUDA tensor of shape (h, w, 3), on the context's device unless `out` is given.  Enqueued on `stream` (a
        torch.cuda.Stream; default torch.cuda.current_stream()) and asynchronous unless want_stats.  Returns the tensor, or
        (tensor, stats dict) with want_stats."""
        import torch
        dev = torch.device("cuda", self.ctx.device)
        if out is None:
            out = torch.empty((h, w, 3), dtype=torch.float32, device=dev)
        elif out.dtype != torch.float32 or out.device != dev or tuple(out.shape) != (h, w, 3) or not out.is_contiguous():
            raise ValueError(f"capture_linear: out must be a contiguous float32 tensor of shape ({h}, {w}, 3) on {dev}, "
                             f"got {out.dtype} {tuple(out.shape)} on {out.device}{'' if out.is_contiguous() else ', not contiguous'}")
        if stream is None:
            stream = torch.cuda.current_stream(dev)
        # torch's default stream is the legacy one (handle 0); NULL would mean the context's private stream, so pass cudaStreamLegacy
        handle = stream.cuda_stream or CUDA_STREAM_LEGACY
        st = Stats() if want_stats else None
        self.ctx.check(lib().lgb_capture_linear(self.ctx.h, self.h, w, h, rank, ranks, C.cast(C.c_void_p(out.data_ptr()), C.POINTER(C.c_float)),
                                                C.c_void_p(handle), C.byref(st) if want_stats else None))
        return (out, st.as_dict()) if want_stats else out

    GUIDES = ("rgb", "normal", "depth", "prim_id", "coverage")

    def capture_guides(self, w, h, rgb=True, normal=True, depth=True, prim_id=True, coverage=True, out=None, rank=0, ranks=1, stream=None,
                       want_stats=False):
        """lgb_capture_guides: per-pixel geometry of the camera rays' closest hits as CUDA tensors, in a dict keyed by the requested
        outputs: normal (h, w, 3) float32, depth (h, w) float32, prim_id (h, w) int32 holding the u32 id (LGB_MISS reads as -1),
        coverage (h, w) float32, and rgb (h, w, 3) float32, the linear film of the same frame.  rgb=False renders a geometry pass
        (primary rays only).  `out` (optional): a dict of caller tensors for some of the requested outputs, checked as
        capture_linear checks its `out`.  Enqueued on `stream` (default torch.cuda.current_stream()), asynchronous unless want_stats.
        Returns the dict, or (dict, stats dict) with want_stats."""
        import torch
        dev = torch.device("cuda", self.ctx.device)
        want = {"rgb": rgb, "normal": normal, "depth": depth, "prim_id": prim_id, "coverage": coverage}
        shapes = {"rgb": (h, w, 3), "normal": (h, w, 3), "depth": (h, w), "prim_id": (h, w), "coverage": (h, w)}
        out = dict(out or {})
        for k in out:
            if k not in want or not want[k]:
                raise ValueError(f"capture_guides: out[{k!r}] is not a requested output")
        res = {}
        for k in self.GUIDES:
            if not want[k]:
                continue
            dtype = torch.int32 if k == "prim_id" else torch.float32
            t = out.get(k)
            if t is None:
                t = torch.empty(shapes[k], dtype=dtype, device=dev)
            elif t.dtype != dtype or t.device != dev or tuple(t.shape) != shapes[k] or not t.is_contiguous():
                raise ValueError(f"capture_guides: out[{k!r}] must be a contiguous {dtype} tensor of shape {shapes[k]} on {dev}, "
                                 f"got {t.dtype} {tuple(t.shape)} on {t.device}{'' if t.is_contiguous() else ', not contiguous'}")
            res[k] = t
        if not res:
            raise ValueError("capture_guides: no output requested")
        g = Guides(*[res[k].data_ptr() if k in res else None for k in self.GUIDES])
        if stream is None:
            stream = torch.cuda.current_stream(dev)
        handle = stream.cuda_stream or CUDA_STREAM_LEGACY           # (see capture_linear)
        st = Stats() if want_stats else None
        self.ctx.check(lib().lgb_capture_guides(self.ctx.h, self.h, w, h, rank, ranks, C.byref(g), C.c_void_p(handle),
                                                C.byref(st) if want_stats else None))
        return (res, st.as_dict()) if want_stats else res

    def capture_profile(self, w, h, d_film_ptr=0):
        """lgb_capture_profile: (list of per-launch dicts in launch order, frame stats)."""
        arr = (KernelTime * 64)()
        n = C.c_uint32()
        st = Stats()
        self.ctx.check(lib().lgb_capture_profile(self.ctx.h, self.h, w, h, C.c_void_p(d_film_ptr) if d_film_ptr else None, arr, 64, C.byref(n), C.byref(st)))
        out = []
        for k in arr[:min(n.value, 64)]:
            out.append({"name": k.name.decode(), "ms": float(k.ms), "node_tests": int(k.node_tests), "filter_tests": list(k.filter_tests),
                        "exact_tests": list(k.exact_tests), "primary_rays": int(k.primary_rays), "primary_hits": int(k.primary_hits),
                        "shadow_rays": int(k.shadow_rays), "shadow_occluded": int(k.shadow_occluded)})
        return out, st.as_dict()

    def trace_rays(self, rays_od):
        rays = np.ascontiguousarray(rays_od, np.float64).reshape(-1, 6)
        n = len(rays)
        ids = np.zeros((n,), np.uint32); t = np.zeros((n,), np.float64); ng = np.zeros((n, 3)); ns = np.zeros((n, 3))
        self.ctx.check(lib().lgb_trace_rays(self.ctx.h, self.h, _ptr(rays, C.c_double), n, _ptr(ids, C.c_uint32), _ptr(t, C.c_double),
                                            _ptr(ng, C.c_double), _ptr(ns, C.c_double)))
        return ids, t, ng, ns

    def destroy(self):
        if self.h:
            if self.ctx.h:                       # (a scene outliving its context is leaked, not freed through a dead context)
                lib().lgb_scene_destroy(self.h)
            self.h = None
            self._keep = None

    def __del__(self):
        try:
            self.destroy()
        except Exception:
            pass
