"""The oracle's ray entry point (`OracleScene.trace_rays(..., normals=True)`) reports the world-space RayIntersection::ng() and
ns() of the closest hit.  tests/test_trace_rays.py compares the device's normals with these, so they are pinned here first: the
reference's own unit-test vectors (SURVEY.md §4, the ones test_known_answers_on_device uses for the device) traced through a
whole scene, and one closed form for a transformed group with swap_backface."""
import numpy as np

from lasgun_b200.api import Aggregate, Material, Scene

PLAST = Material.plastic([0.5, 0.5, 0.5], [0.3, 0.3, 0.3], 0.25)
PLANE = "v -1 0 -1\nv 1 0 -1\nv 1 0 1\nv -1 0 1\nf 1 2 3\nf 1 3 4\n"


def veq(a, b):
    return all(float(x) == float(y) for x, y in zip(a, b))   # -0.0 == 0.0, as Rust's PartialEq


def one(oracle, sc, o, d):
    ids, t, ng, ns = oracle.OracleScene(sc).trace_rays(np.array([list(o) + list(d)], np.float64), normals=True)
    return int(ids[0]), float(t[0]), ng[0], ns[0]


def sphere_scene():
    sc = Scene(); sc.root.add_sphere([0, 0, 0], 1.0, PLAST)
    return sc


def box_scene(mn, mx):
    sc = Scene(); sc.root.add_box(mn, mx, PLAST)
    return sc


def test_trace_normals_sphere_vectors(oracle):
    sc = sphere_scene()
    i, t, ng, _ = one(oracle, sc, [0, 0, 2], [0, 0, -1]); assert i == 0 and t == 1.0 and veq(ng, [0, 0, 1])             # sphere.rs:137
    i, t, ng, _ = one(oracle, sc, [0, 0, 0], [0, 0, 1]); assert i == 0 and t == 1.0 and veq(ng, [0, 0, -1])              # sphere.rs:149
    i, t, ng, _ = one(oracle, sc, [0, 0, -2], [0, 0, 1]); assert i == 0 and t == 1.0 and veq(np.round(ng), [0, 0, -1])   # sphere.rs:160


def test_trace_normals_cuboid_vectors(oracle):     # cuboid.rs:137-245
    unit, wide = ([-1, -1, -1], [1, 1, 1]), ([-1.1, -1.1, -1.0], [1.1, 1.1, 1.0])
    cases = [(unit, [0, 0, -2], [0, 0, 1], 1.0, ("ng", [0, 0, -1])), (wide, [0, 0, -2], [1, 0, 1], 1.0, ("ng", [0, 0, -1])),
             (wide, [0, 0, -2], [1, 1, 1], 1.0, ("ng", [0, 0, -1])), (unit, [0, 0, 0], [0, 0, 1], 1.0, None),
             (unit, [0, 0, 0], [0, -1, 0], 1.0, None), (unit, [0.5, 0.5, 0.5], [1, 0, 1], None, None),
             (unit, [0, 0, 2], [0, 0, -1], 1.0, ("ng", [0, 0, 1])), (unit, [0, 2, 0], [0, -1, 0], 1.0, ("ns", [0, 1, 0])),
             (unit, [0, -2, 0], [0, 1, 0], 1.0, ("ns", [0, -1, 0])), (unit, [0, 2, 2], [0, -0.5, -1], 2.0, ("ng", [0, 1, 0]))]
    for (mn, mx), o, d, t_exp, normal in cases:
        i, t, ng, ns = one(oracle, box_scene(mn, mx), o, d)
        assert i == 0, (o, d)
        if t_exp is not None:
            assert t == t_exp, (o, d, t)
        if normal:
            assert veq(ng if normal[0] == "ng" else ns, normal[1]), (o, d, ng, ns)
        assert abs(np.linalg.norm(ng) - 1.0) < 1e-15 and abs(np.linalg.norm(ns) - 1.0) < 1e-15, (o, d, ng, ns)


def test_trace_normals_triangle_vector(oracle):    # triangle.rs:411
    sc = Scene(); sc.root.add_obj_of(sc.parse_obj(PLANE), PLAST)
    i, t, ng, _ = one(oracle, sc, [0, 1, 0], [0, -1, 0])
    assert i == 0 and t == 1.0 and veq(ng, [0, 1, 0])


def test_trace_normals_swap_backface_in_scaled_group(oracle):
    """A unit cube inside a group scaled by (2, 1, 1): the record comes back through transform_isect, so ng is the outward face
    normal in world space; with swap_backface on the group the same ray reports the opposite ng and ns, at the same t."""
    def scene(swap):
        sc = Scene()
        g = Aggregate(); g.scale(2.0, 1.0, 1.0)
        if swap:
            g.swap_backface()
        g.add_cube([-0.5, -0.5, -0.5], 1.0, PLAST)
        sc.root.add_group(g)
        return sc
    rays = [([0.1, 0.2, 5.0], [0, 0, -1], [0, 0, 1]),          # z face: dpdu / dpdv span x and y, x is scaled
            ([5.0, 0.1, 0.2], [-1, 0, 0], [1, 0, 0]),          # x face at x = 1 (0.5 scaled by 2)
            ([0.3, -4.0, 0.1], [0, 1, 0], [0, -1, 0]),
            ([-6.0, 0.1, -0.2], [1, 0.01, 0.02], [-1, 0, 0])]
    for o, d, n_out in rays:
        i0, t0, ng0, ns0 = one(oracle, scene(False), o, d)
        i1, t1, ng1, ns1 = one(oracle, scene(True), o, d)
        assert i0 == i1 == 0 and t0 == t1 and np.isfinite(t0), (o, d, t0, t1)
        assert veq(ng0, n_out) and veq(ns0, n_out), (o, d, ng0, ns0)
        assert veq(ng1, -np.array(n_out, float)) and veq(ns1, -np.array(n_out, float)), (o, d, ng1, ns1)
    # a miss reports zeros, and without normals=True the entry point keeps its two outputs
    o = oracle.OracleScene(scene(False))
    ids, t, ng, ns = o.trace_rays(np.array([[0, 5.0, 5.0, 0, 0, 1.0]]), normals=True)
    assert ids[0] == oracle.MISS and t[0] == np.inf and not ng.any() and not ns.any()
    assert len(o.trace_rays(np.array([[0.1, 0.2, 5.0, 0, 0, -1.0]]))) == 2
