"""lgb_capture_guides / DeviceScene.capture_guides / lasgun_b200.capture_guides: per-pixel normal, depth, prim_id and coverage.

Against the oracle (ids and t of its capture, shading normals of its trace_rays on its own camera rays) on small scenes, against the
per-sample AOVs of lgb_capture_aov and the linear film of the same scene at full size, bit for bit across the ways a frame can be
rendered and between a colour frame and a geometry pass, in stream order, and refused without writing anything."""
import ctypes as C
import math

import numpy as np
import pytest

from lasgun_b200 import multi, scenes

pytestmark = pytest.mark.gpu

MISS = 0xFFFFFFFF
KEYS = ("normal", "depth", "prim_id", "coverage")

SMALL = {
    "simple_b_9spp": lambda: scenes.simple("b", 2, 192),
    "simple_a_1spp": lambda: scenes.simple("a", 0, 192),
    "cornell_4spp": lambda: scenes.cornell((320, 180), 1),
    "mixed_4spp": lambda: scenes.mixed4k(mesh_n=64, nspheres=6000, res=(256, 144), supersampling=1),
    "ragged_edges": lambda: scenes.simple("b", 1, 100)[0:1] + ((101, 67),),
    "cornell_groups_9spp": lambda: scenes.cornell_groups((192, 192), 2, eye=(0.21, 0.13, 5.0)),      # transformed groups: INST
    "nested_groups_root_4spp": lambda: scenes.nested_groups((160, 120), 1, transformed_root=True)[0:1] + ((160, 120),),
    "materials_depth8": lambda: scenes.materials((160, 120), 0, recursion=8),                          # smooth mesh in transformed groups
    "mixed_whitted_4spp": lambda: scenes.mixed4k(mesh_n=64, nspheres=6000, res=(192, 108), supersampling=1, whitted=True),
    "coincident_planes": lambda: scenes.coincident_planes(),                                           # exact-t ties (lazy tree)
}
FULL = {
    "C1_simple": lambda: scenes.simple("b", 2),
    "C2_mesh1m": scenes.mesh1m,
    "C3_cornell": scenes.cornell,
    "C4_spheres1m": scenes.spheres1m,
}


def _scene(name):
    if name in SMALL:
        return SMALL[name]()
    if name == "orthographic_9spp":
        sc, _ = scenes.mixed4k(mesh_n=48, nspheres=3000, res=(96, 54), supersampling=2)
        cam = sc.set_orthographic_camera(700.0)
        cam.look_at([40.0, 90.0, 520.0], [0.0, 0.0, 0.0], [0.0, 1.0, 0.0]); cam.set_supersampling(2)
        return sc, (96, 54)
    if name == "spp_289":                                # more samples than a block of k_guides holds: passes over one pixel
        sc, _ = scenes.simple("b", 0, 16)
        sc.camera.set_supersampling(16)
        return sc, (20, 12)
    raise KeyError(name)


def _flat(native, sc, name):
    return native.FlatScene(sc, lazy=(name == "coincident_planes"))


def view_len(flat):
    """|view| as the device forms it: sqrt((vx vx + vy vy) + vz vz) in f64."""
    v = [float(c) for c in flat.desc.camera.view]
    return math.sqrt((v[0] * v[0] + v[1] * v[1]) + v[2] * v[2])


def anchor(spp):
    r = math.isqrt(spp)
    return (r // 2) * r + r // 2                         # camera.rs:143


def reduce_aov(ids, t, w, h, spp, vlen):
    """depth, prim_id and coverage of per-sample ids and t (index (y w + x) spp + s), as lgb_capture_guides defines them."""
    ids = np.asarray(ids, np.uint32).reshape(h * w, spp); t = np.asarray(t, np.float64).reshape(h * w, spp)
    a = anchor(spp)
    with np.errstate(invalid="ignore"):
        depth = np.where(ids[:, a] == MISS, np.inf, t[:, a] * vlen).astype(np.float32)
    coverage = ((ids != MISS).sum(axis=1).astype(np.float64) / spp).astype(np.float32)
    return {"depth": depth.reshape(h, w), "prim_id": ids[:, a].reshape(h, w), "coverage": coverage.reshape(h, w)}


def host(g):
    """The guides as numpy, prim_id as the u32 it holds."""
    out = {k: v.cpu().numpy() for k, v in g.items()}
    if "prim_id" in out:
        out["prim_id"] = out["prim_id"].view(np.uint32)
    return out


def guides(native, ctx, flat, w, h, **kw):
    dev = native.DeviceScene(ctx, flat)
    try:
        g, st = dev.capture_guides(w, h, want_stats=True, **kw)
        return host(g), st
    finally:
        dev.destroy()


def f32_down(v):
    f = v.astype(np.float32)
    return np.where(f.astype(np.float64) > v, np.nextafter(f, np.float32(-np.inf)), f)


def f32_up(v):
    f = v.astype(np.float32)
    return np.where(f.astype(np.float64) < v, np.nextafter(f, np.float32(np.inf)), f)


def assert_same_guides(a, b, what=""):
    for k in KEYS:
        assert np.array_equal(a[k], b[k], equal_nan=True), (what, k)


@pytest.mark.parametrize("name", sorted(SMALL) + ["orthographic_9spp", "spp_289"])
def test_oracle_parity(native, oracle, gpu_ctx, name):
    sc, (w, h) = _scene(name)
    spp = sc.camera.num_samples()
    flat = _flat(native, sc, name)
    got, st = guides(native, gpu_ctx, flat, w, h)
    assert st["primary_rays"] == w * h * spp and st["stack_overflow"] == 0
    o = oracle.OracleScene(sc)
    ref = o.capture(w, h, aov=True)
    want = reduce_aov(ref["prim_id"], ref["t"], w, h, spp, view_len(flat))
    assert got["prim_id"].dtype == np.uint32 and got["depth"].dtype == np.float32 and got["normal"].shape == (h, w, 3)
    assert np.array_equal(got["prim_id"], want["prim_id"])
    assert np.array_equal(got["coverage"], want["coverage"])
    assert np.array_equal(got["depth"], want["depth"])           # float32(t_ref |view|), +inf on a miss
    # reference normals: the oracle's shading normal of every camera ray, summed in sample order, times 1/spp
    rays = np.concatenate([o.camera_sample(x, y, w, h) for y in range(h) for x in range(w)])
    ids, _, _, ns = o.trace_rays(rays, normals=True)
    assert np.array_equal(ids, ref["prim_id"])                  # the oracle's rays are its capture's rays
    ns = ns.reshape(h * w, spp, 3)
    n = np.zeros((h * w, 3))
    for s in range(spp):
        n = n + ns[:, s]
    n = (n * (1.0 / spp)).reshape(h, w, 3)
    lo, hi = f32_down(n - 1e-12), f32_up(n + 1e-12)
    ok = (lo <= got["normal"]) & (got["normal"] <= hi)
    assert ok.all(), (int((~ok).sum()), float(np.abs(got["normal"] - n).max()))


@pytest.mark.parametrize("name", sorted(FULL) + ["mixed_4spp", "cornell_groups_9spp", "mixed_whitted_4spp", "spp_289"])
def test_same_frame_as_colour(native, gpu_ctx, name):
    """rgb is the film of capture_linear; depth, prim_id and coverage are the reduction of lgb_capture_aov's per-sample ids and t."""
    sc, ((w, h)) = FULL[name]() if name in FULL else _scene(name)
    spp = sc.camera.num_samples()
    flat = native.FlatScene(sc)
    dev = native.DeviceScene(gpu_ctx, flat)
    try:
        g, st = dev.capture_guides(w, h, want_stats=True)
        lin = dev.capture_linear(w, h, want_stats=True)[0].cpu().numpy()
        got = host(g)
        del g
        aov = dev.capture_aov(w, h)
    finally:
        dev.destroy()
    assert st["primary_rays"] == w * h * spp and st["stack_overflow"] == 0
    assert np.array_equal(got["rgb"], lin)
    want = reduce_aov(aov["prim_id"], aov["t"], w, h, spp, view_len(flat))
    for k in ("depth", "prim_id", "coverage"):
        assert np.array_equal(got[k], want[k]), k
    hit = got["prim_id"] != MISS
    assert np.isfinite(got["normal"]).all() and (got["normal"][got["coverage"] == 0] == 0).all()
    assert np.isfinite(got["depth"][hit]).all() and np.isinf(got["depth"][~hit]).all()


@pytest.mark.parametrize("name", ["mixed_4spp", "simple_b_9spp", "cornell_groups_9spp", "mixed_whitted_4spp", "orthographic_9spp",
                                  "coincident_planes"])
def test_geometry_pass(native, gpu_ctx, name):
    """rgb=False: no shadow, shading or Whitted kernel, and the same guides bit for bit."""
    sc, (w, h) = _scene(name)
    spp = sc.camera.num_samples()
    flat = _flat(native, sc, name)
    dev = native.DeviceScene(gpu_ctx, flat)
    try:
        full, st_full = dev.capture_guides(w, h, want_stats=True)
        geo, st = dev.capture_guides(w, h, rgb=False, want_stats=True)
        only = dev.capture_guides(w, h, rgb=False, normal=False, depth=False, prim_id=False)       # coverage alone
        only = host(only)
        full, geo = host(full), host(geo)
    finally:
        dev.destroy()
    assert "rgb" not in geo and set(only) == {"coverage"}
    assert_same_guides(full, geo)
    assert np.array_equal(only["coverage"], full["coverage"])
    assert st["shadow_rays_traced"] == 0 and st["shadow_occluded"] == 0 and st["secondary_rays"] == 0 and st["shadow_rays"] == 0
    assert st["primary_rays"] == w * h * spp and st["primary_hits"] == st_full["primary_hits"]
    assert st["primary_hits"] == int(np.rint(geo["coverage"].astype(np.float64) * spp).sum())
    assert st["kernel_launches"] < st_full["kernel_launches"]
    if name == "mixed_whitted_4spp":
        assert st_full["secondary_rays"] > 0


@pytest.mark.parametrize("name", ["mixed_4spp", "simple_b_9spp", "cornell_groups_9spp", "spp_289"])
def test_path_invariance(native, gpu_ctx, name):
    """Light grids, camera grid, pixel beams, bands and tile ranks change how the frame is rendered, not one bit of its guides."""
    import torch
    sc, (w, h) = _scene(name)
    flat = native.FlatScene(sc)
    runs = {}
    try:
        for grids in (0, 1):
            gpu_ctx.set_light_grids(grids)
            dev = native.DeviceScene(gpu_ctx, flat)
            try:
                for cam in (0, 1):
                    gpu_ctx.set_camera_grid(cam)
                    for beams in (0, 1):
                        gpu_ctx.set_beams(beams)
                        for rgb in (True, False):
                            runs[(grids, cam, beams, rgb)] = host(dev.capture_guides(w, h, rgb=rgb, want_stats=True)[0])
                gpu_ctx.set_camera_grid(-1); gpu_ctx.set_beams(-1)
                if grids:
                    gpu_ctx.set_wave_budget_mb(1)
                    try:
                        banded, st = dev.capture_guides(w, h, want_stats=True)
                        banded_geo = dev.capture_guides(w, h, rgb=False, want_stats=True)[0]
                    finally:
                        gpu_ctx.set_wave_budget_mb(16384)
                    one, st1 = dev.capture_guides(w, h, want_stats=True)
                    assert st1["bands"] == 1 and (st["bands"] > 1 or name == "spp_289")      # (spp_289: one macro tile, one band)
                    assert_same_guides(host(banded), host(one), "bands")
                    assert_same_guides(host(banded_geo), host(one), "bands, geometry pass")
                    ranks = 4
                    owner = torch.from_numpy(multi.tile_owner_map(w, h, ranks)).cuda()
                    acc = {"normal": torch.full((h, w, 3), float("nan"), device="cuda"), "depth": torch.full((h, w), float("nan"), device="cuda"),
                           "coverage": torch.full((h, w), float("nan"), device="cuda"),
                           "prim_id": torch.full((h, w), 0x7EEEEEEE, dtype=torch.int32, device="cuda")}
                    for r in range(ranks):
                        dev.capture_guides(w, h, rgb=False, out=acc, rank=r, ranks=ranks, want_stats=True)
                        done = owner <= r
                        for k in ("normal", "depth", "coverage"):
                            assert not torch.isnan(acc[k][done]).any() and torch.isnan(acc[k][~done]).all(), (r, k)   # other tiles stay NaN
                        assert (acc["prim_id"][~done] == 0x7EEEEEEE).all()
                    assert_same_guides(host(acc), host(one), "tile ranks")
            finally:
                dev.destroy()
    finally:
        gpu_ctx.set_light_grids(-1); gpu_ctx.set_camera_grid(-1); gpu_ctx.set_beams(-1); gpu_ctx.set_wave_budget_mb(16384)
    first = next(iter(runs.values()))
    for k, g in runs.items():
        assert_same_guides(g, first, k)


def test_whitted_wavefront_and_per_tree(native, gpu_ctx):
    """LGB_OPT_WHITTED 1 (levels) and 0 (k_secondary): the guides describe the camera ray's first hit and do not move."""
    sc, (w, h) = SMALL["mixed_whitted_4spp"]()
    dev = native.DeviceScene(gpu_ctx, native.FlatScene(sc))
    try:
        levels = host(dev.capture_guides(w, h, want_stats=True)[0])
        gpu_ctx.set_whitted(False)
        per_tree = host(dev.capture_guides(w, h, want_stats=True)[0])
    finally:
        gpu_ctx.set_whitted(True)
        dev.destroy()
    assert_same_guides(levels, per_tree)


def test_device_group(native):
    """A 2-GPU device group in one process: the peer's tiles are stored into the leader's buffers; the guides are the one-GPU guides."""
    if native.lib().lgb_device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch
    sc, (w, h) = SMALL["mixed_4spp"]()
    one = native.Context(0)
    try:
        ref, _ = guides(native, one, native.FlatScene(sc), w, h)
    finally:
        one.close()
    group = native.Context(devices=[0, 1])
    try:
        assert group.n_devices == 2
        dev = native.DeviceScene(group, native.FlatScene(sc))
        try:
            for rgb in (True, False):
                out = {"normal": torch.full((h, w, 3), float("nan"), device="cuda:0"), "depth": torch.full((h, w), float("nan"), device="cuda:0"),
                       "coverage": torch.full((h, w), float("nan"), device="cuda:0"), "prim_id": torch.zeros((h, w), dtype=torch.int32, device="cuda:0")}
                if rgb:
                    out["rgb"] = torch.full((h, w, 3), float("nan"), device="cuda:0")
                got = host(dev.capture_guides(w, h, rgb=rgb, out=out, want_stats=True)[0])
                assert_same_guides(got, ref, rgb)
                if rgb:
                    assert np.array_equal(got["rgb"], ref["rgb"])
        finally:
            dev.destroy()
    finally:
        group.close()


def test_stream_order(native, gpu_ctx):
    """Asynchronous renders on a side stream and on torch's default stream, read on the same stream without a host wait."""
    import torch
    sc, (w, h) = SMALL["mixed_4spp"]()
    dev = native.DeviceScene(gpu_ctx, native.FlatScene(sc))
    try:
        want = host(dev.capture_guides(w, h, want_stats=True)[0])

        def fresh_out():
            return {"rgb": torch.empty((h, w, 3), device="cuda"), "normal": torch.empty((h, w, 3), device="cuda"),
                    "depth": torch.empty((h, w), device="cuda"), "coverage": torch.empty((h, w), device="cuda"),
                    "prim_id": torch.empty((h, w), dtype=torch.int32, device="cuda")}
        out = fresh_out()
        s = torch.cuda.Stream()
        with torch.cuda.stream(s):
            for v in out.values():
                v.fill_(-3)
            res = dev.capture_guides(w, h, out=out, stream=s)
            assert all(res[k] is out[k] for k in out)
            got = {k: v.to("cpu", non_blocking=False) for k, v in out.items()}      # queued on s behind the render
        got = host(got)
        assert_same_guides(got, want, "side stream"); assert np.array_equal(got["rgb"], want["rgb"])
        for rgb in (True, False):                             # the default (legacy) stream: clear, render, read, all queued
            for v in out.values():
                v.fill_(-3)
            o = dict(out) if rgb else {k: v for k, v in out.items() if k != "rgb"}
            dev.capture_guides(w, h, rgb=rgb, out=o)
            got = host({k: v.cpu() for k, v in o.items()})
            assert_same_guides(got, want, ("default stream", rgb))
            if rgb:
                assert np.array_equal(got["rgb"], want["rgb"])
        g = dev.capture_guides(w, h)
        assert g["prim_id"].dtype == torch.int32 and g["normal"].shape == (h, w, 3) and g["depth"].device == torch.device("cuda", gpu_ctx.device)
        assert_same_guides(host(g), want, "fresh")
    finally:
        dev.destroy()


def test_public_api(native, gpu_ctx):
    import lasgun_b200
    sc, (w, h) = SMALL["cornell_4spp"]()
    g = lasgun_b200.capture_guides(sc, w, h, ctx=gpu_ctx)
    geo = lasgun_b200.capture_guides(sc, w, h, rgb=False, ctx=gpu_ctx)
    acc = lasgun_b200.Accel(sc, gpu_ctx)
    try:
        again = acc.capture_guides(w, h)
    finally:
        acc.close()
    assert set(g) == {"rgb", *KEYS} and set(geo) == set(KEYS)
    g, geo, again = host(g), host(geo), host(again)
    assert_same_guides(g, again); assert_same_guides(g, geo)
    assert np.array_equal(g["rgb"], again["rgb"])
    assert np.array_equal(g["rgb"], lasgun_b200.capture_linear(sc, w, h, ctx=gpu_ctx).cpu().numpy())


def test_refusals(native, gpu_ctx):
    """No outputs, a bad film size and a scene of another context: LGB_ERR_INVALID; wrong tensors: ValueError.  Nothing is written."""
    import torch
    L = native.lib()
    sc, (w, h) = scenes.simple("b", 1, 64)
    dev = native.DeviceScene(gpu_ctx, native.FlatScene(sc))
    other = native.Context(0)
    odev = native.DeviceScene(other, native.FlatScene(sc))
    try:
        bufs = {"rgb": torch.full((h, w, 3), 7.0, device="cuda"), "normal": torch.full((h, w, 3), 7.0, device="cuda"),
                "depth": torch.full((h, w), 7.0, device="cuda"), "coverage": torch.full((h, w), 7.0, device="cuda"),
                "prim_id": torch.full((h, w), 7, dtype=torch.int32, device="cuda")}
        full = native.Guides(*[bufs[k].data_ptr() for k in native.DeviceScene.GUIDES])
        empty = native.Guides()
        st = native.Stats()
        assert L.lgb_capture_guides(gpu_ctx.h, dev.h, w, h, 0, 1, None, None, C.byref(st)) == native.LGB_ERR_INVALID
        assert L.lgb_capture_guides(gpu_ctx.h, dev.h, w, h, 0, 1, C.byref(empty), None, C.byref(st)) == native.LGB_ERR_INVALID
        assert L.lgb_capture_guides(gpu_ctx.h, dev.h, 0, h, 0, 1, C.byref(full), None, C.byref(st)) == native.LGB_ERR_INVALID
        assert L.lgb_capture_guides(gpu_ctx.h, dev.h, w, 0, 0, 1, C.byref(full), None, None) == native.LGB_ERR_INVALID
        assert L.lgb_capture_guides(gpu_ctx.h, odev.h, w, h, 0, 1, C.byref(full), None, C.byref(st)) == native.LGB_ERR_INVALID
        with pytest.raises(ValueError):
            dev.capture_guides(w, h, rgb=False, normal=False, depth=False, prim_id=False, coverage=False)
        good = {k: v for k, v in bufs.items()}
        for key, bad in (("normal", torch.zeros((h, w, 3), dtype=torch.float64, device="cuda")),
                         ("normal", torch.zeros((h, w, 4), device="cuda")),
                         ("depth", torch.zeros((h, w))),
                         ("depth", torch.zeros((w, h), device="cuda").transpose(0, 1)),
                         ("prim_id", torch.zeros((h, w), dtype=torch.float32, device="cuda")),
                         ("coverage", torch.zeros((h, w, 1), device="cuda")),
                         ("rgb", torch.zeros((h, w, 3), dtype=torch.float16, device="cuda"))):
            with pytest.raises(ValueError):
                dev.capture_guides(w, h, out={**good, key: bad})
        with pytest.raises(ValueError):                       # a buffer for an output that was not requested
            dev.capture_guides(w, h, rgb=False, out=good)
        torch.cuda.synchronize()
        for k, v in bufs.items():
            assert (v == 7).all(), k
    finally:
        odev.destroy(); dev.destroy(); other.close()
