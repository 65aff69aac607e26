"""lgb_scene_set_camera / DeviceScene.set_camera / Accel.set_camera: new views of a resident scene.

A scene created with one camera and moved to another renders, bit for bit, what a scene created with the other camera renders
(every output and the outcome counters; the f32 padding differs, the exact tests do not), matches the oracle, follows the camera
in stream order, across film sizes, device groups and imported scenes, and refuses cameras whose origins leave the world box its
f32 error bound was derived from -- unless the view box declared at creation holds them."""
import ctypes as C
import math

import numpy as np
import pytest

from lasgun_b200 import api, parity, scenes

gpu = pytest.mark.gpu
OUTCOME = ("primary_rays", "primary_hits", "shadow_rays", "shadow_rays_traced", "shadow_occluded", "secondary_rays")


def camera(perspective, param, eye, look, up=(0.0, 1.0, 0.0), ss=0):
    c = api.Camera(perspective, param)
    c.look_at(list(eye), list(look), list(up))
    c.set_supersampling(ss)
    return c


def orbit(eye, look, deg):
    """`eye` turned by `deg` degrees about the vertical axis through `look`."""
    a = math.radians(deg)
    x, z = eye[0] - look[0], eye[2] - look[2]
    return (look[0] + x * math.cos(a) + z * math.sin(a), eye[1], look[2] - x * math.sin(a) + z * math.cos(a))


def view_box(cams, margin=1.0):
    """A box holding the origins of `cams`, orthographic ones widened by 2.5 |image_plane_height|."""
    lo, hi = np.full(3, np.inf), np.full(3, -np.inf)
    for c in cams:
        s = 0.0 if c.perspective else 2.5 * abs(c.param)
        e = np.array(c.look[0])
        lo, hi = np.minimum(lo, e - s), np.maximum(hi, e + s)
    return list(lo - margin), list(hi + margin)


def with_camera(make, cam):
    sc, _ = make()
    sc.set_camera(cam)
    return sc


def host_guides(g):
    out = {k: v.cpu().numpy() for k, v in g.items()}
    out["prim_id"] = out["prim_id"].view(np.uint32)
    return out


def frames(dev, w, h):
    """Every output of one view: RGBA8, linear film, guides, per-sample AOVs; and the outcome counters of capture and capture_aov."""
    rgba, st = dev.capture(w, h)
    lin = dev.capture_linear(w, h, want_stats=True)[0].cpu().numpy()
    g = host_guides(dev.capture_guides(w, h, want_stats=True)[0])
    aov = dev.capture_aov(w, h, li=True)
    out = {"rgba": rgba, "linear": lin, **{"guide_" + k: v for k, v in g.items()},
           "prim_id": aov["prim_id"], "t": aov["t"], "occl": aov["occl"], "li": aov["li"], "aov_rgba": aov["rgba"]}
    counts = {**{k: st[k] for k in OUTCOME}, **{"aov_" + k: aov["stats"][k] for k in OUTCOME}}
    return out, counts


def assert_same(a, b, what=""):
    assert a.keys() == b.keys()
    for k in a:
        assert np.array_equal(a[k], b[k], equal_nan=True), (what, k)


def fresh_frames(native, ctx, sc, w, h, lazy=False):
    dev = native.DeviceScene(ctx, native.FlatScene(sc, lazy=lazy))
    try:
        return frames(dev, w, h)
    finally:
        dev.destroy()


# ---------------------------------------------------------------------------------------------------- no GPU needed

def test_camera_describe_matches_flatten(native):
    """lgh_camera_describe replays HostScene's camera set-up: the lgb_camera FlatScene puts in the desc, bit for bit."""
    cams = [camera(True, 45.0, (25.0, 0.0, 800.0), (25.0, 0.0, 0.0)),
            camera(True, 50.0, (310.0, 60.0, -130.0), (0.0, 0.0, 0.0), ss=3),
            camera(False, 700.0, (40.0, 90.0, 520.0), (0.0, 0.0, 0.0), ss=2),
            camera(True, 60.0, (0.21, 0.13, 5.0), (0.0, 0.0, 0.0), up=(0.1, 1.0, 0.0), ss=16),
            api.Camera(False, 3.0)]                                  # no look_at: the constructor's frame
    for cam in cams:
        sc, _ = scenes.simple("b", 0, 16)
        sc.set_camera(cam)
        flat = native.FlatScene(sc)
        got = native.camera_desc(cam)
        assert bytes(got) == bytes(flat.desc.camera)
    with pytest.raises(native.LasgunError):
        bad = api.Camera(True, 45.0)
        bad.supersampling = 255                                      # set_supersampling refuses it on the host (camera.rs:189)
        native.camera_desc(bad)


def test_view_box_flag(native):
    """Without LGB_SCENE_VIEW_BOX the desc is the one of ABI v5 plus two zero boxes nobody reads; with it FlatScene sets the flag and
    the box, also after the reference tree of a lazy scene is built."""
    sc, _ = scenes.simple("b", 1, 64)
    flat = native.FlatScene(sc)
    assert flat.desc.abi_version == 6 and flat.desc.flags == 0
    assert list(flat.desc.view_lo) == [0.0] * 3 and list(flat.desc.view_hi) == [0.0] * 3
    def probe():
        return {k: v for k, v in flat.build_probe().items() if not k.endswith("_ms")}
    before = probe()
    assert before["ranks_ok"] == 1 and before["boxes_ok"] == 1
    flat.desc.view_lo[:] = [float("nan")] * 3; flat.desc.view_hi[:] = [-1e300] * 3
    assert probe() == before                                         # not read without the flag
    lazy = native.FlatScene(sc, lazy=True, view_box=([-1.0, -2.0, -3.0], [4.0, 5.0, 6.0]))
    for _ in range(2):
        assert lazy.desc.flags == native.LGB_SCENE_VIEW_BOX
        assert list(lazy.desc.view_lo) == [-1.0, -2.0, -3.0] and list(lazy.desc.view_hi) == [4.0, 5.0, 6.0]
        lazy.build_tree()
    assert native.lib().lgb_scene_set_camera(None, None, None) == native.LGB_ERR_INVALID


# ---------------------------------------------------------------------------------------------------- moved equals fresh

def _mixed():
    return scenes.mixed4k(mesh_n=64, nspheres=6000, res=(256, 144), supersampling=1)


MIXED_EYE, MIXED_LOOK = (0.0, 60.0, 520.0), (0.0, 0.0, 0.0)
CASES = {
    # camera grid, light grids, hit setup in k_cprimary
    "mixed_4spp": (_mixed, (256, 144), [camera(True, 50.0, orbit(MIXED_EYE, MIXED_LOOK, 40.0), MIXED_LOOK, ss=1)]),
    # BVH kernels
    "simple_b_9spp": (lambda: scenes.simple("b", 2, 192), (192, 192),
                      [camera(True, 45.0, orbit((25.0, 0.0, 800.0), (25.0, 0.0, 0.0), 30.0), (25.0, 0.0, 0.0), ss=2)]),
    # transformed groups: INST
    "cornell_groups_9spp": (lambda: scenes.cornell_groups((192, 192), 2, eye=(0.21, 0.13, 5.0)), (192, 192),
                            [camera(True, 60.0, orbit((0.21, 0.13, 5.0), (0.0, 0.0, 0.0), 20.0), (0.0, 0.3, 0.0), ss=2)]),
    "mixed_whitted_4spp": (lambda: scenes.mixed4k(mesh_n=64, nspheres=6000, res=(192, 108), supersampling=1, whitted=True), (192, 108),
                           [camera(True, 50.0, orbit(MIXED_EYE, MIXED_LOOK, -35.0), MIXED_LOOK, ss=1)]),
    # perspective -> orthographic -> perspective
    "perspective_orthographic": (_mixed, (192, 108), [camera(False, 700.0, (40.0, 90.0, 520.0), MIXED_LOOK, ss=2),
                                                      camera(True, 50.0, orbit(MIXED_EYE, MIXED_LOOK, 15.0), MIXED_LOOK, ss=1)]),
    # 1 -> 9 -> 289 samples per pixel
    "supersampling": (lambda: scenes.simple("b", 0, 48), (40, 24), [camera(True, 45.0, (25.0, 0.0, 800.0), (25.0, 0.0, 0.0), ss=2),
                                                                     camera(True, 45.0, (25.0, 0.0, 800.0), (25.0, 0.0, 0.0), ss=16)]),
}


@gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_moved_equals_fresh(native, gpu_ctx, name):
    make, (w, h), cams = CASES[name]
    sc, _ = make()
    box = view_box([sc.camera] + cams)
    whitted = (True, False) if "whitted" in name else (True,)
    dev = native.DeviceScene(gpu_ctx, native.FlatScene(sc, view_box=box))
    try:
        for wavefront in whitted:
            gpu_ctx.set_whitted(wavefront)
            for cam in cams:
                dev.set_camera(cam)
                assert dev.spp == cam.num_samples()
                got, counts = frames(dev, w, h)
                want, want_counts = fresh_frames(native, gpu_ctx, with_camera(make, cam), w, h)
                assert_same(got, want, (wavefront, cam.look))
                assert counts == want_counts, (counts, want_counts)
                assert counts["primary_rays"] == w * h * cam.num_samples()
                if "whitted" in name:
                    assert counts["secondary_rays"] > 0
    finally:
        gpu_ctx.set_whitted(True)
        dev.destroy()


@gpu
def test_deferred_bvh_moved_to_orthographic(native, gpu_ctx):
    """A scene created without its device BVH (the camera grid serves its primary rays) builds the tree at the first capture of an
    orthographic view, which the camera grid does not serve, and renders the fresh orthographic scene's frames."""
    make = lambda: scenes.mixed4k(mesh_n=130, nspheres=8000, res=(192, 108), supersampling=1)       # noqa: E731 (>= 32768 primitives)
    w, h = 192, 108
    ortho = camera(False, 700.0, (40.0, 90.0, 520.0), MIXED_LOOK, ss=1)
    try:
        gpu_ctx.set_lazy_bvh(1); gpu_ctx.set_camera_grid(1)
        sc, _ = make()
        dev = native.DeviceScene(gpu_ctx, native.FlatScene(sc, view_box=view_box([sc.camera, ortho])))
        try:
            bytes0 = dev.device_bytes
            first = dev.capture_linear(w, h, want_stats=True)[0].cpu().numpy()
            assert dev.device_bytes == bytes0                        # no tree yet: the camera grid served the frame
            dev.set_camera(ortho)
            got, counts = frames(dev, w, h)
            assert dev.device_bytes > bytes0                         # the tree was built for the orthographic view
            want, want_counts = fresh_frames(native, gpu_ctx, with_camera(make, ortho), w, h)
            assert_same(got, want)
            assert counts == want_counts
            dev.set_camera(sc.camera)
            assert np.array_equal(dev.capture_linear(w, h, want_stats=True)[0].cpu().numpy(), first)
        finally:
            dev.destroy()
    finally:
        gpu_ctx.set_lazy_bvh(-1); gpu_ctx.set_camera_grid(-1)


@gpu
def test_lazy_tree_fetched_by_a_later_view(native, gpu_ctx):
    """coincident_planes created with a view that meets no exact-t tie: the reference tree is not fetched.  Moved to its own camera,
    which meets thousands, the tree is fetched then, and the ids are the fresh scene's."""
    make = scenes.coincident_planes
    sc, (w, h) = make()
    tie_free = camera(True, 55.0, (0.0, 3.5, 6.0), (0.0, 6.0, -4.0))      # looks up over the floor and the boxes
    ties = sc.camera
    sc.set_camera(tie_free)
    flat = native.FlatScene(sc, lazy=True, view_box=view_box([tie_free, ties]))
    dev = native.DeviceScene(gpu_ctx, flat)
    try:
        out = dev.capture_aov(w, h)
        assert not flat.tree_built and out["stats"]["tie_retraces"] == 0
        dev.set_camera(ties)
        out = dev.capture_aov(w, h)
        assert flat.tree_built and out["stats"]["tie_retraces"] > 0
    finally:
        dev.destroy()
    fresh = native.DeviceScene(gpu_ctx, native.FlatScene(with_camera(make, ties), lazy=True))
    try:
        ref = fresh.capture_aov(w, h)
    finally:
        fresh.destroy()
    assert np.array_equal(out["prim_id"], ref["prim_id"]) and np.array_equal(out["t"], ref["t"], equal_nan=True)
    assert np.array_equal(out["rgba"], ref["rgba"])


@gpu
@pytest.mark.parametrize("name", ["simple_b_9spp", "cornell_groups_9spp", "mixed_4spp"])
def test_moved_against_oracle(native, oracle, gpu_ctx, name):
    make, (w, h), cams = CASES[name]
    cam = cams[0]
    sc, _ = make()
    dev = native.DeviceScene(gpu_ctx, native.FlatScene(sc, view_box=view_box([sc.camera, cam])))
    try:
        dev.set_camera(cam)
        out = dev.capture_aov(w, h)
        rgba, _ = dev.capture(w, h)
    finally:
        dev.destroy()
    ref = oracle.OracleScene(with_camera(make, cam)).capture(w, h, aov=True)
    a = parity.aov_report(out, ref)
    assert a["mismatches"] == 0 and a["hit_miss_flips"] == 0, a
    assert a["near_ties"] <= 1e-4 * a["samples"], a
    assert a["t_bit_equal"] == a["t_compared"] and a["occl_diff"] == 0, a
    f = parity.film_report(rgba, ref["rgba"])
    assert f["alpha_equal"] and f["within_1_frac"] >= 0.999 and f["identical_frac"] >= 0.9999, f


@gpu
def test_round_trip(native, gpu_ctx):
    """A -> B at another film size -> A: A's first frame, bit for bit (the camera grid is rebuilt for each view and size)."""
    sc, _ = _mixed()
    w, h = 256, 144
    a_cam = sc.camera
    b_cam = camera(True, 50.0, orbit(MIXED_EYE, MIXED_LOOK, 70.0), MIXED_LOOK, ss=1)
    dev = native.DeviceScene(gpu_ctx, native.FlatScene(sc, view_box=view_box([a_cam, b_cam])))
    try:
        first, counts = frames(dev, w, h)
        dev.set_camera(b_cam)
        dev.capture_linear(192, 160, want_stats=True)
        dev.set_camera(a_cam)
        again, counts2 = frames(dev, w, h)
    finally:
        dev.destroy()
    assert_same(first, again)
    assert counts == counts2


# ---------------------------------------------------------------------------------------------------- the world box

ORBIT = [camera(True, 50.0, orbit((0.0, 200.0, 900.0), MIXED_LOOK, 45.0 * k), MIXED_LOOK) for k in range(8)]
ORBIT_BOX = ([-950.0, 150.0, -950.0], [950.0, 250.0, 950.0])


@gpu
def test_view_box_accepts_an_orbit(native, gpu_ctx):
    """Eight views around the scene, all outside the box of the geometry and the first camera: refused by a scene created without a
    view box, accepted by one created with it, and each renders the fresh scene of that camera (created without a box)."""
    make = lambda: scenes.mixed4k(mesh_n=64, nspheres=6000, res=(128, 72), supersampling=0)        # noqa: E731
    w, h = 128, 72
    sc, _ = make()
    plain = native.DeviceScene(gpu_ctx, native.FlatScene(sc))
    boxed = native.DeviceScene(gpu_ctx, native.FlatScene(sc, view_box=ORBIT_BOX))
    try:
        for cam in ORBIT:
            with pytest.raises(native.LasgunError) as e:
                plain.set_camera(cam)
            assert e.value.status == native.LGB_ERR_UNSUPPORTED
            boxed.set_camera(cam)
            got, counts = frames(boxed, w, h)
            want, want_counts = fresh_frames(native, gpu_ctx, with_camera(make, cam), w, h)
            assert_same(got, want, cam.look)
            assert counts == want_counts
    finally:
        plain.destroy(); boxed.destroy()


@gpu
def test_refusals(native, gpu_ctx):
    """NULL, non-finite, supersampling_root 0 or 257: LGB_ERR_INVALID; outside the box, also by an orthographic camera's slack:
    LGB_ERR_UNSUPPORTED, with the box in the message.  After each the scene renders the frame it rendered before."""
    L = native.lib()
    sc, (w, h) = scenes.mixed4k(mesh_n=48, nspheres=3000, res=(96, 54), supersampling=1)
    dev = native.DeviceScene(gpu_ctx, native.FlatScene(sc, view_box=ORBIT_BOX))
    try:
        before = dev.capture_linear(w, h, want_stats=True)[0].cpu().numpy()
        rgba0, _ = dev.capture(w, h)
        good = native.camera_desc(ORBIT[3])

        def variant(**kw):
            d = native.CameraDesc.from_buffer_copy(good)
            for k, v in kw.items():
                if isinstance(v, tuple):
                    getattr(d, k)[v[0]] = v[1]
                else:
                    setattr(d, k, v)
            return d
        invalid = [None, variant(supersampling_root=0), variant(supersampling_root=257), variant(origin=(0, float("nan"))),
                   variant(view=(2, float("inf"))), variant(aux=(1, float("-inf"))), variant(image_plane_height=float("nan")),
                   variant(sample_distance=float("inf"))]
        for d in invalid:
            assert L.lgb_scene_set_camera(gpu_ctx.h, dev.h, C.byref(d) if d is not None else None) == native.LGB_ERR_INVALID
        assert L.lgb_scene_set_camera(None, dev.h, C.byref(good)) == native.LGB_ERR_INVALID
        outside = camera(True, 50.0, (0.0, 200.0, 1200.0), MIXED_LOOK)
        ortho_in = camera(False, 100.0, (0.0, 200.0, 900.0), MIXED_LOOK)         # origin inside, but 2.5 x 100 of slack is not
        persp_in = camera(True, 50.0, (0.0, 200.0, 900.0), MIXED_LOOK)
        for cam in (outside, ortho_in):
            rc = L.lgb_scene_set_camera(gpu_ctx.h, dev.h, C.byref(native.camera_desc(cam)))
            assert rc == native.LGB_ERR_UNSUPPORTED
            msg = L.lgb_last_error(gpu_ctx.h).decode()
            assert "box [-950, 950] x [" in msg and "LGB_SCENE_VIEW_BOX" in msg, msg
        assert dev.spp == 4
        assert np.array_equal(dev.capture_linear(w, h, want_stats=True)[0].cpu().numpy(), before)
        assert np.array_equal(dev.capture(w, h)[0], rgba0)
        dev.set_camera(persp_in)                                     # the same origin as a perspective camera is inside
        assert dev.spp == 1
    finally:
        dev.destroy()


# ---------------------------------------------------------------------------------------------------- stream order, groups, import, API

@gpu
@pytest.mark.parametrize("resize", [False, True])
def test_stream_order(native, gpu_ctx, resize):
    """capture_linear of A queued on one torch stream, set_camera(B), capture_linear of B queued on another, no host wait between:
    each film is its own view's, also when B's film has another size (both rebuild the camera grid behind A's capture)."""
    import torch
    sc, _ = _mixed()
    w, h = 256, 144
    w2, h2 = (200, 120) if resize else (w, h)
    a_cam, b_cam = sc.camera, camera(True, 50.0, orbit(MIXED_EYE, MIXED_LOOK, 50.0), MIXED_LOOK, ss=1)
    dev = native.DeviceScene(gpu_ctx, native.FlatScene(sc, view_box=view_box([a_cam, b_cam])))
    try:
        want_a = dev.capture_linear(w, h, want_stats=True)[0].cpu()
        dev.set_camera(b_cam)
        want_b = dev.capture_linear(w2, h2, want_stats=True)[0].cpu()
        dev.set_camera(a_cam)
        s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
        out_a = torch.full((h, w, 3), float("nan"), device="cuda")
        out_b = torch.full((h2, w2, 3), float("nan"), device="cuda")
        torch.cuda.synchronize()
        dev.capture_linear(w, h, out=out_a, stream=s1)
        dev.set_camera(b_cam)
        dev.capture_linear(w2, h2, out=out_b, stream=s2)
        torch.cuda.synchronize()
        assert torch.equal(out_a.cpu(), want_a) and torch.equal(out_b.cpu(), want_b)
    finally:
        dev.destroy()


@gpu
def test_device_group(native):
    """A device group's scene moves on every device: its frame is the moved one-GPU scene's."""
    if native.lib().lgb_device_count() < 2:
        pytest.skip("needs 2 GPUs")
    make, (w, h), cams = CASES["mixed_4spp"]
    sc, _ = make()
    box = view_box([sc.camera] + cams)
    one = native.Context(0)
    try:
        dev = native.DeviceScene(one, native.FlatScene(sc, view_box=box))
        dev.set_camera(cams[0])
        ref_lin = dev.capture_linear(w, h, want_stats=True)[0].cpu().numpy()
        ref_g = host_guides(dev.capture_guides(w, h, want_stats=True)[0])
        dev.destroy()
    finally:
        one.close()
    group = native.Context(devices=[0, 1])
    try:
        dev = native.DeviceScene(group, native.FlatScene(sc, view_box=box))
        try:
            dev.capture_linear(w, h, want_stats=True)                # the first view's camera grid on both devices
            dev.set_camera(cams[0])
            lin = dev.capture_linear(w, h, want_stats=True)[0].cpu().numpy()
            g = host_guides(dev.capture_guides(w, h, want_stats=True)[0])
        finally:
            dev.destroy()
    finally:
        group.close()
    assert np.array_equal(lin, ref_lin)
    assert_same(g, ref_g)


@gpu
def test_imported_scene(native, gpu_ctx):
    """An exported scene imported into a second context on the same GPU takes set_camera against the box of its layout."""
    import torch
    from lasgun_b200 import multi
    make, (w, h), cams = CASES["mixed_4spp"]
    sc, _ = make()
    dev = native.DeviceScene(gpu_ctx, native.FlatScene(sc, view_box=view_box([sc.camera] + cams)))
    other = native.Context(0)
    try:
        layout, ptr, nbytes = dev.export()
        arena = torch.as_tensor(multi._DevicePointer(ptr, nbytes), device="cuda").clone()
        twin = native.DeviceScene.adopt(other, layout, arena.data_ptr(), dev.spp, keep=arena)
        try:
            far = camera(True, 50.0, (0.0, 200.0, 1200.0), MIXED_LOOK)
            with pytest.raises(native.LasgunError) as e:
                twin.set_camera(far)
            assert e.value.status == native.LGB_ERR_UNSUPPORTED
            for d in (dev, twin):
                d.set_camera(cams[0])
            a = (dev.capture(w, h)[0], dev.capture_linear(w, h, want_stats=True)[0].cpu().numpy())
            b = (twin.capture(w, h)[0], twin.capture_linear(w, h, want_stats=True)[0].cpu().numpy())
        finally:
            twin.destroy()
    finally:
        dev.destroy(); other.close()
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


@gpu
def test_public_api(native, gpu_ctx):
    import lasgun_b200
    make, (w, h), cams = CASES["simple_b_9spp"]
    sc, _ = make()
    cam = cams[0]
    acc = lasgun_b200.Accel(sc, gpu_ctx, view_box=view_box([sc.camera, cam]))
    try:
        lin = acc.set_camera(cam).capture_linear(w, h).cpu().numpy()
        g = host_guides(acc.capture_guides(w, h))
    finally:
        acc.close()
    moved = with_camera(make, cam)
    assert np.array_equal(lin, lasgun_b200.capture_linear(moved, w, h, ctx=gpu_ctx).cpu().numpy())
    assert_same(g, host_guides(lasgun_b200.capture_guides(moved, w, h, ctx=gpu_ctx)))
