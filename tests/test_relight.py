"""lgb_scene_set_lights / DeviceScene.set_lights / Accel.set_lights: relighting a resident scene.

A scene created with one set of lights and relit with another renders, bit for bit, what a scene created with the other set renders
(every output and the outcome counters), whatever the count (0 to LGB_MAX_LIGHTS, across the light-grid limit), matches the oracle,
follows the lights in stream order, across device groups and imported scenes, and refuses lights whose position lies beyond the reach
of the shadow beams' f32 cull -- unless the view box declared at creation holds them."""
import ctypes as C
import math

import numpy as np
import pytest

from lasgun_b200 import parity, scenes

gpu = pytest.mark.gpu
OUTCOME = ("primary_rays", "primary_hits", "shadow_rays", "shadow_rays_traced", "shadow_occluded", "secondary_rays")
WHITE = [1.0, 0.0, 0.0]                                              # falloff of the configs' lights


def ring(n, radius, height, scale=1.0):
    """n lights on a horizontal circle (heights staggered), intensities summing to about 1.2."""
    out = []
    for k in range(n):
        a = 2.0 * math.pi * (k + 0.3) / max(n, 1)
        out.append(([radius * math.cos(a), height + 0.1 * radius * (k % 4), radius * math.sin(a)],
                    [1.2 / n, 0.9 / n + 0.01 * (k % 3), 0.6 / n], [1.0, 0.01 * (k % 2), 0.0]))
    return [(list(map(lambda v: v * scale, p)), i, f) for p, i, f in out]


def relit(make, lights, ambient=None):
    """The scene of `make` created with `lights` (and `ambient`, if given) in place of its own."""
    sc, _ = make()
    sc.lights = [tuple(list(map(float, v)) for v in l) for l in lights]
    if ambient is not None:
        sc.ambient = list(ambient)
    return sc


def host_guides(g):
    out = {k: v.cpu().numpy() for k, v in g.items()}
    out["prim_id"] = out["prim_id"].view(np.uint32)
    return out


def frames(dev, w, h):
    """Every output of one lighting: RGBA8, linear film, guides, per-sample AOVs; and the outcome counters of capture and capture_aov."""
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


def fresh_frames(native, ctx, sc, w, h, **flat_kw):
    dev = native.DeviceScene(ctx, native.FlatScene(sc, **flat_kw))
    try:
        return frames(dev, w, h)
    finally:
        dev.destroy()


# ---------------------------------------------------------------------------------------------------- no GPU needed

def test_light_records_match_flatten(native):
    """light_descs builds the lgb_light array FlatScene puts in the desc, byte for byte, for 0, 1, 2 and 32 lights."""
    for lights in ([], ring(1, 300.0, 200.0), scenes.mixed4k(mesh_n=8, nspheres=10, res=(8, 8))[0].lights, ring(32, 450.0, 300.0)):
        sc, _ = scenes.simple("b", 0, 16)
        sc.lights = list(lights)
        flat = native.FlatScene(sc)
        got = native.light_descs(lights)
        assert flat.desc.n_lights == len(lights) and len(got) == len(lights)
        assert C.sizeof(native.LightDesc) == 72
        if lights:
            assert bytes(got) == C.string_at(flat.desc.lights, 72 * len(lights))


def test_set_lights_symbol(native):
    assert "lgb_scene_set_lights" in native.ABI_SYMBOLS
    assert hasattr(C.CDLL(native.SO_PATH), "lgb_scene_set_lights")
    assert native.lib().lgb_scene_set_lights(None, None, None, 0, None) == native.LGB_ERR_INVALID


# ---------------------------------------------------------------------------------------------------- relit equals fresh

def _mixed():
    return scenes.mixed4k(mesh_n=64, nspheres=6000, res=(256, 144), supersampling=1)


def _mixed_whitted():
    return scenes.mixed4k(mesh_n=64, nspheres=6000, res=(192, 108), supersampling=1, whitted=True)


MIXED_A = _mixed()[0].lights
MIXED_B = [([-300.0, 450.0, 520.0], [0.7, 0.8, 0.9], WHITE), ([500.0, 300.0, 200.0], [0.5, 0.45, 0.4], WHITE)]
SIMPLE_FAR = [([-3000.0, 2500.0, 4000.0], [0.9, 0.9, 0.9], WHITE), ([400.0, 100.0, 150.0], [0.7, 0.0, 0.7], WHITE)]   # beyond the box, within 4 M
CASES = {
    # light grids, camera grid: the count walks 2 -> 1 -> 9 (no grids) -> 0 -> 32 -> 2
    "mixed_counts": (_mixed, (256, 144), None,
                     [(MIXED_B, None), (ring(1, 450.0, 350.0), None), (ring(9, 450.0, 300.0), None), ([], None),
                      (ring(32, 450.0, 300.0), None), (MIXED_A, None)]),
    # BVH shadow rays with shadow beams forced on (k_sbeam starts its f32 cull at the light), one light beyond the box
    "simple_beams": (lambda: scenes.simple("b", 2, 96), (96, 96), 1, [(SIMPLE_FAR, None), (ring(3, 900.0, 300.0), [0.1, 0.2, 0.3])]),
    # transformed groups
    "cornell_groups": (lambda: scenes.cornell_groups((128, 128), 2, eye=(0.21, 0.13, 5.0)), (128, 128), None,
                       [([([0.5, 1.5, 0.8], [0.9, 0.8, 0.7], WHITE)], None), (ring(2, 1.5, 1.0), None)]),
    # Whitted, both forms
    "mixed_whitted": (_mixed_whitted, (192, 108), None, [(MIXED_B, None), (ring(3, 450.0, 350.0), [0.05, 0.1, 0.2])]),
    # ambient only, intensity / falloff only: nothing is rebuilt
    "ambient_only": (_mixed, (256, 144), None, [(MIXED_A, [0.3, 0.05, 0.15])]),
    "intensity_only": (_mixed, (256, 144), None,
                       [([(p, [1.7, 0.2, 0.5], [1.0, 0.002, 0.0]) for p, _, _ in MIXED_A], None)]),
}


@gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_relit_equals_fresh(native, gpu_ctx, name):
    make, (w, h), beams, steps = CASES[name]
    sc, _ = make()
    whitted = (True, False) if "whitted" in name else (True,)
    if beams is not None:
        gpu_ctx.set_beams(beams)
    dev = native.DeviceScene(gpu_ctx, native.FlatScene(sc))
    try:
        for wavefront in whitted:
            gpu_ctx.set_whitted(wavefront)
            for lights, ambient in steps:
                amb = ambient if ambient is not None else sc.ambient
                dev.set_lights(lights, amb)
                got, counts = frames(dev, w, h)
                want, want_counts = fresh_frames(native, gpu_ctx, relit(make, lights, amb), w, h)
                assert_same(got, want, (wavefront, len(lights)))
                assert counts == want_counts, (len(lights), counts, want_counts)
                assert counts["shadow_rays"] <= counts["primary_hits"] * len(lights)
                if "whitted" in name:
                    assert counts["secondary_rays"] > 0
    finally:
        gpu_ctx.set_whitted(True)
        gpu_ctx.set_beams(-1)
        dev.destroy()


@gpu
def test_deferred_bvh_relit_past_the_grids(native, gpu_ctx):
    """A scene created without its device BVH (camera grid + light grids serve the frame) relit with 9 lights, which the light grids do
    not take: the next capture builds the tree and renders the fresh 9-light scene; back at 2 lights the grids return and the frame is
    the first one."""
    make = lambda: scenes.mixed4k(mesh_n=130, nspheres=8000, res=(192, 108), supersampling=1)       # noqa: E731 (>= 32768 primitives)
    w, h = 192, 108
    nine = ring(9, 450.0, 300.0)
    try:
        gpu_ctx.set_lazy_bvh(1); gpu_ctx.set_camera_grid(1)
        sc, _ = make()
        dev = native.DeviceScene(gpu_ctx, native.FlatScene(sc))
        try:
            bytes0 = dev.device_bytes
            first = dev.capture_linear(w, h, want_stats=True)[0].cpu().numpy()
            assert dev.device_bytes == bytes0                        # no tree: the grids served the frame
            dev.set_lights(nine, sc.ambient)
            got, counts = frames(dev, w, h)
            want, want_counts = fresh_frames(native, gpu_ctx, relit(make, nine), w, h)
            assert_same(got, want)
            assert counts == want_counts
            dev.set_lights(sc.lights, sc.ambient)
            again = dev.capture_linear(w, h, want_stats=True)[0].cpu().numpy()
            assert dev.device_bytes > bytes0                         # the same grids again, and now the tree
            assert np.array_equal(first, again)
        finally:
            dev.destroy()
    finally:
        gpu_ctx.set_lazy_bvh(-1); gpu_ctx.set_camera_grid(-1)


@gpu
@pytest.mark.parametrize("name", ["simple_b_9spp", "mixed_4spp"])
def test_relit_against_oracle(native, oracle, gpu_ctx, name):
    if name == "simple_b_9spp":
        make, (w, h), lights = (lambda: scenes.simple("b", 2, 128)), (128, 128), SIMPLE_FAR
    else:
        make, (w, h), lights = _mixed, (256, 144), MIXED_B
    sc, _ = make()
    amb = [0.15, 0.1, 0.05]
    dev = native.DeviceScene(gpu_ctx, native.FlatScene(sc))
    try:
        dev.set_lights(lights, amb)
        out = dev.capture_aov(w, h)
        rgba, _ = dev.capture(w, h)
    finally:
        dev.destroy()
    ref = oracle.OracleScene(relit(make, lights, amb)).capture(w, h, aov=True)
    a = parity.aov_report(out, ref)
    assert a["mismatches"] == 0 and a["hit_miss_flips"] == 0, a
    assert a["near_ties"] <= 1e-4 * a["samples"], a
    assert a["t_bit_equal"] == a["t_compared"] and a["occl_diff"] == 0, a
    f = parity.film_report(rgba, ref["rgba"])
    assert f["alpha_equal"] and f["within_1_frac"] >= 0.999 and f["identical_frac"] >= 0.9999, f


@gpu
def test_round_trip(native, gpu_ctx):
    """A -> B (moved, other intensities, other ambient) -> A: A's first frame, bit for bit."""
    sc, _ = _mixed()
    w, h = 256, 144
    dev = native.DeviceScene(gpu_ctx, native.FlatScene(sc))
    try:
        first, counts = frames(dev, w, h)
        dev.set_lights(MIXED_B, [0.3, 0.3, 0.3])
        dev.capture_linear(w, h, want_stats=True)
        dev.set_lights(sc.lights, sc.ambient)
        again, counts2 = frames(dev, w, h)
    finally:
        dev.destroy()
    assert_same(first, again)
    assert counts == counts2


# ---------------------------------------------------------------------------------------------------- stream order

@gpu
@pytest.mark.parametrize("moved", [False, True])
def test_stream_order(native, gpu_ctx, moved):
    """capture_linear with A queued on one torch stream, set_lights(B), capture_linear queued on another, no host wait between: each
    film is its own lighting's -- with B a new intensity (the slot is rewritten behind A's capture) and with B a moved light (the light
    grids are rebuilt behind it too)."""
    import torch
    sc, _ = _mixed()
    w, h = 256, 144
    a_lights = sc.lights
    b_lights = MIXED_B if moved else [(p, [1.5, 0.1, 0.3], f) for p, _, f in a_lights]
    b_amb = [0.25, 0.0, 0.1]
    dev = native.DeviceScene(gpu_ctx, native.FlatScene(sc))
    try:
        want_a = dev.capture_linear(w, h, want_stats=True)[0].cpu()
        dev.set_lights(b_lights, b_amb)
        want_b = dev.capture_linear(w, h, want_stats=True)[0].cpu()
        assert not torch.equal(want_a, want_b)
        dev.set_lights(a_lights, sc.ambient)
        s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
        out_a = torch.full((h, w, 3), float("nan"), device="cuda")
        out_b = torch.full((h, w, 3), float("nan"), device="cuda")
        torch.cuda.synchronize()
        dev.capture_linear(w, h, out=out_a, stream=s1)
        dev.set_lights(b_lights, b_amb)
        dev.capture_linear(w, h, out=out_b, stream=s2)
        torch.cuda.synchronize()
        assert torch.equal(out_a.cpu(), want_a) and torch.equal(out_b.cpu(), want_b)
    finally:
        dev.destroy()


# ---------------------------------------------------------------------------------------------------- refusals and the reach

@gpu
def test_refusals(native, gpu_ctx):
    """NULL arguments, a scene of another context, non-finite components: LGB_ERR_INVALID; 33 lights and a light beyond 4 M:
    LGB_ERR_UNSUPPORTED, the box named in the message.  After each the scene renders the frames it rendered before."""
    L = native.lib()
    sc, _ = scenes.mixed4k(mesh_n=48, nspheres=3000, res=(96, 54), supersampling=1)
    w, h = 96, 54
    dev = native.DeviceScene(gpu_ctx, native.FlatScene(sc))
    other = native.Context(0)
    try:
        before = dev.capture_linear(w, h, want_stats=True)[0].cpu().numpy()
        rgba0, _ = dev.capture(w, h)
        good = native.light_descs(MIXED_B)
        amb = native._d3([0.1, 0.1, 0.1])

        def variant(i, field, k, v):
            d = native.light_descs(MIXED_B)
            getattr(d[i], field)[k] = v
            return d
        for ctx_h, scene_h, lights, n, a in ((None, dev.h, good, 2, amb), (gpu_ctx.h, None, good, 2, amb), (gpu_ctx.h, dev.h, good, 2, None),
                                             (gpu_ctx.h, dev.h, None, 2, amb), (other.h, dev.h, good, 2, amb)):
            assert L.lgb_scene_set_lights(ctx_h, scene_h, lights, n, a) == native.LGB_ERR_INVALID
        for d in (variant(0, "position", 1, float("nan")), variant(1, "intensity", 2, float("inf")), variant(0, "falloff", 0, float("-inf"))):
            assert L.lgb_scene_set_lights(gpu_ctx.h, dev.h, d, 2, amb) == native.LGB_ERR_INVALID
        assert L.lgb_scene_set_lights(gpu_ctx.h, dev.h, good, 2, native._d3([0.1, float("nan"), 0.1])) == native.LGB_ERR_INVALID
        many = native.light_descs(ring(33, 450.0, 300.0))
        assert L.lgb_scene_set_lights(gpu_ctx.h, dev.h, many, 33, amb) == native.LGB_ERR_UNSUPPORTED
        for far in ([2401.0, 0.0, 0.0], [0.0, -2500.0, 0.0], [0.0, 300.0, 1e6]):            # M = 600 (the ground box): 4 M = 2400
            d = native.light_descs([MIXED_B[0], (far, [0.5, 0.5, 0.5], WHITE)])
            assert L.lgb_scene_set_lights(gpu_ctx.h, dev.h, d, 2, amb) == native.LGB_ERR_UNSUPPORTED
            msg = L.lgb_last_error(gpu_ctx.h).decode()
            assert "light 1 at" in msg and "box [-600, 600] x [" in msg and "LGB_SCENE_VIEW_BOX" in msg, msg
        assert np.array_equal(dev.capture_linear(w, h, want_stats=True)[0].cpu().numpy(), before)
        assert np.array_equal(dev.capture(w, h)[0], rgba0)
        dev.set_lights([([2400.0, -2400.0, 2400.0], [0.9, 0.9, 0.9], WHITE)], [0.1, 0.1, 0.1])     # exactly 4 M: accepted
        dev.set_lights([], [0.1, 0.1, 0.1])
    finally:
        dev.destroy(); other.close()


@gpu
def test_view_box_holds_a_far_light(native, gpu_ctx):
    """A light beyond the reach of a plain scene is accepted by the scene whose view box holds it, and that scene relit renders the
    fresh scene created with the light (and the same view box), shadow beams on."""
    make = lambda: scenes.simple("b", 2, 96)                          # noqa: E731
    w, h = 96, 96
    far = [([-9000.0, 12000.0, 9500.0], [1.6, 1.5, 1.4], WHITE)]      # M = 2200 (the large sphere), 4 M = 8800
    box = ([-9001.0, -10.0, -10.0], [10.0, 12001.0, 9501.0])
    sc, _ = make()
    plain = native.DeviceScene(gpu_ctx, native.FlatScene(sc))
    boxed = native.DeviceScene(gpu_ctx, native.FlatScene(sc, view_box=box))
    try:
        gpu_ctx.set_beams(1)
        with pytest.raises(native.LasgunError) as e:
            plain.set_lights(far, sc.ambient)
        assert e.value.status == native.LGB_ERR_UNSUPPORTED
        boxed.set_lights(far, sc.ambient)
        got, counts = frames(boxed, w, h)
        want, want_counts = fresh_frames(native, gpu_ctx, relit(make, far), w, h, view_box=box)
        assert_same(got, want)
        assert counts == want_counts
    finally:
        gpu_ctx.set_beams(-1)
        plain.destroy(); boxed.destroy()


@gpu
def test_creation_lights_of_every_config_accepted(native, gpu_ctx):
    """Every config's own lights lie within the reach of its scene created without a view box (mesh1m's at 1.25 M, mixed4k's and
    spheres1m's outside the box)."""
    for name, make in sorted(scenes.CONFIGS.items()):
        sc, _ = make()
        dev = native.DeviceScene(gpu_ctx, native.FlatScene(sc, lazy=True))
        try:
            dev.set_lights(sc.lights, sc.ambient)
        finally:
            dev.destroy()


# ---------------------------------------------------------------------------------------------------- groups, import, API

@gpu
def test_device_group(native):
    """A device group's scene relit on every device: its frames are the relit one-GPU scene's (a moved light, then 9 lights)."""
    if native.lib().lgb_device_count() < 2:
        pytest.skip("needs 2 GPUs")
    sc, _ = _mixed()
    w, h = 256, 144
    steps = [(MIXED_B, [0.2, 0.1, 0.0]), (ring(9, 450.0, 300.0), [0.1, 0.1, 0.1])]
    ref = []
    one = native.Context(0)
    try:
        dev = native.DeviceScene(one, native.FlatScene(sc))
        for lights, amb in steps:
            dev.set_lights(lights, amb)
            ref.append((dev.capture_linear(w, h, want_stats=True)[0].cpu().numpy(), host_guides(dev.capture_guides(w, h, want_stats=True)[0])))
        dev.destroy()
    finally:
        one.close()
    group = native.Context(devices=[0, 1])
    try:
        dev = native.DeviceScene(group, native.FlatScene(sc))
        try:
            dev.capture_linear(w, h, want_stats=True)                # the creation lights' frame on both devices
            for (lights, amb), (lin_ref, g_ref) in zip(steps, ref):
                dev.set_lights(lights, amb)
                lin = dev.capture_linear(w, h, want_stats=True)[0].cpu().numpy()
                g = host_guides(dev.capture_guides(w, h, want_stats=True)[0])
                assert np.array_equal(lin, lin_ref)
                assert_same(g, g_ref)
        finally:
            dev.destroy()
    finally:
        group.close()


@gpu
def test_imported_scene(native, gpu_ctx):
    """An exported scene imported into a second context on the same GPU takes set_lights in its own arena and grids: relit, it renders
    what the relit original renders, and the original is not changed by the import's lights."""
    import torch
    from lasgun_b200 import multi
    sc, _ = _mixed()
    w, h = 256, 144
    dev = native.DeviceScene(gpu_ctx, native.FlatScene(sc))
    other = native.Context(0)
    try:
        dev.set_lights(MIXED_B, [0.2, 0.2, 0.2])                     # export carries the lights in effect
        layout, ptr, nbytes = dev.export()
        arena = torch.as_tensor(multi._DevicePointer(ptr, nbytes), device="cuda").clone()
        twin = native.DeviceScene.adopt(other, layout, arena.data_ptr(), dev.spp, keep=arena)
        try:
            assert np.array_equal(twin.capture(w, h)[0], dev.capture(w, h)[0])
            with pytest.raises(native.LasgunError) as e:
                twin.set_lights([([0.0, 3000.0, 0.0], [1.0, 1.0, 1.0], WHITE)], [0.1, 0.1, 0.1])
            assert e.value.status == native.LGB_ERR_UNSUPPORTED
            b_dev = dev.capture_linear(w, h, want_stats=True)[0].cpu().numpy()
            nine = ring(9, 450.0, 300.0)
            for d in (dev, twin):
                d.set_lights(nine, [0.1, 0.1, 0.1])
            a = (dev.capture(w, h)[0], dev.capture_linear(w, h, want_stats=True)[0].cpu().numpy())
            b = (twin.capture(w, h)[0], twin.capture_linear(w, h, want_stats=True)[0].cpu().numpy())
            twin.set_lights(sc.lights, sc.ambient)
            twin.capture_linear(w, h, want_stats=True)
            dev.set_lights(MIXED_B, [0.2, 0.2, 0.2])
            assert np.array_equal(dev.capture_linear(w, h, want_stats=True)[0].cpu().numpy(), b_dev)
        finally:
            twin.destroy()
    finally:
        dev.destroy(); other.close()
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


@gpu
def test_public_api(native, gpu_ctx):
    import lasgun_b200
    make = lambda: scenes.simple("b", 2, 128)                         # noqa: E731
    w, h = 128, 128
    sc, _ = make()
    amb = [0.05, 0.15, 0.1]
    acc = lasgun_b200.Accel(sc, gpu_ctx)
    try:
        lin = acc.set_lights(SIMPLE_FAR, amb).capture_linear(w, h).cpu().numpy()
    finally:
        acc.close()
    assert np.array_equal(lin, lasgun_b200.capture_linear(relit(make, SIMPLE_FAR, amb), w, h, ctx=gpu_ctx).cpu().numpy())
