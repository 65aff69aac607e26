"""lgb_capture_linear / DeviceScene.capture_linear / lasgun_b200.capture_linear: the linear float32 film.

Each pixel must be the f32 rounding of the colour the RGBA8 film quantises (the in-order sum of the samples times 1/spp,
integrate.rs:16-20): against the oracle's per-sample radiance on the small scenes, against the byte film at full size, bit for bit
across the ways a frame can be rendered, in stream order, and refused where lgb_capture_device refuses."""
import ctypes as C

import numpy as np
import pytest

from lasgun_b200 import multi, scenes

pytestmark = pytest.mark.gpu

# the plastic scenes: fused lean kernel (k_shade_lean), INST fused kernel (k_shade), k_resolve (spp > 256)
PLASTIC = {
    "simple_b_9spp": lambda: scenes.simple("b", 2, 192),
    "simple_a_1spp": lambda: scenes.simple("a", 0, 192),
    "cornell_4spp": lambda: scenes.cornell((320, 180), 1),
    "mixed_4spp": lambda: scenes.mixed4k(mesh_n=64, nspheres=6000, res=(256, 144), supersampling=1),
    "ragged_edges": lambda: scenes.simple("b", 1, 100)[0:1] + ((101, 67),),
    "cornell_groups_9spp": lambda: scenes.cornell_groups((192, 192), 2, eye=(0.21, 0.13, 5.0)),      # transformed groups: INST
    "nested_groups_root_4spp": lambda: scenes.nested_groups((160, 120), 1, transformed_root=True)[0:1] + ((160, 120),),
}
WHITTED = {
    "simplereflect_9spp": lambda: scenes.simplereflect(2, 160),
    "materials_depth8": lambda: scenes.materials((160, 120), 0, recursion=8),
    "mixed_whitted_4spp": lambda: scenes.mixed4k(mesh_n=64, nspheres=6000, res=(192, 108), supersampling=1, whitted=True),
}
FULL = {
    "C1_simple": lambda: scenes.simple("b", 2),
    "C2_mesh1m": scenes.mesh1m,
    "C3_cornell": scenes.cornell,
    "C4_spheres1m": scenes.spheres1m,
    "C5_mixed4k": scenes.mixed4k,
}


def _variant(name):
    """Corners of the configuration space the five configs do not reach (the scenes of test_gpu_parity's test_variants)."""
    if name == "orthographic_9spp":
        sc, _ = scenes.mixed4k(mesh_n=48, nspheres=3000, res=(96, 54), supersampling=2)
        cam = sc.set_orthographic_camera(700.0)
        cam.look_at([40.0, 90.0, 520.0], [0.0, 0.0, 0.0], [0.0, 1.0, 0.0]); cam.set_supersampling(2)
        return sc, (96, 54)
    if name == "spp_289":                                # more samples than a block holds: radiance buffer + k_resolve
        sc, _ = scenes.simple("b", 0, 16)
        sc.camera.set_supersampling(16)
        return sc, (20, 12)
    if name == "lights_6":
        sc, _ = scenes.spheres1m(count=4000, res=64)
        for i in range(3):
            sc.add_point_light([300.0 * (i - 1), -700.0, 900.0 - 200.0 * i], [0.2, 0.3, 0.25], [1.0, 0.0, 0.0])
        sc.camera.set_supersampling(1)
        return sc, (80, 64)
    raise KeyError(name)


def _scene(name):
    if name in PLASTIC:
        return PLASTIC[name]()
    if name in WHITTED:
        return WHITTED[name]()
    return _variant(name)


def oracle_linear(ref_li, w, h, spp):
    """The reference pixel colour: the per-sample li summed in sample order, then times 1/spp (integrate.rs:16-20), f64."""
    li = ref_li.reshape(h * w, spp, 3)
    c = np.zeros((h * w, 3))
    for s in range(spp):
        c = c + li[:, s]
    return (c * (1.0 / spp)).reshape(h, w, 3)


def outliers(dev, ref, rel):
    """Fraction of pixels whose colour differs from `ref` by more than `rel` of its magnitude (the bar of radiance_outliers)."""
    dev = np.asarray(dev, np.float64).reshape(-1, 3); ref = np.asarray(ref, np.float64).reshape(-1, 3)
    d = np.abs(dev - ref).max(axis=1)
    scale = np.maximum(np.abs(ref).max(axis=1), 1e-3)
    return float((d > rel * scale).mean())


def quantise(c):
    """img.rs:56-67 on f64 colours: clamp to [0, 1], times 255, round half away from zero."""
    x = np.clip(np.asarray(c, np.float64), 0.0, 1.0) * 255.0
    k = np.floor(x)
    return (k + (x - k >= 0.5)).astype(np.uint8)


def byte_bounds(v):
    """The least and greatest byte the quantiser gives for an f64 colour that rounds to the float32 `v`: every such colour lies
    between the midpoints of v and its two float32 neighbours (exact in f64), and the quantiser is monotonic."""
    v = np.asarray(v, np.float32)
    lo = (v.astype(np.float64) + np.nextafter(v, np.float32(-np.inf)).astype(np.float64)) / 2
    hi = (v.astype(np.float64) + np.nextafter(v, np.float32(np.inf)).astype(np.float64)) / 2
    return quantise(lo), quantise(hi)


def linear(native, ctx, sc, w, h, **kw):
    dev = native.DeviceScene(ctx, native.FlatScene(sc))
    try:
        rgb, st = dev.capture_linear(w, h, want_stats=True, **kw)
        return rgb.cpu().numpy(), st
    finally:
        dev.destroy()


@pytest.mark.parametrize("name", sorted(PLASTIC) + ["orthographic_9spp", "spp_289", "lights_6"] + sorted(WHITTED))
def test_oracle_parity(native, oracle, gpu_ctx, name):
    sc, (w, h) = _scene(name)
    spp = sc.camera.num_samples()
    ref = oracle_linear(oracle.OracleScene(sc).capture(w, h, li=True)["li"], w, h, spp)
    rgb, st = linear(native, gpu_ctx, sc, w, h)
    assert rgb.dtype == np.float32 and rgb.shape == (h, w, 3)
    assert st["primary_rays"] == w * h * spp and st["stack_overflow"] == 0
    if name in WHITTED:
        assert outliers(rgb, np.float32(ref), 1e-6) <= 2e-3
    else:
        assert outliers(rgb, np.float32(ref), 1e-9) <= 1e-4


def test_hdr_beyond_one(native, oracle, gpu_ctx):
    """Lights of intensity far above 1: the linear film keeps what the byte film clamps to 255."""
    sc, (w, h) = scenes.simple("b", 1, 128)
    sc.lights = [(p, [8.0 * c for c in i], f) for p, i, f in sc.lights]
    spp = sc.camera.num_samples()
    ref = oracle_linear(oracle.OracleScene(sc).capture(w, h, li=True)["li"], w, h, spp)
    bright = (ref > 1.0).any(axis=-1)
    assert bright.mean() >= 0.05, bright.mean()
    dev = native.DeviceScene(gpu_ctx, native.FlatScene(sc))
    try:
        rgb = dev.capture_linear(w, h).cpu().numpy()
        rgba, _ = dev.capture(w, h)
    finally:
        dev.destroy()
    assert outliers(rgb, np.float32(ref), 1e-9) <= 1e-4
    assert outliers(rgb[bright], np.float32(ref[bright]), 1e-9) <= 1e-4
    assert rgb[bright].max() > 1.0
    over = ref > 1.0
    assert (rgba[..., :3][over] == 255).all()              # the byte film saturates where the linear one goes on


@pytest.mark.parametrize("name", sorted(FULL))
def test_consistent_with_byte_film_full_size(native, gpu_ctx, name):
    """The five configs at full size (mixed4k: camera grid + light grids + the fused lean kernel at the benchmark's size): the
    byte film is the quantisation of the linear film's colour.  The float32 rounding hides which side of a byte boundary an f64
    colour within half a float32 ulp of it lay on (the background of `simple` is 0.1 = 25.5 / 255 exactly, at many pixels): there
    the byte may be either neighbour, everywhere else it must be the one byte; no pixel is left out."""
    import torch
    sc, (w, h) = FULL[name]()
    dev = native.DeviceScene(gpu_ctx, native.FlatScene(sc))
    try:
        film = torch.zeros((h, w, 4), dtype=torch.uint8, device="cuda")
        dev.capture_device(w, h, film.data_ptr(), want_stats=True)
        rgb, st = dev.capture_linear(w, h, want_stats=True)
        assert st["primary_rays"] == w * h * sc.camera.num_samples() and st["stack_overflow"] == 0
        rgba = film.cpu().numpy()
        v = rgb.cpu().numpy()
    finally:
        dev.destroy()
    assert np.isfinite(v).all()
    lo, hi = byte_bounds(v)
    b = rgba[..., :3]
    assert ((lo <= b) & (b <= hi)).all(), int((~((lo <= b) & (b <= hi))).sum())
    assert (lo == hi).mean() >= 0.999                    # one byte decided by the float alone almost everywhere


@pytest.mark.parametrize("name", ["mixed_4spp", "simple_b_9spp", "cornell_groups_9spp", "spp_289"])
def test_path_invariance(native, gpu_ctx, name):
    """Light grids, camera grid, pixel beams, bands and tile ranks change how the frame is rendered, not one bit of its linear film."""
    import torch
    sc, (w, h) = _scene(name)
    flat = native.FlatScene(sc)
    films = {}
    try:
        for grids in (0, 1):
            gpu_ctx.set_light_grids(grids)
            dev = native.DeviceScene(gpu_ctx, flat)
            try:
                for cam in (0, 1):
                    gpu_ctx.set_camera_grid(cam)
                    for beams in (0, 1):
                        gpu_ctx.set_beams(beams)
                        films[(grids, cam, beams)], _ = dev.capture_linear(w, h, want_stats=True)
                gpu_ctx.set_camera_grid(-1); gpu_ctx.set_beams(-1)
                if grids:
                    gpu_ctx.set_wave_budget_mb(1)
                    try:
                        banded, st = dev.capture_linear(w, h, want_stats=True)
                    finally:
                        gpu_ctx.set_wave_budget_mb(16384)
                    one, st1 = dev.capture_linear(w, h, want_stats=True)
                    assert st1["bands"] == 1 and (st["bands"] > 1 or name == "spp_289")      # (spp_289: one macro tile, one band)
                    assert torch.equal(banded, one)
                    ranks = 4
                    owner = torch.from_numpy(multi.tile_owner_map(w, h, ranks)).cuda()
                    acc = torch.full((h, w, 3), float("nan"), dtype=torch.float32, device="cuda")
                    for r in range(ranks):
                        dev.capture_linear(w, h, out=acc, rank=r, ranks=ranks, want_stats=True)
                        done = owner <= r
                        assert not torch.isnan(acc[done]).any() and torch.isnan(acc[~done]).all()      # the other tiles stay NaN
                    assert torch.equal(acc, one)
            finally:
                dev.destroy()
    finally:
        gpu_ctx.set_light_grids(-1); gpu_ctx.set_camera_grid(-1); gpu_ctx.set_beams(-1); gpu_ctx.set_wave_budget_mb(16384)
    first = next(iter(films.values()))
    for k, f in films.items():
        assert torch.equal(f, first), k


def test_whitted_wavefront_and_per_tree(native, gpu_ctx):
    """LGB_OPT_WHITTED 1 (levels, k_resolve) and 0 (k_secondary: another order of the f64 products) agree under the Whitted bar."""
    sc, (w, h) = WHITTED["mixed_whitted_4spp"]()
    dev = native.DeviceScene(gpu_ctx, native.FlatScene(sc))
    try:
        levels = dev.capture_linear(w, h, want_stats=True)[0].cpu().numpy()
        gpu_ctx.set_whitted(False)
        per_tree = dev.capture_linear(w, h, want_stats=True)[0].cpu().numpy()
    finally:
        gpu_ctx.set_whitted(True)
        dev.destroy()
    assert outliers(per_tree, levels, 1e-6) <= 2e-3


def test_device_group(native):
    """A 2-GPU device group in one process: the peer's tiles are stored into the leader's buffer; the film is the one-GPU film."""
    if native.lib().lgb_device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch
    sc, (w, h) = PLASTIC["mixed_4spp"]()
    one = native.Context(0)
    try:
        ref = linear(native, one, sc, w, h)[0]
    finally:
        one.close()
    group = native.Context(devices=[0, 1])
    try:
        assert group.n_devices == 2
        dev = native.DeviceScene(group, native.FlatScene(sc))
        try:
            out = torch.full((h, w, 3), float("nan"), dtype=torch.float32, device="cuda:0")
            dev.capture_linear(w, h, out=out, want_stats=True)
            assert np.array_equal(out.cpu().numpy(), ref)
        finally:
            dev.destroy()
    finally:
        group.close()


def test_stream_order(native, gpu_ctx):
    """Asynchronous renders on a side stream and on torch's default stream, read on the same stream without a host wait."""
    import torch
    sc, (w, h) = PLASTIC["mixed_4spp"]()
    dev = native.DeviceScene(gpu_ctx, native.FlatScene(sc))
    try:
        want, _ = dev.capture_linear(w, h, want_stats=True)
        want = want.cpu()
        s = torch.cuda.Stream()
        out = torch.empty((h, w, 3), dtype=torch.float32, device="cuda")
        with torch.cuda.stream(s):
            out.fill_(float("nan"))
            res = dev.capture_linear(w, h, out=out, stream=s)
            assert res is out
            got = out.to("cpu", non_blocking=False)           # queued on s behind the render
        assert torch.equal(got, want)
        for _ in range(2):                                    # the default (legacy) stream: clear, render, read, all queued
            out.fill_(float("nan"))
            dev.capture_linear(w, h, out=out)
            assert torch.equal(out.cpu(), want)
        fresh = dev.capture_linear(w, h)
        assert fresh.shape == (h, w, 3) and fresh.dtype == torch.float32 and fresh.device == torch.device("cuda", gpu_ctx.device)
        assert torch.equal(fresh.cpu(), want)
    finally:
        dev.destroy()


def test_public_api(native, gpu_ctx):
    import lasgun_b200
    sc, (w, h) = PLASTIC["cornell_4spp"]()
    rgb = lasgun_b200.capture_linear(sc, w, h, ctx=gpu_ctx)
    acc = lasgun_b200.Accel(sc, gpu_ctx)
    try:
        again = acc.capture_linear(w, h)
    finally:
        acc.close()
    assert rgb.shape == (h, w, 3) and rgb.dtype.is_floating_point
    assert np.array_equal(rgb.cpu().numpy(), again.cpu().numpy())
    assert np.array_equal(rgb.cpu().numpy(), linear(native, gpu_ctx, sc, w, h)[0])


def test_refusals(native, gpu_ctx):
    """NULL film, w == 0 and a scene of another context: LGB_ERR_INVALID, and a sentinel-filled film is left as it was."""
    import torch
    L = native.lib()
    sc, (w, h) = scenes.simple("b", 1, 64)
    dev = native.DeviceScene(gpu_ctx, native.FlatScene(sc))
    other = native.Context(0)
    odev = native.DeviceScene(other, native.FlatScene(sc))
    try:
        buf = torch.full((h, w, 3), 7.0, dtype=torch.float32, device="cuda")
        fp = C.cast(C.c_void_p(buf.data_ptr()), C.POINTER(C.c_float))
        st = native.Stats()
        assert L.lgb_capture_linear(gpu_ctx.h, dev.h, w, h, 0, 1, None, None, C.byref(st)) == native.LGB_ERR_INVALID
        assert L.lgb_capture_linear(gpu_ctx.h, dev.h, 0, h, 0, 1, fp, None, C.byref(st)) == native.LGB_ERR_INVALID
        assert L.lgb_capture_linear(gpu_ctx.h, dev.h, w, 0, 0, 1, fp, None, None) == native.LGB_ERR_INVALID
        assert L.lgb_capture_linear(gpu_ctx.h, odev.h, w, h, 0, 1, fp, None, C.byref(st)) == native.LGB_ERR_INVALID
        torch.cuda.synchronize()
        assert (buf == 7.0).all()
        for bad in (torch.zeros((h, w, 3), dtype=torch.float64, device="cuda"), torch.zeros((h, w, 4), dtype=torch.float32, device="cuda"),
                    torch.zeros((h, w, 3), dtype=torch.float32), torch.zeros((w, h, 3), dtype=torch.float32, device="cuda").transpose(0, 1)):
            with pytest.raises(ValueError):
                dev.capture_linear(w, h, out=bad)
    finally:
        odev.destroy(); dev.destroy(); other.close()
