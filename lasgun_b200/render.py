"""`capture(scene, film)` and friends (src/lib.rs:42-162) on the B200 path.

capture = replay the description into the C++ host (BVH build + flatten, Accel::from) ->
lgb_scene_create (H2D) -> lgb_capture (kernels + D2H).  No CPU fallback exists.
"""
from __future__ import annotations

from . import _native as N
from .api import Film, Scene


class Accel:
    """`Accel::from(&scene)` (lib.rs:42, bvh.rs:135): the scene's BVH, flattened and resident on the GPU."""

    def __init__(self, scene: Scene, ctx: N.Context | None = None, lazy: bool = False, view_box=None):
        """view_box=(lo, hi): the world box every camera origin set_camera will be given lies in (an orbit, a fly-through)."""
        self.scene = scene
        self.ctx = ctx or N.default_context()
        self.flat = N.FlatScene(scene, lazy=lazy, view_box=view_box)
        self.dev = N.DeviceScene(self.ctx, self.flat)

    @staticmethod
    def from_scene(scene: Scene, **kw):
        return Accel(scene, **kw)

    def set_camera(self, camera):
        """A new view of this resident scene (api.Camera): captures from now on render it, without rebuilding anything but the camera
        grid.  Its origin must lie in the box of the scene, the first camera and view_box.  Returns self."""
        self.dev.set_camera(camera)
        return self

    def set_lights(self, lights, ambient):
        """Relight this resident scene: captures from now on render with `lights` ((position, intensity, falloff) triples, as
        Scene.add_point_light takes them) and the ambient term `ambient`, without a new scene; only the light grids follow a light
        that moved.  Returns self."""
        self.dev.set_lights(lights, ambient)
        return self

    def capture_linear(self, w: int, h: int, out=None):
        """The linear film of this resident scene: a float32 CUDA tensor (h, w, 3), enqueued on torch.cuda.current_stream()."""
        return self.dev.capture_linear(w, h, out=out)

    def capture_guides(self, w: int, h: int, rgb: bool = True, **kw):
        """Per-pixel normal, depth, prim_id and coverage of this resident scene (and, with rgb, the linear film of the same frame):
        a dict of CUDA tensors, enqueued on torch.cuda.current_stream() (DeviceScene.capture_guides)."""
        return self.dev.capture_guides(w, h, rgb=rgb, **kw)

    def close(self):
        self.dev.destroy()


def capture(scene: Scene, film: Film, ctx: N.Context | None = None):
    """lib.rs:55.  Blocking; fills film.pixels() (row-major RGBA8).  Returns the device stats."""
    root = Accel(scene, ctx, lazy=True)          # the reference BVH is built only if a ray meets an exact-t tie
    try:
        _, stats = root.dev.capture(film.w, film.h, out=film.output)
    finally:
        root.close()
    return stats


def capture_linear(scene: Scene, w: int, h: int, ctx: N.Context | None = None):
    """The linear film of `capture`: the in-order sample sum times 1/spp (integrate.rs:16-20) of every pixel as float32, neither
    clamped to [0, 1] nor quantised -- a torch.float32 CUDA tensor of shape (h, w, 3), returned once the frame is complete."""
    import torch
    root = Accel(scene, ctx, lazy=True)
    try:
        rgb = root.capture_linear(w, h)
        torch.cuda.current_stream(rgb.device).synchronize()
    finally:
        root.close()
    return rgb


def capture_guides(scene: Scene, w: int, h: int, rgb: bool = True, ctx: N.Context | None = None):
    """Per-pixel geometry of the camera rays' closest hits -- shading normal summed over the samples times 1/spp, depth along the
    view axis, primitive id and coverage of every pixel -- and, with rgb, the linear film of `capture_linear` from the same frame:
    a dict of CUDA tensors, returned once the frame is complete."""
    import torch
    root = Accel(scene, ctx, lazy=True)
    try:
        out = root.capture_guides(w, h, rgb=rgb)
        torch.cuda.current_stream(next(iter(out.values())).device).synchronize()
    finally:
        root.close()
    return out


def capture_subset(k: int, n: int, root: Accel, film: Film):
    """lib.rs:110: pixels k, k+n, ... of the row-major film only."""
    return root.dev.capture_subset(k, n, film.w, film.h, film.output)


def render(scene: Scene, resolution):
    """lib.rs:46."""
    film = Film(resolution[0], resolution[1])
    capture(scene, film)
    return film
