"""Cost of a new view of a resident scene: an orbit of --views cameras around the look-at point of the workload's camera, at its
distance and height, on a scene created with a view box that holds the orbit.  Per workload (default: mixed4k, 3840x2160 at 16 spp,
and spheres1m, 2048x2048 at 1 spp), host clock around work that ends in a stream synchronise:

  (a) moved:  set_camera + capture_linear of a new view (the camera grid is rebuilt inside the capture)
  (b) render: capture_linear again with the camera not moving (--frames per view)
  (c) fresh:  FlatScene + DeviceScene + capture_linear of a new view (the status quo: a new scene per view; --fresh-views of them)

One untimed orbit warms up every shape first.  (a) - (b) is the per-view cost of the camera-grid rebuild.  Prints one JSON line per
run: ms per view (median, min, max, stdev) of each, and the GPU's name and power limit; --out FILE also writes it there.

    python scripts/camera_views_timing.py [--workloads mixed4k,spheres1m] [--views 16] [--rounds 2] [--frames 3] [--fresh-views 4] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys
import time

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from guides_timing import gpu_info, summary  # noqa: E402


def orbit_cameras(cam, n):
    """n look_at cameras on the horizontal circle through cam's origin around its look-at point, same fov and supersampling."""
    from lasgun_b200 import api
    (ox, oy, oz), look, up = cam.look
    r = math.hypot(ox - look[0], oz - look[2])
    a0 = math.atan2(ox - look[0], oz - look[2])
    out = []
    for k in range(n):
        a = a0 + 2.0 * math.pi * k / n
        c = api.Camera(cam.perspective, cam.param)
        c.look_at([look[0] + r * math.sin(a), oy, look[2] + r * math.cos(a)], list(look), list(up))
        c.set_supersampling(cam.supersampling)
        out.append(c)
    return out


def run(workload, args):
    import torch
    from lasgun_b200 import _native as N
    from lasgun_b200 import scenes
    sc, (w, h) = scenes.CONFIGS[workload]()
    cams = orbit_cameras(sc.camera, args.views)
    eyes = [c.look[0] for c in cams]
    box = ([min(e[k] for e in eyes) - 1.0 for k in range(3)], [max(e[k] for e in eyes) + 1.0 for k in range(3)])
    ctx = N.Context(0)
    dev = N.DeviceScene(ctx, N.FlatScene(sc, lazy=True, view_box=box))
    stream = torch.cuda.Stream()
    rgb = torch.empty((h, w, 3), dtype=torch.float32, device="cuda")

    def frame():
        dev.capture_linear(w, h, out=rgb, stream=stream)
        stream.synchronize()

    for c in cams:                                               # warm-up: every view once, then a few frames of the last
        dev.set_camera(c); frame()
    for _ in range(args.frames):
        frame()
    moved, still = [], []
    for _ in range(args.rounds):
        for c in cams:
            t0 = time.perf_counter()
            dev.set_camera(c)
            frame()
            moved.append((time.perf_counter() - t0) * 1e3)
            for _ in range(args.frames):
                t0 = time.perf_counter()
                frame()
                still.append((time.perf_counter() - t0) * 1e3)
    dev.destroy()
    fresh = []
    for k, c in enumerate(cams[:args.fresh_views + 1]):          # (the first fresh scene is warm-up)
        sc.set_camera(c)
        t0 = time.perf_counter()
        d = N.DeviceScene(ctx, N.FlatScene(sc, lazy=True))
        d.capture_linear(w, h, out=rgb, stream=stream)
        stream.synchronize()
        t = (time.perf_counter() - t0) * 1e3
        d.destroy()
        if k:
            fresh.append(t)
    ctx.close()
    res = {"workload": workload, "w": w, "h": h, "spp": sc.camera.num_samples(), "views": args.views, "rounds": args.rounds,
           "ms_per_view": {"a_set_camera_and_capture": summary(moved), "b_capture_same_view": summary(still), "c_new_scene_and_capture": summary(fresh)}}
    m = {k: v["median"] for k, v in res["ms_per_view"].items()}
    res["a_minus_b_median_ms"] = m["a_set_camera_and_capture"] - m["b_capture_same_view"]
    res["c_over_a_median"] = m["c_new_scene_and_capture"] / m["a_set_camera_and_capture"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="mixed4k,spheres1m")
    ap.add_argument("--views", type=int, default=16)
    ap.add_argument("--rounds", type=int, default=2, help="timed orbits")
    ap.add_argument("--frames", type=int, default=3, help="frames per view with the camera not moving")
    ap.add_argument("--fresh-views", type=int, default=4, help="views rendered through a new scene each")
    ap.add_argument("--out")
    args = ap.parse_args()
    info = gpu_info()
    lines = []
    for wl in args.workloads.split(","):
        res = run(wl, args)
        res.update(info)
        lines.append(json.dumps(res))
        print(lines[-1], flush=True)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
