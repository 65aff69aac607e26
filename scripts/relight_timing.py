"""Cost of relighting a resident scene (lgb_scene_set_lights).  Per workload (default: mixed4k, 3840x2160 at 16 spp, and spheres1m,
2048x2048 at 1 spp), host clock around work that ends in a stream synchronise:

  (a) intensity: set_lights with new intensities and ambient, positions unchanged, + capture_linear (only the light slot is rewritten)
  (b) moved:     set_lights with the first light moved (turned about the vertical axis) + capture_linear (the light grids are rebuilt)
  (c) repeat:    capture_linear again with nothing changed (--frames per round)
  (d) fresh:     FlatScene + DeviceScene + capture_linear of the scene created with the moved lights (the status quo; --fresh of them)

One untimed round warms up every shape first.  (b) - (c) is the per-move cost of the light-grid rebuild, (a) - (c) what an intensity
change costs.  Prints one JSON line per workload: ms (median, min, max, stdev) of each, and the GPU's name and power limit; --out FILE
also writes them there.

    python scripts/relight_timing.py [--workloads mixed4k,spheres1m] [--rounds 16] [--frames 3] [--fresh 4] [--out FILE]
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


def moved(lights, k):
    """`lights` with the first one turned by 2 (k + 1) degrees about the vertical axis through the origin."""
    (x, y, z), i, f = lights[0]
    a = math.radians(2.0 * (k + 1))
    return [([x * math.cos(a) + z * math.sin(a), y, -x * math.sin(a) + z * math.cos(a)], i, f)] + list(lights[1:])


def dimmed(lights, k):
    """`lights` with every intensity scaled by 0.9 - 0.01 (k % 8)."""
    s = 0.9 - 0.01 * (k % 8)
    return [(p, [c * s for c in i], f) for p, i, f in lights]


def run(workload, args):
    import torch
    from lasgun_b200 import _native as N
    from lasgun_b200 import scenes
    sc, (w, h) = scenes.CONFIGS[workload]()
    base, amb = list(sc.lights), list(sc.ambient)
    ctx = N.Context(0)
    dev = N.DeviceScene(ctx, N.FlatScene(sc, lazy=True))
    stream = torch.cuda.Stream()
    rgb = torch.empty((h, w, 3), dtype=torch.float32, device="cuda")

    def frame():
        dev.capture_linear(w, h, out=rgb, stream=stream)
        stream.synchronize()

    def timed(fn):
        t0 = time.perf_counter()
        fn()
        return (time.perf_counter() - t0) * 1e3

    def one_round(k, out):
        lights = moved(base, k)
        out[1].append(timed(lambda: (dev.set_lights(lights, amb), frame())))
        out[0].append(timed(lambda: (dev.set_lights(dimmed(lights, k), [c * 0.9 for c in amb]), frame())))
        for _ in range(args.frames):
            out[2].append(timed(frame))

    frame()
    one_round(args.rounds, ([], [], []))                          # warm-up
    res_abc = ([], [], [])
    for k in range(args.rounds):
        one_round(k, res_abc)
    dev.destroy()
    fresh = []
    for k in range(args.fresh + 1):                              # (the first fresh scene is warm-up)
        sc.lights = moved(base, k)
        t0 = time.perf_counter()
        d = N.DeviceScene(ctx, N.FlatScene(sc, lazy=True))
        d.capture_linear(w, h, out=rgb, stream=stream)
        stream.synchronize()
        t = (time.perf_counter() - t0) * 1e3
        d.destroy()
        if k:
            fresh.append(t)
    ctx.close()
    res = {"workload": workload, "w": w, "h": h, "spp": sc.camera.num_samples(), "lights": len(base), "rounds": args.rounds,
           "ms": {"a_intensity_and_capture": summary(res_abc[0]), "b_moved_and_capture": summary(res_abc[1]),
                  "c_repeat_capture": summary(res_abc[2]), "d_new_scene_and_capture": summary(fresh)}}
    m = {k: v["median"] for k, v in res["ms"].items()}
    res["a_minus_c_median_ms"] = m["a_intensity_and_capture"] - m["c_repeat_capture"]
    res["b_minus_c_median_ms"] = m["b_moved_and_capture"] - m["c_repeat_capture"]
    res["d_over_b_median"] = m["d_new_scene_and_capture"] / m["b_moved_and_capture"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="mixed4k,spheres1m")
    ap.add_argument("--rounds", type=int, default=16, help="timed rounds: one move, one intensity change, --frames repeats")
    ap.add_argument("--frames", type=int, default=3, help="repeat frames per round")
    ap.add_argument("--fresh", type=int, default=4, help="frames rendered through a new scene each")
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
