"""Cost of the guides: on a resident scene (default: mixed4k, 3840x2160 at 16 spp), four calls alternated frame by frame in one
process after warm-up -- lgb_capture_device (RGBA8), lgb_capture_linear (f32 film), lgb_capture_guides with the film and every
guide, and lgb_capture_guides without the film (a geometry pass: primary rays and k_guides only).

Each frame is timed with CUDA events around the call on one torch stream (no stats, so nothing synchronises inside the call).
With --kernels, a separate torch.profiler pass after the timed frames adds the mean device time of every kernel of the two guides
calls.  Prints one JSON line: ms/frame per call (median, min, max, stdev over the frames) and the GPU's name and power limit;
--out FILE also writes it there.

    python scripts/guides_timing.py [--workload mixed4k] [--frames 20] [--warmup 3] [--kernels] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    import torch
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_and_max_sm_clock"] = q
    except (OSError, subprocess.SubprocessError):
        info["power_limit_and_max_sm_clock"] = "unknown"
    return info


def summary(ms):
    return {"median": statistics.median(ms), "min": min(ms), "max": max(ms), "stdev": statistics.stdev(ms) if len(ms) > 1 else 0.0, "n": len(ms)}


def kernel_times(runs, frames):
    """Mean device time per launch of every kernel each call launches (torch.profiler, CUDA activities)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    out = {}
    for k, f in runs.items():
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(frames):
                f()
            torch.cuda.synchronize()
        per = {}
        for e in prof.key_averages():
            if e.device_type.name == "CUDA" and e.count:
                t = getattr(e, "device_time_total", None)
                if t is None:
                    t = e.cuda_time_total
                per[e.key.split("(")[0][:80]] = {"ms_per_launch": t / e.count / 1000.0, "launches_per_frame": e.count / frames}
        out[k] = per
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="mixed4k")
    ap.add_argument("--frames", type=int, default=20, help="timed frames per call")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--kernels", action="store_true", help="also profile the kernels of the guides calls")
    ap.add_argument("--out")
    args = ap.parse_args()
    import torch

    from lasgun_b200 import _native as N
    from lasgun_b200 import scenes
    sc, (w, h) = scenes.CONFIGS[args.workload]()
    ctx = N.Context(0)
    dev = N.DeviceScene(ctx, N.FlatScene(sc, lazy=True))
    stream = torch.cuda.Stream()
    film = torch.empty((h, w, 4), dtype=torch.uint8, device="cuda")
    rgb = torch.empty((h, w, 3), dtype=torch.float32, device="cuda")
    g = {"rgb": torch.empty((h, w, 3), device="cuda"), "normal": torch.empty((h, w, 3), device="cuda"), "depth": torch.empty((h, w), device="cuda"),
         "prim_id": torch.empty((h, w), dtype=torch.int32, device="cuda"), "coverage": torch.empty((h, w), device="cuda")}
    geo = {k: v for k, v in g.items() if k != "rgb"}
    runs = {
        "rgba8": lambda: dev.capture_device(w, h, film.data_ptr(), stream=stream.cuda_stream),
        "linear_f32": lambda: dev.capture_linear(w, h, out=rgb, stream=stream),
        "guides_with_rgb": lambda: dev.capture_guides(w, h, out=g, stream=stream),
        "geometry_pass": lambda: dev.capture_guides(w, h, rgb=False, out=geo, stream=stream),
    }
    for _ in range(args.warmup):
        for f in runs.values():
            f()
    stream.synchronize()
    ms = {k: [] for k in runs}
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(len(runs) * args.frames)]
    i = 0
    for _ in range(args.frames):
        for k, f in runs.items():
            a, b = ev[i]; i += 1
            a.record(stream); f(); b.record(stream)
            b.synchronize()
            ms[k].append(a.elapsed_time(b))
    st = {k: dev.capture_guides(w, h, rgb=k == "guides_with_rgb", out=g if k == "guides_with_rgb" else geo, want_stats=True)[1]
          for k in ("guides_with_rgb", "geometry_pass")}
    res = {"workload": args.workload, "w": w, "h": h, "spp": sc.camera.num_samples(),
           "ms_per_frame": {k: summary(v) for k, v in ms.items()},
           "kernel_launches": {k: v["kernel_launches"] for k, v in st.items()}}
    med = {k: v["median"] for k, v in res["ms_per_frame"].items()}
    res["guides_minus_linear_median_ms"] = med["guides_with_rgb"] - med["linear_f32"]
    res["geometry_over_linear_median"] = med["geometry_pass"] / med["linear_f32"]
    if args.kernels:
        res["kernels"] = kernel_times({k: runs[k] for k in ("guides_with_rgb", "geometry_pass")}, 5)
    res.update(gpu_info())
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")
    dev.destroy()
    ctx.close()


if __name__ == "__main__":
    main()
