"""Cost of the linear film: lgb_capture_linear ((h, w, 3) float32, 12 B/pixel) against lgb_capture_device (RGBA8, 4 B/pixel) on a
resident scene (default: mixed4k, 3840x2160 at 16 spp), alternated frame by frame in one process after warm-up.

Each frame is timed with CUDA events around the call on one torch stream (no stats, so nothing synchronises inside the call).
Prints one JSON line: ms/frame per format (median, min, max, stdev over the frames), the difference of the medians and the GPU's
name and power limit; --out FILE also writes it there.

    python scripts/linear_film_timing.py [--workload mixed4k] [--frames 20] [--warmup 3] [--out FILE]
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="mixed4k")
    ap.add_argument("--frames", type=int, default=20, help="timed frames per format")
    ap.add_argument("--warmup", type=int, default=3)
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
    runs = {
        "rgba8": lambda: dev.capture_device(w, h, film.data_ptr(), stream=stream.cuda_stream),
        "linear_f32": lambda: dev.capture_linear(w, h, out=rgb, stream=stream),
    }
    for _ in range(args.warmup):
        for f in runs.values():
            f()
    stream.synchronize()
    ms = {k: [] for k in runs}
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(2 * args.frames)]
    i = 0
    for _ in range(args.frames):
        for k, f in runs.items():
            a, b = ev[i]; i += 1
            a.record(stream); f(); b.record(stream)
            b.synchronize()
            ms[k].append(a.elapsed_time(b))
    res = {"workload": args.workload, "w": w, "h": h, "spp": sc.camera.num_samples(), "film_bytes": {"rgba8": w * h * 4, "linear_f32": w * h * 12},
           "ms_per_frame": {k: summary(v) for k, v in ms.items()}}
    res["linear_minus_rgba8_median_ms"] = res["ms_per_frame"]["linear_f32"]["median"] - res["ms_per_frame"]["rgba8"]["median"]
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
