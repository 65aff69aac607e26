#!/usr/bin/env python
"""bench.py — Mrays/s (primary + shadow) and ms/frame of the lasgun render loop on 1/2/4/8 B200.

  python bench.py --gpus N --steps K --warmup W [--workload mixed4k] [--impl reference] [--dump-outputs DIR]

A step is one full frame of the workload (default: BASELINE.json's config 5, `mixed4k`, 3840x2160 at
16 spp — the config the 1/2/4/8-GPU metric is quoted on; it fits one GPU).  Rays are counted with the
reference's semantics: primary = w*h*spp, shadow = lights * primary hits (integrate.rs:47-50).
  value  scene, BVH, light grids and camera grid resident in HBM, frame rendered into a device film (rank 0's after the NVLink
         stores of the other ranks); CUDA events around exactly K frames, max over ranks
  e2e    `capture(scene, film)` as the reference defines it (lib.rs:55-104), with HOST buffers, every step: flatten of the host
         scene (the reference's own HLBVH build is deferred: the device asks for it only when a ray meets two primitives at
         bit-identical t), lgb_scene_create (device BVH + light grids, H2D of the scene), lgb_capture (camera grid, render, D2H of
         the film into PAGEABLE memory, as a reference-side `Film` is), lgb_scene_destroy
  roofline  per kernel, largest first, from lgb_capture_profile (CUDA events around every launch, live, in this process):
         ops = the launch's own unit counts (node / primitive tests, rays, hits, light evaluations: the library's work counters)
         x SURVEY 8d's constants of record; peak = SM count x observed SM clock x lanes x 2 (128 lanes for the f32 filter / walk
         work, 64 for the f64 hit setup and shading; a launch that does both is held to the blend of the two by its own op mix);
         no microbenchmark in any denominator.
--impl reference times the CPU oracle (C++ restatement of the reference algorithm — the Rust build
cannot be compiled here) on all host threads over a bounded sample of the same frame.
--dump-outputs DIR writes the film of the last timed step (see dump_outputs), so that two builds run with the same arguments can be
compared pixel for pixel.
"""
from __future__ import annotations

import argparse
import ctypes as C
import hashlib
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark writes nothing into the tree it runs from (which may be read-only)

import numpy as np  # noqa: E402

from lasgun_b200 import scenes  # noqa: E402

METRIC = "Mrays/s (primary+shadow)"
# Constants of record, SURVEY.md §8(d): FP32 operations (FMA = 2) and bytes fetched per unit of work.
OPS = {"node": 26, "sphere": (26, 39), "tri": (47, 68), "cuboid": 31, "camera": 30, "hit": 110, "light": 25 + 120, "ambient": 120,
       "background": 15, "film": 12}
BYTES = {"node": 32, "sphere": 16, "tri": 48, "cuboid": 32, "ref": 4, "film": 4}
OTHER_CONFIGS = ("simple", "mesh1m", "cornell", "spheres1m")
DUMP_PIXELS = 1 << 21      # --dump-outputs: 32 MiB of f32 RGBA + 16 MiB of f64 pixel indices at most


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return {"hbm_gbs": float(p["hbm_gbs"]), "sm_max_mhz": float(p.get("sm_max_mhz", 1965.0)), "source": "measured (MEASURED_PEAKS.json)"}
    except Exception:
        return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0, "source": "fallback (B200_PROFILING.md)"}


def kernel_source_hash():
    """Hash of the CUDA sources the shipped library is built from: an ncu capture is only quoted if it was taken from the same code."""
    h = hashlib.sha256()
    d = os.path.join(ROOT, "lasgun_b200", "csrc")
    for f in sorted(os.listdir(d)):
        if f.endswith((".cu", ".cuh")):
            h.update(f.encode()); h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


class ClockSampler:
    """Samples SM clock and throttle reasons during the timed region (nvidia_ml_py)."""
    HW = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.samples, self.reasons, self.stop_flag, self.max_mhz, self.thread = [], set(), False, None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        while not self.stop_flag:
            try:
                t = time.perf_counter()
                mhz = self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)
                r = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                self.samples.append((t, mhz, r))
            except Exception:
                pass
            time.sleep(0.01)

    def start(self):
        """Started BEFORE the warm-up: the thread's start-up and NVML's first queries (milliseconds, and they serialise with kernel
        launches in the driver) must not land inside a timed region that at 8 GPUs is only a dozen milliseconds long."""
        if self.nv:
            self.thread = threading.Thread(target=self._run, daemon=True)
            self.thread.start()

    def mark(self):
        return time.perf_counter()

    def stop(self, t0=None, t1=None):
        self.stop_flag = True
        if self.thread:
            self.thread.join()
        inside = [x for x in self.samples if t0 is None or t0 <= x[0] <= t1]
        note = None
        if not inside and self.samples:           # a region shorter than the sampling period: the samples on either side of it
            inside = sorted(self.samples, key=lambda x: min(abs(x[0] - t0), abs(x[0] - t1)))[:2]
            note = "timed region shorter than the 10 ms sampling period: the two nearest samples"
        reasons = set()
        for _, _, r in inside:
            for bit, name in self.HW.items():
                if r & bit:
                    reasons.add(name)
        out = {"sm_mhz": statistics.median(x[1] for x in inside) if inside else None, "sm_max_mhz": self.max_mhz,
               "reasons": sorted(reasons), "samples": len(inside)}
        if note:
            out["note"] = note
        return out


def dump_outputs(path, rgba, pixels=None):
    """The film a step delivered: DIR/film_rgba.npy (k, 4) float32 RGBA8 values and DIR/film_pixel_index.npy (k,) float64 row-major
    pixel indices y * width + x.  `pixels` are the indices the step rendered (default: all); of more than DUMP_PIXELS a fixed,
    seeded sample is kept, so that runs with the same arguments write the same pixels."""
    flat = np.asarray(rgba).reshape(-1, 4)
    idx = np.arange(len(flat)) if pixels is None else np.sort(pixels)
    if len(idx) > DUMP_PIXELS:
        idx = np.sort(np.random.default_rng(0).choice(idx, DUMP_PIXELS, replace=False))
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "film_rgba.npy"), flat[idx].astype(np.float32))
    np.save(os.path.join(path, "film_pixel_index.npy"), idx.astype(np.float64))


def workload(name, args):
    if name == "mixed4k" and args.small:
        return scenes.mixed4k(mesh_n=80, nspheres=8000, res=(480, 270), supersampling=1)
    return scenes.CONFIGS[name]()


def scene_census(sc):
    """Primitive counts of a scene description (both arms name the workload with the same keys)."""
    tri = sph = cub = 0

    def walk(ag):
        nonlocal tri, sph, cub
        for item in ag.contents:
            kind = item[0]
            if kind == "sphere":
                sph += 1
            elif kind == "spheres":
                sph += len(item[2])
            elif kind in ("cube", "box"):
                cub += 1
            elif kind == "mesh":
                ref = item[1]
                mesh = sc.meshes[ref.index] if hasattr(ref, "index") else ref
                tri += len(mesh.faces) // 3 if not hasattr(mesh.faces, "shape") else int(mesh.faces.size) // 3
            elif kind == "group":
                walk(item[1])
    walk(sc.root)
    return {"triangles": int(tri), "spheres": int(sph), "cuboids": int(cub)}


def reference_sample(osc, w, h, threads, target_s, spp, n_lights):
    """Bounded sample of the frame on the CPU oracle: capture_subset(k, n) for k < threads."""
    probe_n = max(threads, (w * h) // (threads * 64))
    t0 = time.time(); osc.capture(w, h, threads=threads, counters=True, subset=(probe_n, 0, threads)); dt = max(time.time() - t0, 1e-4)
    pixels = threads * ((w * h + probe_n - 1) // probe_n)
    rate = pixels / dt
    want_pixels = min(w * h, max(pixels, int(rate * target_s)))
    n = max(threads, (w * h * threads) // want_pixels)
    return n


def run_reference(args):
    from oracle import pyoracle as po
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sc, (w, h) = workload(args.workload, args)
    threads = po.hardware_threads()
    osc = po.OracleScene(sc)
    spp, nl = sc.camera.num_samples(), len(sc.lights)
    n = reference_sample(osc, w, h, threads, args.ref_seconds / max(1, args.steps + args.warmup), spp, nl)
    times, rays = [], 0
    for i in range(args.warmup + args.steps):
        r = osc.capture(w, h, threads=threads, counters=True, subset=(n, 0, threads))
        if i >= args.warmup:
            times.append(r["render_ms"]); rays = r["counters"]["primary"] + r["counters"]["shadow"]
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, r["rgba"], np.concatenate([np.arange(k, w * h, n) for k in range(threads)]))
    ms = sum(times) / len(times)
    value = rays / (ms * 1e-3) / 1e6
    frame_rays_est = rays * (n / threads)
    line = {
        "metric": METRIC, "value": value, "unit": "Mrays/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "impl": "reference",
        # the keys of the device arm's config, so that the two lines name the workload alike (what only a device has is null)
        "config": {"workload": args.workload, "film": [w, h], "spp": spp, "lights": nl, **scene_census(sc), "bvh_nodes": None, "device_bvh_nodes": None,
                   "parallelism": f"cpu_threads{threads}", "film_gather": None, "l2_policy": "host CPU arm: none"},
        "cpu_baseline": {"value": value, "unit": "Mrays/s", "cores": threads, "kind": "port",
                         "sample": f"capture_subset(k, n={n}) for k in 0..{threads} of the {w}x{h} frame ({rays} rays/step); "
                                   "C++ restatement of the reference algorithm, not the Rust build",
                         "bvh_build_ms": osc.build_ms, "ms_per_frame_est": ms * n / threads},
        "e2e": {"value": value, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "est_frame_rays": frame_rays_est,
    }
    print(json.dumps(line))


def traversal_ops(k):
    """FP32 ops (SURVEY §8d) of the node and primitive tests one launch executed: a node fetch tests two child boxes (26 ops each); a
    primitive test that stops at the filter counts the reject path, one that runs the exact test the hit path."""
    f, e = k["filter_tests"], k["exact_tests"]
    ops = 2 * k["node_tests"] * OPS["node"]
    ops += (f[0] - e[0]) * OPS["sphere"][0] + e[0] * OPS["sphere"][1]
    ops += f[1] * OPS["cuboid"]
    ops += (f[2] - e[2]) * OPS["tri"][0] + e[2] * OPS["tri"][1]
    byts = 2 * k["node_tests"] * BYTES["node"] + f[0] * BYTES["sphere"] + f[1] * BYTES["cuboid"] + f[2] * BYTES["tri"]
    return ops, byts


def kernel_table(timed, counted, frame, w, h, nl, sm_count, clock_mhz, traffic):
    """One row per launch of the frame: its own duration (events around it) and the SURVEY-8d ops of the units it processed."""
    fp32_peak = sm_count * clock_mhz * 1e6 * 128 * 2 / 1e9       # Gop/s, FMA = 2
    fp64_peak = sm_count * clock_mhz * 1e6 * 64 * 2 / 1e9
    hits, prim = frame["primary_hits"], frame["primary_rays"]
    rows = []
    for t, c in zip(timed, counted):
        name = t["name"]
        ops, byts = traversal_ops(c)
        ops64 = 0                                    # the part of the launch's work that is f64 reference arithmetic end to end
        units = {}
        if name.startswith(("k_primary", "k_leafp", "k_beam", "k_cprimary")):
            ops += c["primary_rays"] * OPS["camera"]; units["camera_rays"] = c["primary_rays"]
        if name.startswith("k_setup") or "+setup" in name:          # k_cprimary(+setup), k_gshadow(+setup): hit setup at the kernel's tail
            ops64 += hits * OPS["hit"]; units["hits"] = hits
        if name.startswith("k_shade"):
            # one light evaluation (setup 25 + plastic BSDF 120) per unoccluded light that can contribute, the ambient evaluation per
            # hit, the background per miss, quantise + store per pixel
            evals = frame["shadow_rays_traced"] - frame["shadow_occluded"]
            ops64 += evals * OPS["light"] + hits * OPS["ambient"] + (prim - hits) * OPS["background"] + w * h * OPS["film"]
            byts += w * h * BYTES["film"]
            units.update(light_evaluations=evals, hits=hits, pixels=w * h)
        # a launch that mixes the two (the walk in f32 filters, its setup tail in f64) is measured against the blend of the two issue
        # rates weighted by its own op mix: the time the launch would take at peak is ops32 / fp32_peak + ops64 / fp64_peak
        total = ops + ops64
        at_peak = ops / fp32_peak + ops64 / fp64_peak
        peak = total / at_peak if at_peak > 0 else fp32_peak
        ach = total / (t["ms"] * 1e-3) / 1e9 if t["ms"] > 0 else 0.0
        bound = "fp64_issue" if ops == 0 else "fp32_issue" if ops64 == 0 else "fp32+fp64_issue"
        row = {"kernel": name, "launch_ms": t["ms"], "ops_per_launch": total, "fp64_ops_per_launch": ops64, "bytes_per_launch": byts, "achieved_gops": ach,
               "bound": bound, "peak_gops": peak, "frac": ach / peak,
               "node_tests": c["node_tests"], "filter_tests": c["filter_tests"], "exact_tests": c["exact_tests"], **units}
        key = name.split("[")[0].split("(")[0]
        if traffic and key in traffic:
            row["traffic"] = traffic[key]
        rows.append(row)
    return rows, fp32_peak, fp64_peak


def ncu_traffic(workload):
    """dram read + write bytes per launch, per kernel, from the committed `ncu --set full` capture of THIS source (else None)."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            t = json.load(f)
        if t.get("source_hash") != kernel_source_hash():
            return None, "profiles/ncu_traffic.json was captured from other kernel sources (hash %s, built %s): not quoted" % (t.get("source_hash"), kernel_source_hash())
        return t.get(workload), "ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum per launch (profiles/%s)" % t.get("capture", "?")
    except Exception:
        return None, "no profiles/ncu_traffic.json"


def quick_config(N, ctx, name, args, film_cache):
    """A short measurement of one of the other BASELINE configs: kernel-only ms/frame (median of a few frames), e2e of one capture
    through the C ABI with host buffers, and the dominant kernel's roofline fraction."""
    import torch
    sc, (w, h) = scenes.CONFIGS[name]()
    spp, nl = sc.camera.num_samples(), len(sc.lights)
    host = N.HostScene(sc)
    dev = N.DeviceScene(ctx, N.FlatScene(host))
    film = torch.zeros((h, w, 4), dtype=torch.uint8, device="cuda")
    for _ in range(3):
        st = dev.capture_device(w, h, film.data_ptr(), want_stats=True)
    ms = statistics.median(dev.capture_device(w, h, film.data_ptr(), want_stats=True)["render_ms"] for _ in range(7))
    rays = st["primary_rays"] + nl * st["primary_hits"]
    timed, _ = dev.capture_profile(w, h, film.data_ptr())
    ctx.set_count_work(True)
    counted, stc = dev.capture_profile(w, h, film.data_ptr())
    ctx.set_count_work(False)
    dev.destroy()
    L = N.lib()
    host_film = np.zeros((h, w, 4), dtype=np.uint8)
    e2e = []
    for i in range(3):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        flat = N.FlatScene(host, lazy=True)
        hs = C.c_void_p()
        flat.desc.expected_film_pixels = w * h          # capture(scene, film) knows its film
        ctx.check(L.lgb_scene_create(ctx.h, C.byref(flat.desc), C.byref(hs)))
        ctx.check(L.lgb_capture(ctx.h, hs, w, h, host_film.ctypes.data_as(C.POINTER(C.c_uint8)), None))
        L.lgb_scene_destroy(hs)
        e2e.append((time.perf_counter() - t0) * 1e3)
    return {"film": [w, h], "spp": spp, "lights": nl, "rays_per_frame": rays, "kernel_ms_per_frame": ms, "value": rays / (ms * 1e-3) / 1e6,
            "e2e_ms_per_frame": statistics.median(e2e[1:]), "e2e_value": rays / (statistics.median(e2e[1:]) * 1e-3) / 1e6,
            "timed": timed, "counted": counted, "frame": stc}


def run_gpu(args):
    import torch
    import torch.distributed as dist

    from lasgun_b200 import _native as N
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torchrun --nproc-per-node N for --gpus N")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))      # (NCCL_DEBUG is left as the driver set it; its log goes to stderr)
    ctx = N.Context(local)
    if os.environ.get("LGB_SIDE") == "0":              # experiments: the shadow chains of the lights on one stream
        ctx.set_side_streams(False)
    sc, (w, h) = workload(args.workload, args)
    spp, nl = sc.camera.num_samples(), len(sc.lights)
    hscene_host = N.HostScene(sc)                      # the built `Scene` (scene construction is not part of capture)
    flat = N.FlatScene(hscene_host)
    dev = N.DeviceScene(ctx, flat)
    film = torch.zeros((h, w, 4), dtype=torch.uint8, device="cuda")
    # everything (our kernels, NCCL, the timing events) runs on ONE non-default torch stream so that
    # torch.cuda.Event brackets exactly the launches it is supposed to
    tstream = torch.cuda.Stream()
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream
    assert stream != 0

    from lasgun_b200 import multi

    # N > 1: rank 0 owns the film, the other ranks' kernels store their tiles into it over NVLink (multi.SharedFilm);
    # --gather nccl keeps per-rank films and SUM-reduces them instead
    shared = multi.SharedFilm(ctx, w, h, rank, world, N) if (world > 1 and args.gather == "p2p") else None

    def step():
        return multi.capture_distributed(dev, w, h, film, rank, world, stream, shared=shared)

    # one counted frame (not timed): ray counts of the frame, summed over ranks
    st = dev.capture_device(w, h, film.data_ptr(), rank=rank, ranks=world, stream=stream, want_stats=True)
    cnt = torch.tensor([st["primary_rays"], st["primary_hits"], st["shadow_rays_traced"], st["shadow_occluded"]], dtype=torch.int64, device="cuda")
    if world > 1:
        dist.all_reduce(cnt)
    tot = cnt.tolist()
    frame = {"primary_rays": tot[0], "primary_hits": tot[1], "shadow_rays_traced": tot[2], "shadow_occluded": tot[3]}
    rays_frame = frame["primary_rays"] + nl * frame["primary_hits"]

    sampler = ClockSampler(local); sampler.start()
    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    torch.cuda.synchronize()
    t_region0 = sampler.mark()
    ev[0].record()
    for _ in range(args.steps):
        last = step()
    ev[1].record()
    torch.cuda.synchronize()
    t_region1 = sampler.mark()
    # the whole frame is on rank 0; copied now, before the measurements below render into the same film
    last_film = last.cpu().numpy() if args.dump_outputs and rank == 0 else None
    if world > 1:
        dist.barrier()
    clocks = sampler.stop(t_region0, t_region1)
    total_ms = torch.tensor([ev[0].elapsed_time(ev[1])], device="cuda")
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    ms_per_step = float(total_ms.item()) / args.steps
    value = rays_frame / (ms_per_step * 1e-3) / 1e6

    gather_same, same_as_one_gpu = None, None
    if world > 1:
        # not timed: the film of this N-GPU frame against (a) the NCCL-gathered film of the same ranks and (b) the film ONE GPU renders
        out = multi.capture_distributed(dev, w, h, film, rank, world, stream, shared=shared)
        frame_n = out.clone() if rank == 0 else None
        if shared is not None:
            multi.capture_distributed(dev, w, h, film, rank, world, stream)
            torch.cuda.synchronize()
            if rank == 0:
                gather_same = bool(torch.equal(film, frame_n))
        if rank == 0:
            one = torch.zeros((h, w, 4), dtype=torch.uint8, device="cuda")
            dev.capture_device(w, h, one.data_ptr(), rank=0, ranks=1, stream=stream)
            torch.cuda.synchronize()
            same_as_one_gpu = bool(torch.equal(one, frame_n))
        dist.barrier()

    # per-kernel: events around every launch of this rank's share of the frame (one stream), best of a few frames; a second
    # pass with the work counters on gives every launch's unit counts
    timed = None
    for _ in range(3):
        k, stp = dev.capture_profile(w, h, film.data_ptr()) if world == 1 else (None, None)
        if k is not None and (timed is None or sum(x["ms"] for x in k) < sum(x["ms"] for x in timed)):
            timed = k
    counted = None
    if world == 1:
        ctx.set_count_work(True)
        counted, _ = dev.capture_profile(w, h, film.data_ptr())
        ctx.set_count_work(False)
    kern_ms = [dev.capture_device(w, h, film.data_ptr(), rank=rank, ranks=world, stream=stream, want_stats=True) for _ in range(max(3, args.steps))]
    kms = torch.tensor([statistics.median(s["render_ms"] for s in kern_ms)], device="cuda")
    if world > 1:
        dist.all_reduce(kms, op=dist.ReduceOp.MAX)
    kernel_ms = float(kms[0].item())
    s2 = kern_ms[-1]

    # e2e through the C ABI with host buffers (rank-local frame share; film gathered on the host side of rank 0).
    # The caller's film is PAGEABLE host memory, as the reference's Film (a Vec<[u8; 4]>) is; the pinned variant is reported beside it.
    host_film = np.zeros((h, w, 4), dtype=np.uint8)
    host_film_pinned_t = torch.zeros((h, w, 4), dtype=torch.uint8).pin_memory()
    e2e_ms, e2e_parts, e2e_pinned = [], [], []
    L = N.lib()
    flat_i = None
    for variant in ("pageable", "pinned"):
        target = host_film if variant == "pageable" else host_film_pinned_t.numpy()
        for i in range(args.e2e_steps + 1):
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            if world == 1:
                flat_i = N.FlatScene(hscene_host, lazy=True)   # Accel::from minus the reference BVH build: that runs (callback) only if a ray meets an exact-t tie
                t1 = time.perf_counter()
                hscene = C.c_void_p()
                flat_i.desc.expected_film_pixels = w * h          # capture(scene, film) knows its film
                ctx.check(L.lgb_scene_create(ctx.h, C.byref(flat_i.desc), C.byref(hscene)))
                t2 = time.perf_counter()
                ctx.check(L.lgb_capture(ctx.h, hscene, w, h, target.ctypes.data_as(C.POINTER(C.c_uint8)), None))
                L.lgb_scene_destroy(hscene)
            else:
                # SPMD: every rank holds the scene description (as every rank of a torchrun job does), flattens it and creates its own
                # device scene -- 1.5 + 3.3 ms in parallel on all ranks, no reference tree (lazy) and nothing to broadcast.  Building on
                # rank 0 and broadcasting the arena (multi.replicate_scene, for jobs where only rank 0 has the scene) needs the
                # reference tree up front and cost 8 + 11 ms here.
                flat_i = N.FlatScene(hscene_host, lazy=True)
                t1 = time.perf_counter()
                flat_i.desc.expected_film_pixels = w * h
                dev_i = N.DeviceScene(ctx, flat_i)
                t2 = time.perf_counter()
                out = multi.capture_distributed(dev_i, w, h, film, rank, world, stream, shared=shared)
                if rank == 0:
                    torch.from_numpy(target).copy_(out, non_blocking=(variant == "pinned"))
                torch.cuda.synchronize()
                dev_i.destroy()
            t3 = time.perf_counter()
            dt = torch.tensor([(t3 - t0) * 1e3], device="cuda")
            if world > 1:
                dist.all_reduce(dt, op=dist.ReduceOp.MAX)
            if i > 0:
                (e2e_ms if variant == "pageable" else e2e_pinned).append(float(dt.item()))
                if variant == "pageable":
                    e2e_parts.append(((t1 - t0) * 1e3, (t2 - t1) * 1e3, (t3 - t2) * 1e3))
    e2e = statistics.median(e2e_ms)
    # N > 1, once more as ONE process driving all N GPUs (lgb_init_devices: the reference's own shape -- one blocking capture that fans
    # out inside, lib.rs:55-104): rank 0 measures while the other ranks wait on the host (a store key, no GPU activity)
    group = None
    if world > 1 and not args.no_group:
        store = dist.distributed_c10d._get_default_store()
        if rank == 0:
            try:
                gctx = N.Context(devices=list(range(world)))
                gms, gparts, gkern = [], [], []
                for i in range(args.e2e_steps + 1):
                    t0 = time.perf_counter()
                    fl = N.FlatScene(hscene_host, lazy=True)
                    t1 = time.perf_counter()
                    hs = C.c_void_p()
                    fl.desc.expected_film_pixels = w * h          # capture(scene, film) knows its film
                    gctx.check(L.lgb_scene_create(gctx.h, C.byref(fl.desc), C.byref(hs)))
                    t2 = time.perf_counter()
                    st_g = N.Stats()
                    gctx.check(L.lgb_capture(gctx.h, hs, w, h, host_film.ctypes.data_as(C.POINTER(C.c_uint8)), C.byref(st_g)))
                    L.lgb_scene_destroy(hs)
                    t3 = time.perf_counter()
                    if i > 0:
                        gms.append((t3 - t0) * 1e3); gparts.append(((t1 - t0) * 1e3, (t2 - t1) * 1e3, (t3 - t2) * 1e3)); gkern.append(float(st_g.render_ms))
                gdev = N.DeviceScene(gctx, N.FlatScene(hscene_host, lazy=True))
                gfilm = torch.zeros((h, w, 4), dtype=torch.uint8, device="cuda:0")
                for _ in range(3):
                    gdev.capture_device(w, h, gfilm.data_ptr(), want_stats=True)
                tk = []
                for _ in range(max(3, args.steps)):
                    t0 = time.perf_counter(); gdev.capture_device(w, h, gfilm.data_ptr(), want_stats=True); tk.append((time.perf_counter() - t0) * 1e3)
                one = torch.zeros((h, w, 4), dtype=torch.uint8, device="cuda")
                dev.capture_device(w, h, one.data_ptr(), rank=0, ranks=1, stream=stream)
                torch.cuda.synchronize()
                group = {"devices": world, "e2e_ms_per_frame": statistics.median(gms), "e2e_value": rays_frame / (statistics.median(gms) * 1e-3) / 1e6,
                         "parts_ms": dict(zip(("flatten", "scene_create_replicate_grids", "capture_readback_destroy"), [statistics.median(p[i] for p in gparts) for i in range(3)])),
                         "slowest_device_render_ms": statistics.median(gkern),
                         "resident_ms_per_frame_host_clock": statistics.median(tk), "resident_value": rays_frame / (statistics.median(tk) * 1e-3) / 1e6,
                         "identical_to_one_gpu": bool(torch.equal(one.cpu(), gfilm.cpu()))}
                gdev.destroy(); gctx.close()
            except Exception as ex:          # the per-process path above is the contract; this one must not take it down
                group = {"error": repr(ex)}
            store.set("lgb_group_done", "1")
        else:
            store.wait(["lgb_group_done"])
    scene_bytes = int(dev.device_bytes)
    d_ = flat.desc                                   # what lgb_scene_create copies to the device: the caller's arrays (+ rank tables when the tree is given)
    h2d_bytes = int(d_.n_spheres * 40 + d_.n_cuboids * 56 + d_.n_triangles * (44 + (36 if d_.tri_normals else 0)))
    h2d_bytes_lazy = h2d_bytes                       # (every rank uploads its own copy at N > 1: per rank, as the key says per step of one process)

    # The e2e headline is the call a user of the reference makes: ONE host process, capture(scene, film) (lib.rs:55-104), fanning out
    # over the N GPUs inside the library (lgb_init_devices).  The one-process-per-GPU form of the same frame (every rank flattens and
    # creates its own scene, peer-stored film) is reported beside it; at N = 1 the two are the same call.
    per_process = {"value": rays_frame / (e2e * 1e-3) / 1e6, "unit": "Mrays/s", "ms_per_frame": e2e,
                   "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": w * h * 4, "film_memory": "pageable",
                   "ms_per_frame_pinned_film": statistics.median(e2e_pinned),
                   "reference_tree_built": bool(flat_i is not None and flat_i.tree_built),
                   "parts_ms": dict(zip(("flatten", "scene_create_device_bvh_grids_upload", "camera_grid_render_readback_destroy"),
                                        [statistics.median(p[i] for p in e2e_parts) for i in range(3)]))}
    if world > 1 and group and "error" not in group:
        e2e_line = {"value": group["e2e_value"], "unit": "Mrays/s", "ms_per_frame": group["e2e_ms_per_frame"],
                    "h2d_bytes_per_step": h2d_bytes_lazy, "d2h_bytes_per_step": w * h * 4, "film_memory": "pageable",
                    "path": "one host process, %d GPUs as a device group (lgb_init_devices): FlatScene(lazy) + lgb_scene_create + lgb_capture into a pageable host film" % world,
                    "reference_tree_built": False, "parts_ms": group["parts_ms"], "identical_to_one_gpu": group["identical_to_one_gpu"],
                    "slowest_device_render_ms": group["slowest_device_render_ms"],
                    "resident_ms_per_frame_host_clock": group["resident_ms_per_frame_host_clock"], "resident_value": group["resident_value"],
                    "one_process_per_gpu": per_process}
    else:
        e2e_line = dict(per_process)
        if world > 1:
            e2e_line["path"] = "one process per GPU (every rank creates its own scene, film peer-stored into rank 0)"
            e2e_line["one_process_device_group"] = group
    if rank == 0:
        peaks = load_peaks()
        sm_count = torch.cuda.get_device_properties(local).multi_processor_count
        clock = float(clocks["sm_mhz"] or peaks["sm_max_mhz"])
        line = {
            "metric": METRIC, "value": value, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": args.workload, "film": [w, h], "spp": spp, "lights": nl, "triangles": int(flat.desc.n_triangles),
                       "spheres": int(flat.desc.n_spheres), "cuboids": int(flat.desc.n_cuboids), "bvh_nodes": int(flat.desc.n_nodes),
                       "device_bvh_nodes": int(dev.node_count) if hasattr(dev, "node_count") else None, "parallelism": f"tiles{world}",
                       "film_gather": None if world == 1 else {
                           "how": "peer stores into rank 0's film (CUDA IPC over NVLink)" if shared is not None else "NCCL reduce(SUM) of disjoint tiles",
                           "identical_to_nccl_gather": gather_same, "identical_to_one_gpu": same_as_one_gpu},
                       "l2_policy": "per-frame working set (wavefront buffers %.0f MB + scene %.0f MB) exceeds the 126 MB L2" % (frame["primary_rays"] * 57 / 1e6 / world, scene_bytes / 1e6)},
            "ms_per_frame": ms_per_step, "kernel_ms_per_frame": kernel_ms, "rays_per_frame": rays_frame,
            "rays_traced_per_frame": frame["primary_rays"] + frame["shadow_rays_traced"],
            "e2e": e2e_line,
            "gpu_launches": int(s2["kernel_launches"]) * args.steps,
            "work_per_frame": frame,
            "clocks": clocks,
        }
        if world == 1 and timed and counted:
            traffic, traffic_note = ncu_traffic(args.workload)
            rows, fp32_peak, fp64_peak = kernel_table(timed, counted, frame, w, h, nl, sm_count, clock, traffic)
            rows.sort(key=lambda r: -r["launch_ms"])
            top = rows[0]
            tsum = sum(r["launch_ms"] for r in rows)
            ceil = ctx.measure()
            line["roofline"] = {
                "kernel": top["kernel"], "share_of_frame": top["launch_ms"] / tsum,
                "bound": "hbm" if False else top["bound"], "achieved": top["achieved_gops"], "peak": top["peak_gops"], "unit": "Gop/s (FMA=2)",
                "frac": top["frac"], "traffic": top.get("traffic"), "traffic_source": traffic_note,
                "launch_ms": top["launch_ms"], "ops_per_launch": top["ops_per_launch"],
                "peak_source": "%d SMs x %.0f MHz (median SM clock sampled during the timed region) x %s lanes x 2" % (
                    sm_count, clock, {"fp64_issue": "64", "fp32_issue": "128"}.get(top["bound"], "128 (f32 part) / 64 (f64 part), blended by the launch's op mix")),
                "ops_definition": "the launch's own unit counts (work counters of an untimed frame of the same kernels) x SURVEY 8d constants of record",
                "kernels": [{k: v for k, v in r.items() if k not in ("filter_tests", "exact_tests")} for r in rows],
                "frame": {"ops": sum(r["ops_per_launch"] for r in rows), "sum_of_launch_ms": tsum,
                          "frac_fp32_issue": sum(r["ops_per_launch"] for r in rows) / (tsum * 1e-3) / 1e9 / fp32_peak,
                          "frac_blended": sum(r["ops_per_launch"] / r["peak_gops"] for r in rows) / 1e9 / (tsum * 1e-3)},
                "hbm": {"compulsory_bytes": scene_bytes + w * h * 4, "peak_gbs": peaks["hbm_gbs"], "peak_source": peaks["source"],
                        "traffic_per_frame": sum(r["traffic"] for r in rows if "traffic" in r) if traffic else None},
                "microbenchmarks_not_used_as_peaks": {"fp32_ffma_glanes": ceil["fp32_ffma_glanes"], "fp64_dfma_glanes": ceil["fp64_dfma_glanes"], "l2_read_gbs": ceil["l2_read_gbs"]},
            }
        if world == 1 and not args.no_cpu_baseline:
            from oracle import pyoracle as po
            threads = po.hardware_threads()
            osc = po.OracleScene(sc)
            n = reference_sample(osc, w, h, threads, args.cpu_seconds, spp, nl)
            r = osc.capture(w, h, threads=threads, counters=True, subset=(n, 0, threads))
            rays = r["counters"]["primary"] + r["counters"]["shadow"]
            # spot-check the device film at the oracle's sampled pixels (the checker, not the product)
            idx = np.concatenate([np.arange(k, w * h, n) for k in range(threads)])
            same = (host_film.reshape(-1, 4)[idx] == r["rgba"].reshape(-1, 4)[idx]).all(axis=1).mean()
            line["cpu_baseline"] = {"value": rays / (r["render_ms"] * 1e-3) / 1e6, "unit": "Mrays/s", "cores": threads, "kind": "port",
                                    "sample": f"capture_subset(k, n={n}) for k in 0..{threads} of the {w}x{h} frame ({rays} rays, {r['render_ms']:.0f} ms); "
                                              "C++ restatement of the reference algorithm, not the Rust build",
                                    "bvh_build_ms": osc.build_ms, "device_film_identical_frac_at_sample": float(same)}
        if world == 1 and not args.no_other_configs and not args.small and args.workload == "mixed4k":
            # the other four BASELINE configs, briefly (kernel-only, e2e, dominant kernel): extra keys of the same line
            others = {}
            for name in OTHER_CONFIGS:
                try:
                    q = quick_config(N, ctx, name, args, None)
                    qw, qh = q["film"]
                    rows, _, _ = kernel_table(q.pop("timed"), q.pop("counted"), q.pop("frame"), qw, qh, q["lights"], sm_count, clock, None)
                    rows.sort(key=lambda r: -r["launch_ms"])
                    q["dominant_kernel"] = {k: rows[0][k] for k in ("kernel", "launch_ms", "ops_per_launch", "achieved_gops", "peak_gops", "bound", "frac")}
                    q["kernels_ms"] = {r["kernel"]: r["launch_ms"] for r in rows}
                    others[name] = q
                except Exception as e:      # a failing side measurement must not take the headline line down with it
                    others[name] = {"error": repr(e)}
            line["other_configs"] = others
        if last_film is not None:
            dump_outputs(args.dump_outputs, last_film)
        print(json.dumps(line))
    dev.destroy()
    if shared is not None:
        torch.cuda.synchronize(); dist.barrier()
        if rank != 0:
            shared.close()
        dist.barrier()
        if rank == 0:
            shared.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--gather", default="p2p", choices=["p2p", "nccl"], help="N>1 film gather: peer stores into rank 0's film, or NCCL reduce")
    ap.add_argument("--workload", default="mixed4k", choices=sorted(scenes.CONFIGS))
    ap.add_argument("--small", action="store_true", help="tiny variant of mixed4k (CPU smoke of the bench logic)")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--ref-seconds", type=float, default=60.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true")
    ap.add_argument("--no-group", action="store_true", help="N>1: skip the one-process device-group measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the film of the last timed step as .npy files into DIR")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
