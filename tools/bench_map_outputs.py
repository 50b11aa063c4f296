#!/usr/bin/env python
"""Cost of the map outputs of laserMapping.cpp:803-848 on the device; prints one JSON line.

1. The three-stage stream at HDL-64 scale (device-resident raw scans) in three variants, alternated in one process:
   aloam_scan_stream_mapped (registered clouds not asked for), aloam_scan_stream_mapped_registered into a device buffer, and
   into a page-locked host buffer.  Each timed region is one call over --scans scans after a warm-up call on a reset context;
   --reps regions per variant; median, min and max of the time per scan.
2. aloam_mapper_export latency (ALOAM_MAP_SURROUND and ALOAM_MAP_ALL, into device memory and into pageable host memory)
   against the size of the store after N frames of the same stream.

    python tools/bench_map_outputs.py [--scans 64] [--warmup 8] [--reps 7] [--export-frames 8,32,64]"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_card():
    """name and power limit of GPU 0, read in the same run as the measurement"""
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
        name, power = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power}
    except Exception as e:   # the measurement stands without it; say so
        return {"name": None, "power_limit": None, "error": repr(e)}


def stats(xs):
    xs = np.asarray(xs)
    med = float(np.median(xs))
    return {"median": med, "min": float(xs.min()), "max": float(xs.max()), "spread_pct": 100.0 * float(xs.max() - xs.min()) / med}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scans", type=int, default=64)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--export-frames", default="8,32,64")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_map_outputs.py measures on a CUDA device; none is available")
    pkg = importlib.import_module("a-loam_b200")
    synth = importlib.import_module("a-loam_b200.synth")
    W, K = args.warmup, args.scans
    raws = [synth.scan("HDL-64", k) for k in range(W + K)]
    counts = [r.shape[0] for r in raws]
    dev = [torch.from_numpy(r).cuda() for r in raws]
    ptrs = [d.data_ptr() for d in dev]
    ctx = pkg.Aloam(n_scans=64, max_points=max(counts) + 1024, max_map_points=600000)
    cap = sum(counts)
    out_dev = torch.empty((cap, 4), dtype=torch.float32, device="cuda")
    out_pin = torch.empty((cap, 4), dtype=torch.float32).pin_memory()

    def call(variant, lo, hi):
        if variant == "registered_null":
            return ctx.scan_stream_mapped(ptrs[lo:hi], counts[lo:hi], True)
        buf = out_dev if variant == "registered_device" else out_pin
        o, m, off, _ = ctx.scan_stream_mapped_registered(ptrs[lo:hi], counts[lo:hi], True, buf.data_ptr(), cap)
        return o, m

    variants = ["registered_null", "registered_device", "registered_pinned_host"]
    times = {v: [] for v in variants}
    poses = {}
    for rep in range(args.reps + 1):           # rep 0 warms every variant up (module loads, lazily created buffers)
        for v in variants:
            ctx.reset_odometry(); ctx.mapper_reset()
            call(v, 0, W)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            o, m = call(v, W, W + K)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            if rep:
                times[v].append(1e3 * dt / K)
            poses[v] = np.concatenate([o, m], axis=1)
    full_points = float(np.mean([c for c in counts[W:]]))   # upper bound of the full clouds (the raw scans)
    stream = {v: {"ms_per_scan": stats(times[v]), "scans_per_s_median": 1e3 / float(np.median(times[v]))} for v in variants}
    same = all(np.array_equal(poses[v], poses["registered_null"]) for v in variants)

    exports = []
    host_frames = [int(s) for s in args.export_frames.split(",") if s]
    for n in host_frames:
        n = min(n, W + K)
        ctx.reset_odometry(); ctx.mapper_reset()
        ctx.scan_stream_mapped(ptrs[:n], counts[:n], True)
        rec = {"frames": n}
        for name, region in (("surround", pkg.MAP_SURROUND), ("all", pkg.MAP_ALL)):
            size = ctx.mapper_export_ptr(region, 0, 0)
            buf = torch.empty((max(size, 1), 4), dtype=torch.float32, device="cuda")
            host = np.empty((max(size, 1), 4), np.float32)
            for _ in range(3):
                ctx.mapper_export_ptr(region, buf.data_ptr(), size); ctx.mapper_export_ptr(region, host.ctypes.data, size)
            td, th = [], []
            for _ in range(20):
                t0 = time.perf_counter(); ctx.mapper_export_ptr(region, buf.data_ptr(), size); td.append(1e3 * (time.perf_counter() - t0))
                t0 = time.perf_counter(); ctx.mapper_export_ptr(region, host.ctypes.data, size); th.append(1e3 * (time.perf_counter() - t0))
            rec[name] = {"points": size, "ms_device_out": stats(td), "ms_pageable_host_out": stats(th)}
        exports.append(rec)
    ctx.close()
    print(json.dumps({
        "tool": "tools/bench_map_outputs.py", "gpu": gpu_card(), "torch_device": torch.cuda.get_device_name(0),
        "workload": "HDL-64 synthetic scans (a-loam_b200.synth), device-resident, aloam_scan_stream_mapped[_registered]; %d warm-up + %d timed "
                    "scans per region, %d regions per variant, variants alternated" % (W, K, args.reps),
        "stream": stream, "poses_identical_across_variants": bool(same), "mean_raw_points_per_scan": full_points,
        "export": exports}))


if __name__ == "__main__":
    main()
