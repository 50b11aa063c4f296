#!/usr/bin/env python
"""bench.py -- scans/sec of the A-LOAM per-scan registration hot path on B200 (BASELINE.json metric).

Headline (`value`, `e2e`): BASELINE configs[1].  A "step" = one HDL-64-shaped synthetic scan (64x2000 firing pattern,
~128k returns, ~102k kept) through the whole scan-to-scan path: feature extraction -> 2 x (correspondence search + LM
solve) -> pose integration -> index build for the next scan.  Scans are consecutive poses of one seeded trajectory; the
odometry of scan k depends on scan k-1 exactly as in the reference (warm start + "last" clouds).
  value : K scans already resident in HBM through ONE pipelined aloam_scan_stream call
  e2e   : the same call on pinned HOST buffers (H2D of every raw scan and D2H of the poses inside the timed region)
The K-step region is timed REPEATS times on consecutive, never-seen-before stretches of the trajectory (exactly K steps
each, barrier + synchronize on both sides); the line reports the median repeat.  L2 hygiene: every step reads a raw scan
that has not been touched before and the distinct raw scans of a run exceed the 126 MB L2.

Sub-records in the same JSON line:
  mapping : BASELINE configs[2] (N = 1: 1M-point voxel map) / configs[3] (N > 1: N x 1M-point map sharded over the ranks,
            one ncclAllReduce of the normal equations per LM evaluation): per step the rank's shard is re-indexed (the
            reference rebuilds both kd-trees per frame) and the scan is registered with 2 x <= 4 LM iterations; L2 is
            flushed between steps; pose error vs the CPU oracle; roofline of the index build (K0) and the 5-NN kernel.
  batch   : BASELINE configs[4]: HDL-32 32x2200 scan stream, 16 trajectories in flight in ONE context (shared launches).
  pose_rmse_vs_oracle_{m,rad}: RMSE of the K timed world poses against the CPU oracle run on the same scans.
--impl reference : the CPU oracle (a C++ restatement of the reference's Ceres+PCL path -- the reference itself cannot be
  built in this image) run as the reference runs it: extraction and odometry as two pipelined single-threaded stages.
Multi-GPU: one process per GPU; the odometry path does not shard (replicas, weak scaling, no data-path collective), the
mapping path shards the map; every time is the max over ranks.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

SENSOR = "HDL-64"
REPEATS = 7               # timed K-step regions (median reported)
L2_BYTES = 126e6
NOMINAL_SCAN_BYTES = 16 * 127_600   # ~127.6k returns per synthetic HDL-64 scan


def frozen_config(args, K, W):
    """identical for both arms (`--impl reference` prints the same dict): a function of the command line only"""
    n_scans = 1 + W + REPEATS * K
    return {"workload": "HDL-64 synthetic 64x2000 scan-to-scan odometry (BASELINE.json configs[1]): feature extraction + "
                        "2 x (k-NN association + <=4-iter LM) + index build, consecutive scans of one trajectory",
            "sensor": SENSOR, "azimuth_steps": 2000, "beams": 64, "outer_iters": 2, "inner_iters": 4,
            "parallelism": "replicas x%d (independent scan streams, no collective); mapping sub-record: map sharded x%d" % (max(args.gpus, 1), max(args.gpus, 1)),
            "repeats": REPEATS,
            "l2": "every step reads a raw scan never touched before; %d distinct raw scans of ~%.2f MB = ~%.0f MB per run %s the 126 MB L2"
                  % (n_scans, NOMINAL_SCAN_BYTES / 1e6, n_scans * NOMINAL_SCAN_BYTES / 1e6,
                     ">" if n_scans * NOMINAL_SCAN_BYTES > L2_BYTES else "< (NOT larger than)")}


_POLLER = r"""
import sys, time
import pynvml as nv
nv.nvmlInit()
bus = sys.argv[1]
try:
    h = nv.nvmlDeviceGetHandleByPciBusId(bus.encode()) if bus != '-' else nv.nvmlDeviceGetHandleByIndex(int(sys.argv[2]))
except Exception:
    h = nv.nvmlDeviceGetHandleByIndex(int(sys.argv[2]))
mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
out = sys.stdout
while True:
    try:
        sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
        r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
    except Exception:
        sm = None
    if sm is not None:
        # raises once bench.py is gone (its end of the pipe closes), which ends the poller with it
        out.write('%.6f %d %d %d\n' % (time.time(), sm, mx, r)); out.flush()
    time.sleep(0.002)
"""


class ClockSampler:
    """SM clock and clock-event (throttle) reasons sampled WHILE the timed regions run.  The samples come from a separate
    process that polls NVML every 2 ms (a thread of this process is starved by the launch loop); it is spawned early,
    `start()` / `stop()` only mark the window.  One synchronous sample is added at each end, so the result is never empty."""
    BITS = [("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4)]

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []
        self.t0 = None
        self.edge = []
        self.nv = None
        self.h = None
        bus = "-"
        try:
            import torch
            pr = torch.cuda.get_device_properties(gpu_index)
            bus = "%08X:%02X:%02X.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        except Exception:
            pass
        try:
            self.proc = subprocess.Popen([sys.executable, "-c", _POLLER, bus, str(gpu_index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            try:
                self.h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode()) if bus != "-" else pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        except Exception:
            self.nv = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line)

    def _edge_sample(self):
        if self.nv is None:
            return
        try:
            self.edge.append((time.time(), float(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)),
                              float(self.nv.nvmlDeviceGetMaxClockInfo(self.h, self.nv.NVML_CLOCK_SM)),
                              int(self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))))
        except Exception:
            pass

    def start(self):
        self._edge_sample()
        self.t0 = time.time()

    def stop(self):
        t1 = time.time()
        self._edge_sample()
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
            self.th.join(timeout=2)
        rows = list(self.edge)
        inside = 0
        for line in self.lines:
            p = line.split()
            if len(p) == 4:
                t = float(p[0])
                if self.t0 is not None and self.t0 <= t <= t1:
                    rows.append((t, float(p[1]), float(p[2]), int(p[3]))); inside += 1
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["NVML unavailable"], "samples": 0}
        reasons = sorted({n for r in rows for n, b in self.BITS if r[3] & b})
        return {"sm_mhz": float(np.median([r[1] for r in rows])), "sm_max_mhz": max(r[2] for r in rows), "reasons": reasons,
                "samples": len(rows), "samples_inside_timed_region": inside, "source": "nvml (poller process, 2 ms)"}


def rot_angle(q1, q2):
    return 2.0 * float(np.arccos(min(1.0, abs(float(np.dot(q1, q2))))))


def cpu_odometry_sequential(orc, synth, scans, sensor=SENSOR):
    """single-threaded oracle: extract -> register -> integrate -> set_last per scan.
    Returns (seconds, extraction seconds, odometry seconds, world poses (n, 7))"""
    ns, _, mr = synth.SENSORS[sensor][:3]
    od = orc.Odometry()
    q = np.array([0, 0, 0, 1.0]); t = np.zeros(3)
    qw = np.array([0, 0, 0, 1.0]); tw = np.zeros(3)
    t_ext = t_odo = 0.0
    poses = np.zeros((len(scans), 7))
    t0 = time.perf_counter()
    for k, raw in enumerate(scans):
        a = time.perf_counter()
        f = orc.Features(raw, ns, mr, orc.SORT_LITERAL)
        b = time.perf_counter()
        if k > 0:
            q, t, _ = od.register(f.sharp, f.flat, q, t)
            qw, tw = orc.integrate_pose(qw, tw, q, t)
        od.set_last(f.less_sharp, f.less_flat)
        c = time.perf_counter()
        t_ext += b - a
        t_odo += c - b
        poses[k, :4] = qw; poses[k, 4:] = tw
    return time.perf_counter() - t0, t_ext, t_odo, poses


def cpu_pipeline_two_stage(orc, synth, scans, warmup):
    """the reference's process structure for this path: ascanRegistration | alaserOdometry, one thread each.
    Returns seconds for the scans after `warmup` (steady state, measured at the odometry stage output)."""
    import queue
    ns, _, mr = synth.SENSORS[SENSOR][:3]
    qu = queue.Queue(maxsize=4)

    def extractor():
        for raw in scans:
            qu.put(orc.Features(raw, ns, mr, orc.SORT_LITERAL))
        qu.put(None)

    th = threading.Thread(target=extractor, daemon=True)
    od = orc.Odometry()
    q = np.array([0, 0, 0, 1.0]); t = np.zeros(3)
    qw = np.array([0, 0, 0, 1.0]); tw = np.zeros(3)
    th.start()
    k = 0
    t_start = None
    while True:
        f = qu.get()
        if f is None:
            break
        if k == warmup + 1:
            t_start = time.perf_counter()
        if k > 0:
            q, t, _ = od.register(f.sharp, f.flat, q, t)
            qw, tw = orc.integrate_pose(qw, tw, q, t)
        od.set_last(f.less_sharp, f.less_flat)
        k += 1
    return time.perf_counter() - t_start


class _QuietStdout:
    """the reference's nodes print timing lines with printf / std::cout: park fd 1 on /dev/null while they run (the bench's one JSON
    line must be the only thing on stdout) and flush the C buffers before it comes back"""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        self.null = os.open(os.devnull, os.O_WRONLY)
        os.dup2(self.null, 1)
        return self

    def __exit__(self, *exc):
        import ctypes
        try:
            ctypes.CDLL(None).fflush(None)
        finally:
            os.dup2(self.saved, 1)
            os.close(self.saved); os.close(self.null)
        return False


def _ref_private(name, tag):
    """a private copy of an oracle/_ref library (the reference keeps its state in file-scope globals); None if it is not built"""
    import ctypes, shutil, tempfile
    src = os.path.join(os.path.dirname(os.path.abspath(__file__)), "oracle", "_ref", name)
    if not os.path.exists(src):
        return None
    dst = os.path.join(tempfile.mkdtemp(prefix="aloam_ref_"), name.replace(".so", "_%s.so" % tag))
    shutil.copy(src, dst)
    return ctypes.CDLL(dst)


def ref_source_pipeline_two_stage(synth, scans, warmup, tag):
    """as cpu_pipeline_two_stage, but the two stages are THE REFERENCE'S OWN scanRegistration.cpp and laserOdometry.cpp (oracle/_ref:
    compiled unmodified against the stand-in headers of oracle/ref_shim; kd-tree, VoxelGrid and the LM minimiser behind the stand-ins are
    the oracle's).  Returns (seconds for the scans after `warmup`, world poses) or None if oracle/_ref is not built."""
    import ctypes as C
    import queue
    reg, odo = _ref_private("libref_registration.so", tag), _ref_private("libref_odometry.so", tag)
    if reg is None or odo is None:
        return None
    ns, _, mr = synth.SENSORS[SENSOR][:3]
    fp = C.POINTER(C.c_float); dp = C.POINTER(C.c_double); ip = C.POINTER(C.c_int)
    reg.ref_reg_init.argtypes = [C.c_int, C.c_double]
    reg.ref_reg_process.argtypes = [fp, C.c_int, C.c_int, C.c_double]
    reg.ref_reg_cloud.argtypes = [C.c_char_p, fp, C.c_int]
    reg.ref_reg_voxel_sort_mode.argtypes = [C.c_int]
    odo.ref_odom_init.argtypes = [C.c_int]
    odo.ref_odom_process.argtypes = [fp, C.c_int, fp, C.c_int, fp, C.c_int, fp, C.c_int, fp, C.c_int, C.c_double]
    odo.ref_odom_state.argtypes = [dp, dp, dp, dp, ip]
    reg.ref_reg_init(ns, float(mr)); reg.ref_reg_voxel_sort_mode(0)
    odo.ref_odom_init(1)
    topics = [b"/laser_cloud_sharp", b"/laser_cloud_less_sharp", b"/laser_cloud_flat", b"/laser_cloud_less_flat", b"/velodyne_cloud_2"]
    qu = queue.Queue(maxsize=4)

    def extractor():
        for k, raw in enumerate(scans):
            raw = np.ascontiguousarray(raw, np.float32)
            reg.ref_reg_process(raw.ctypes.data_as(fp), raw.shape[0], raw.shape[1], 0.1 * (k + 1))
            clouds = []
            for tpc in topics:
                n = reg.ref_reg_cloud(tpc, None, 0)
                a = np.zeros((max(n, 0), 4), np.float32)
                if n > 0:
                    reg.ref_reg_cloud(tpc, a.ctypes.data_as(fp), n)
                clouds.append(a)
            qu.put((k, clouds))
        qu.put(None)

    th = threading.Thread(target=extractor, daemon=True)
    poses = np.zeros((len(scans), 7))
    th.start()
    t_start = None
    while True:
        item = qu.get()
        if item is None:
            break
        k, clouds = item
        if k == warmup + 1:
            t_start = time.perf_counter()
        args = []
        for a in clouds:
            args += [a.ctypes.data_as(fp), a.shape[0]]
        odo.ref_odom_process(*args, 0.1 * (k + 1))
        q = np.zeros(4); t = np.zeros(3); qw = np.zeros(4); tw = np.zeros(3); cnt = np.zeros(2, np.int32)
        odo.ref_odom_state(q.ctypes.data_as(dp), t.ctypes.data_as(dp), qw.ctypes.data_as(dp), tw.ctypes.data_as(dp), cnt.ctypes.data_as(ip))
        poses[k, :4] = qw; poses[k, 4:] = tw
    return time.perf_counter() - t_start, poses


def pose_rmse(got, ref):
    """translation RMSE [m] and rotation RMSE [rad] (angle 2 acos|q.q'|) over rows of (q xyzw, t)"""
    dt = np.linalg.norm(got[:, 4:] - ref[:, 4:], axis=1)
    dr = np.array([rot_angle(a[:4], b[:4]) for a, b in zip(got, ref)])
    return float(np.sqrt(np.mean(dt ** 2))), float(np.sqrt(np.mean(dr ** 2))), float(dt.max()), float(dr.max())


def peak_hbm():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def committed_traffic(kernel):
    """dram bytes per launch from the committed `ncu --set full` captures (profiles/traffic.json), or None"""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(path):
        return json.load(open(path)).get(kernel)
    return None


# ---------------------------------------------------------------------------------------------------------------------
def mapping_record(args, synth, pkg, ctx_feat, rank, world, local_rank, dist, torch, K, W):
    """BASELINE configs[2] / [3]: scan-to-map against a 1M-point-per-GPU voxel map (N > 1: sharded, real ncclAllReduce)."""
    shard = importlib.import_module("a-loam_b200.shard")
    total_pts = 1_000_000 * world
    Km = K
    Wm = 3

    def feats(raw):
        f = ctx_feat.extract_features(raw)
        return f["less_sharp"], f["less_flat"]
    cmap, smap = synth.build_map(feats, total_pts)
    my_c, my_s = shard.shard_cloud(cmap, rank, world), shard.shard_cloud(smap, rank, world)
    m_loc = len(my_c) + len(my_s)
    def make_ctx():
        cx = pkg.Aloam(n_scans=64, device=local_rank, max_points=200000, max_map_points=max(len(my_c), len(my_s)) + 1024)
        if world > 1:
            idb = torch.zeros(128, dtype=torch.uint8, device="cuda")
            if rank == 0:
                idb = torch.tensor(list(pkg.Aloam.comm_unique_id()), dtype=torch.uint8, device="cuda")
            dist.broadcast(idb, 0)
            cx.comm_init(rank, world, bytes(idb.cpu().tolist()))
        return cx
    ctx = make_ctx()
    stacks = []
    for k in synth.MAP_QUERY_SCANS[:Wm + Km]:
        f = ctx_feat.extract_features(synth.scan(SENSOR, k))
        q, t = synth.pose(k)
        x0 = np.concatenate([q, t + np.array([0.05, -0.04, 0.02])])
        stacks.append((ctx_feat.voxel_filter(f["less_sharp"], 0.4), ctx_feat.voxel_filter(f["less_flat"], 0.8), x0, k))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    dev_c, dev_s = torch.from_numpy(my_c).cuda(), torch.from_numpy(my_s).cuda()
    pin_c, pin_s = torch.from_numpy(my_c).pin_memory(), torch.from_numpy(my_s).pin_memory()
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")   # 2 x L2

    def run(host, profile=False, ctx=None):
        ctx = ctx or ctx_main
        mc, ms = (pin_c, pin_s) if host else (dev_c, dev_s)
        step_s = []
        poses = []
        launches = 0
        ctx.profile_enable(False)
        for i in range(Wm + Km):
            if i == Wm and profile:
                ctx.profile_enable(True)
            flush.fill_(i & 0xFF)          # L2 flush between steps (the shard + its index fit in L2)
            barrier()
            l0 = ctx.launch_count()
            t0 = time.perf_counter()
            ctx.map_upload_ptr(mc.data_ptr(), mc.shape[0], ms.data_ptr(), ms.shape[0])
            # past the last query scan the stacks repeat: a step re-uploads and re-indexes the map after an L2 flush either way
            cs, ss, x0, _k = stacks[i % len(stacks)]
            x, st = ctx.mapping_register(cs, ss, x0)
            t1 = time.perf_counter()
            if i >= Wm:
                step_s.append(t1 - t0); poses.append(x); launches += ctx.launch_count() - l0
        ts = torch.tensor(step_s, dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(ts, op=dist.ReduceOp.MAX)     # every step: the slowest rank
        return float(ts.sum()), poses, launches, st

    ctx_main = ctx
    secs, poses, launches, st = run(False)
    secs_host, poses_host, _, _ = run(True)
    run(False, profile=True)
    prof = ctx.profile_read()
    ctx.profile_enable(False)
    exchange = "none (1 GPU)"
    nccl_ab = None
    if world > 1:
        exchange = ("NVLink peer memory inside the LM kernel: every rank pushes its 32 partial sums into every rank's mailbox and sums in rank order; one launch per solve"
                    if ctx.comm_uses_peer_memory() else "ncclAllReduce(32 f64) between per-evaluation kernels")
        # A/B: the same steps with the NCCL exchange (1 + 4 evaluations x (kernel, ncclAllReduce, kernel) per solve)
        os.environ["ALOAM_NO_PEER"] = "1"
        ctx_b = make_ctx()
        del os.environ["ALOAM_NO_PEER"]
        secs_b, poses_b, launches_b, _ = run(False, ctx=ctx_b)
        nccl_ab = {"value": Km / secs_b, "unit": "scans/s", "ms_per_step": 1e3 * secs_b / Km, "gpu_launches": launches_b,
                   "same_poses_as_peer_path_1e-9": bool(all(np.abs(a - b).max() < 1e-9 for a, b in zip(poses, poses_b)))}
        ctx_b.close()
    rec = None
    if rank == 0:
        import pyoracle as orc
        peak, peak_src = peak_hbm()
        per_kernel = {k: {"ms_per_launch": v[0] / v[1], "launches_per_step": v[1] / Km, "ms_per_step": v[0] / Km} for k, v in prof.items()}
        nq = int(len(stacks[Wm][0]) + len(stacks[Wm][1]))
        # oracle on the WHOLE map (what the sharded ranks must reproduce together): pose parity + CPU baseline
        m = orc.Mapping()
        t0 = time.perf_counter(); m.set_map(cmap, smap); tree_s = time.perf_counter() - t0
        n_chk = min(3, Km)
        err_t = err_r = 0.0
        reg_s = 0.0
        for j in range(n_chk):
            cs, ss, x0, _k = stacks[Wm + j]
            t0 = time.perf_counter(); xr, _info = m.register(cs, ss, x0); reg_s += time.perf_counter() - t0
            err_t = max(err_t, float(np.abs(poses[j][4:] - xr[4:]).max())); err_r = max(err_r, rot_angle(poses[j][:4], xr[:4]))
        cpu_val = 1.0 / (tree_s + reg_s / n_chk)
        roofs = {}
        for name, alg in (("k_map_grid(4 launches)", 36 * m_loc), ("k_map_knn5", 16 * m_loc + 16 * nq + 8 * 5 * nq)):
            if name in per_kernel:
                launches_per_unit = 4 if "grid" in name else 1
                ms_unit = per_kernel[name]["ms_per_launch"] * launches_per_unit
                ach = alg / (ms_unit * 1e-3) / 1e9
                roofs[name] = {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "algorithmic_bytes": alg,
                               "ms": ms_unit, "traffic": committed_traffic(name.split("(")[0] + ("_%dM" % (m_loc // 1_000_000 or 1)))}
        if "k_map_knn5" in roofs:
            roofs["k_map_knn5"]["note"] = ("grid-pruned search: it touches only the 27 cells around each query, far fewer bytes than the 16 M of the "
                                           "algorithmic model (SURVEY.md 8d); `traffic` is the measured DRAM volume")
        rec = {"metric": "scans/sec", "value": Km / secs, "unit": "scans/s", "n_gpus": world, "steps": Km, "warmup": Wm, "ms_per_step": 1e3 * secs / Km,
               "scaling": "weak", "config": {"workload": "HDL-64 scan-to-map (BASELINE.json configs[%d]): %d-point synthetic voxel map (%d corner + %d surf) inside the "
                                                         "250x250x150 m submap volume, %s; per step the rank's shard (%d points) is re-indexed and the scan registered with "
                                                         "2 outer x <=4 inner LM iterations" % (2 if world == 1 else 3, total_pts, len(cmap), len(smap),
                                                         "1 GPU" if world == 1 else "x-slab shards + 1-cell halo over %d GPUs, one all-reduce of the 32 normal-equation sums per LM evaluation" % world, m_loc),
                                            "stack_points": nq, "l2": "256 MB written between steps (shard + index fit in L2 otherwise)"},
               "gpu_launches": launches, "exchange": exchange, "ncclAllReduce_path": nccl_ab,
               "e2e": {"value": Km / secs_host, "unit": "scans/s", "ms_per_step": 1e3 * secs_host / Km, "h2d_bytes_per_step": 16 * m_loc + 16 * nq, "d2h_bytes_per_step": 56 + 4 * 560,
                       "api": "aloam_map_upload + aloam_mapping_register with the shard and the stacks in host memory"},
               "roofline": roofs, "per_kernel": per_kernel,
               "cpu_baseline": {"value": cpu_val, "unit": "scans/s", "cores": 1, "kind": "port",
                                "sample": "%d scans against the whole %d-point map: two kd-tree builds %.3f s per frame (laserMapping.cpp:558-559) + "
                                          "2 x (5-NN + fits + LM) %.3f s" % (n_chk, total_pts, tree_s, reg_s / n_chk)},
               "pose_vs_oracle_max": {"m": err_t, "rad": err_r, "scans": n_chk, "tolerance": 1e-4},
               "host_equals_device_path": bool(all(np.array_equal(a, b) for a, b in zip(poses, poses_host))),
               "last_stats": st}
    ctx.close()
    del flush
    return rec


def mapped_record(args, synth, pkg, rank, world, local_rank, dist, torch, K, W, scans, counts, dev, host, oracle_odom):
    """the three reference nodes in one call (SURVEY.md 8 f-2): aloam_scan_stream_mapped = extraction + odometry + scan-to-map with
    the map cube store, every hand-off on the device.  One replica per GPU (the cube store is not sharded)."""
    maxn = max(counts)
    n = 1 + W + K
    ctx = pkg.Aloam(n_scans=64, device=local_rank, max_points=maxn + 1024, max_map_points=600000)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def run(base, device_resident):
        ctx.reset_odometry(); ctx.mapper_reset()
        ptrs = [base[i].data_ptr() for i in range(n)]
        o0, m0 = ctx.scan_stream_mapped(ptrs[:1 + W], counts[:1 + W], device_resident)
        barrier()
        l0 = ctx.launch_count()
        t0 = time.perf_counter()
        o1, m1 = ctx.scan_stream_mapped(ptrs[1 + W:], counts[1 + W:n], device_resident)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        barrier()
        return t1 - t0, np.concatenate([o0, o1]), np.concatenate([m0, m1]), ctx.launch_count() - l0
    secs, odom, mapped, launches = run(dev, True)
    secs_h, _, mapped_h, _ = run(host, False)
    # kernel breakdown of one synchronous frame (aloam_scan_to_pose + aloam_mapper_step), CUDA events around every launch
    ctx.reset_odometry(); ctx.mapper_reset()
    for i in range(1 + W):
        q, t, _ = ctx.scan_to_pose_device(dev[i].data_ptr(), counts[i])
        f = ctx.extract_features(scans[i]); ctx.mapper_step(f["less_sharp"], f["less_flat"], q, t)
    ctx.profile_enable(True)
    sync_s = 0.0
    for i in range(1 + W, 1 + W + min(K, 5)):
        q, t, _ = ctx.scan_to_pose_device(dev[i].data_ptr(), counts[i])
        f = ctx.extract_features(scans[i])
        t0 = time.perf_counter(); ctx.mapper_step(f["less_sharp"], f["less_flat"], q, t); sync_s += time.perf_counter() - t0
    prof = ctx.profile_read()
    ctx.profile_enable(False)
    st = ctx.mapper_state()
    tt = torch.tensor([secs, secs_h], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    secs, secs_h = float(tt[0]), float(tt[1])
    rec = None
    if rank == 0:
        import pyoracle as orc
        nf = min(K, 5)
        per_kernel = {k: {"ms_per_launch": v[0] / v[1], "launches_per_step": v[1] / nf, "ms_per_step": v[0] / nf} for k, v in prof.items()
                      if k in ("k_cube_store", "k_voxel", "k_map_grid(4 launches)", "k_map_knn5", "k_map_fit", "k_lm_solve")}
        # oracle mapping loop on the oracle's odometry poses over the first frames (kd-tree builds make it slow)
        n_chk = min(n, 1 + W + 4)
        cm = orc.CubeMap()
        ns, _, mr = synth.SENSORS[SENSOR][:3]
        ref = []
        t0 = time.perf_counter()
        for k in range(n_chk):
            fo = orc.Features(scans[k], ns, mr)
            pose, _ = cm.step(fo.less_sharp, fo.less_flat, oracle_odom[k, :4], oracle_odom[k, 4:], 0.4, 0.8)
            ref.append(pose)
        cpu_s = (time.perf_counter() - t0) / n_chk
        rm, rr, mm, mr_ = pose_rmse(mapped[1:n_chk], np.array(ref)[1:])
        rec = {"metric": "scans/sec", "value": K * world / secs, "unit": "scans/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": 1e3 * secs / K,
               "scaling": "weak (replicas)",
               "config": {"workload": "HDL-64 stream through all three stages: extraction + scan-to-scan odometry + scan-to-map against the growing map cube store "
                                      "(aloam_scan_stream_mapped; gather of <= 75 cubes, index build, 2 x (5-NN + fits + LM), insertion, per-cube VoxelGrid, all on the device)",
                          "map_points_after_run": int(st["total_corner"] + st["total_surf"])},
               "e2e": {"value": K * world / secs_h, "unit": "scans/s", "h2d_bytes_per_step": 16 * int(np.mean(counts)), "d2h_bytes_per_step": 112},
               "gpu_launches": launches,
               "mapper_step_sync_ms": 1e3 * sync_s / nf, "per_kernel_mapper_step": per_kernel,
               "host_equals_device_path": bool(np.array_equal(mapped, mapped_h)),
               "map_pose_rmse_vs_oracle_m": rm, "map_pose_rmse_vs_oracle_rad": rr, "map_pose_max_vs_oracle_m": mm, "scans_checked": n_chk - 1,
               "cpu_baseline": {"value": 1.0 / cpu_s, "unit": "scans/s", "cores": 1, "kind": "port",
                                "sample": "%d frames of the oracle's alaserMapping loop alone (extraction and odometry not included): kd-tree builds + 2 x (5-NN + fits + LM) "
                                          "+ insertion + per-cube VoxelGrid" % n_chk}}
    ctx.close()
    return rec


def batch_record(args, synth, pkg, rank, world, local_rank, dist, torch, K, W):
    """BASELINE configs[4]: HDL-32 32x2200, B trajectories in flight in ONE context / ONE host thread (shared launches)."""
    if not hasattr(pkg.Aloam, "scan_stream_batch"):
        return None
    B = 16
    sensor = "HDL-32"
    Kb, Wb = K, 3
    n = 1 + Wb + Kb
    # B trajectories = B differently seeded noise realisations of the trajectory (same poses, different returns)
    scans = [[synth.scan(sensor, k, seed=synth.BASE_SEED + 100 + 16 * rank + b) for k in range(n)] for b in range(B)]
    maxn = max(s.shape[0] for tr in scans for s in tr)
    host = torch.zeros((n, B, maxn, 4), dtype=torch.float32).pin_memory()
    counts = np.zeros((n, B), np.int32)
    for b in range(B):
        for k in range(n):
            s = scans[b][k]; host[k, b, :s.shape[0]] = torch.from_numpy(s); counts[k, b] = s.shape[0]
    dev = host.to("cuda")
    ctx = pkg.Aloam(n_scans=32, device=local_rank, max_points=maxn + 1024, max_batch=B, max_ring_points=2304)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def run(base):
        ctx.reset_odometry()
        ptrs = np.array([[base[k, b].data_ptr() for b in range(B)] for k in range(n)], np.uint64)
        ctx.scan_stream_batch(ptrs[:1 + Wb], counts[:1 + Wb], base is dev)
        barrier()
        l0 = ctx.launch_count()
        t0 = time.perf_counter()
        poses = ctx.scan_stream_batch(ptrs[1 + Wb:], counts[1 + Wb:], base is dev)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        barrier()
        return t1 - t0, poses, ctx.launch_count() - l0
    secs, poses, launches = run(dev)
    secs_host, poses_h, _ = run(host)
    tt = torch.tensor([secs, secs_host], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    secs, secs_host = float(tt[0]), float(tt[1])
    rec = None
    if rank == 0:
        # parity: lane 0 equals its solo run bit for bit; lane 0 vs the CPU oracle
        solo = pkg.Aloam(n_scans=32, device=local_rank, max_points=maxn + 1024, max_ring_points=2304)
        sp, _ = solo.scan_stream([dev[k, 0].data_ptr() for k in range(n)], counts[:, 0], True)
        solo.close()
        import pyoracle as orc
        _, _, _, op = cpu_odometry_sequential(orc, synth, scans[0][:1 + Wb + min(Kb, 8)], sensor)
        got = np.concatenate([np.zeros((0, 7)), poses[:min(Kb, 8), 0]])
        rm, rr, mm, mr_ = pose_rmse(got, op[1 + Wb:])
        rec = {"metric": "scans/sec", "value": B * Kb * world / secs, "unit": "scans/s", "n_gpus": world, "steps": Kb, "warmup": Wb, "batch": B,
               "ms_per_step": 1e3 * secs / Kb, "scaling": "weak",
               "config": {"workload": "HDL-32 synthetic 32x2200 scan stream (BASELINE.json configs[4]), %d trajectories in flight per GPU in one context "
                                      "(aloam_scan_stream_batch: every kernel launch covers all %d scans of a step)" % (B, B),
                          "points_per_scan_raw": int(counts.mean())},
               "e2e": {"value": B * Kb * world / secs_host, "unit": "scans/s", "h2d_bytes_per_step": int(16 * counts[1 + Wb:].sum() / Kb), "d2h_bytes_per_step": 56 * B},
               "gpu_launches": launches,
               "lane0_equals_solo_run": bool(np.array_equal(poses[:, 0], sp[1 + Wb:])),
               "host_equals_device_path": bool(np.array_equal(poses, poses_h)),
               "pose_rmse_vs_oracle_m": rm, "pose_rmse_vs_oracle_rad": rr}
    ctx.close()
    return rec


def dump_outputs(out_dir, poses, stats):
    """what the caller of the headline path receives from its last timed aloam_scan_stream call (K device-resident scans):
    poses.npy (K, 7) float64 world poses (q xyzw, t), and stats_last.npy float64 [n_corner_corr, n_plane_corr, lm_iters,
    accepted_steps, flags, termination[4], init_cost, final_cost] of its last scan (ms_total, a time, is left out)"""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "poses.npy"), np.ascontiguousarray(poses, np.float64))
    d = stats.as_dict()
    np.save(os.path.join(out_dir, "stats_last.npy"), np.array(
        [d["n_corner_corr"], d["n_plane_corr"], d["lm_iters"], d["accepted_steps"], d["flags"]] + d["termination"] + [d["init_cost"], d["final_cost"]],
        np.float64))


def emit(line):
    sys.stdout.flush()
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = os.dup(1)


def main():
    os.dup2(2, 1)   # from here on fd 1 is stderr; the JSON line is written to the saved descriptor by emit()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-mapping", action="store_true", help="skip the scan-to-map sub-record (configs[2] / [3])")
    ap.add_argument("--no-batch", action="store_true", help="skip the batched-stream sub-record (configs[4])")
    ap.add_argument("--no-mapped", action="store_true", help="skip the full three-stage stream (odometry + map cube store)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last timed aloam_scan_stream call "
                    "returned as DIR/poses.npy and DIR/stats_last.npy (the inputs are seeded: same arguments, same inputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    K, W = args.steps, max(args.warmup, 3)   # never fewer than 3 untimed warm-up steps
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    n_scans_needed = 1 + W + REPEATS * K
    config = frozen_config(args, K, W)
    synth = importlib.import_module("a-loam_b200.synth")

    if args.impl == "reference":
        if rank != 0:
            return 0
        import pyoracle as orc
        n_ref = 1 + W + K
        scans = [synth.scan(SENSOR, k, seed=synth.BASE_SEED + 1) for k in range(n_ref)]
        # weak scaling like the GPU arm: one independent scan stream (a two-thread pipeline) per GPU of the job, as far as
        # the host has cores for them
        n_rep = max(1, min(args.gpus, (os.cpu_count() or 2) // 2))
        secs_rep = [None] * n_rep
        kind = ["reference"]

        def rep(j):
            # the reference's own sources where oracle/_ref is built (this container builds it; it travels with the snapshot),
            # the oracle port otherwise
            r = None
            try:
                r = ref_source_pipeline_two_stage(synth, scans, W, "rep%d" % j)
            except Exception as e:   # noqa
                sys.stderr.write("[bench] oracle/_ref arm failed (%r): falling back to the oracle port\n" % (e,))
            if r is None:
                kind[0] = "port"
                secs_rep[j] = cpu_pipeline_two_stage(orc, synth, scans, W)
            else:
                secs_rep[j] = r[0]
        with _QuietStdout():
            ths = [threading.Thread(target=rep, args=(j,)) for j in range(n_rep)]
            for t_ in ths: t_.start()
            for t_ in ths: t_.join()
        secs = max(secs_rep)
        val = n_rep * K / secs
        line = {"impl": "reference", "metric": "scans/sec", "value": val, "unit": "scans/s", "n_gpus": args.gpus, "steps": K,
                "warmup": W, "ms_per_step": 1e3 * secs / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32/f64", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": val, "unit": "scans/s", "cores": 2 * n_rep, "kind": kind[0],
                                 "sample": ("%d independent stream(s) of %d consecutive HDL-64 scans after %d warm-up; " % (n_rep, K, W)) + (
                                     "the reference's own scanRegistration.cpp and laserOdometry.cpp (oracle/_ref: compiled unmodified, g++ -O3 "
                                     "no -march, against stand-in headers for ROS / PCL / Eigen / Ceres; kd-tree, VoxelGrid and the LM minimiser "
                                     "behind them are the oracle's restatements), one thread per node like the reference's two ROS processes"
                                     if kind[0] == "reference" else
                                     "CPU oracle (C++ restatement of the Ceres+PCL path, g++ -O3 no -march), extraction and odometry as two "
                                     "pipelined single-threaded stages like the reference's two ROS nodes")},
                "e2e": {"value": val, "unit": "scans/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        emit(line)
        return 0

    import torch
    import torch.distributed as dist
    pkg = importlib.import_module("a-loam_b200")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback for the product path)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    sampler = ClockSampler(local_rank)   # spawns the NVML poller now; the window is marked around the timed regions
    scans = [synth.scan(SENSOR, k, seed=synth.BASE_SEED + 1 + rank) for k in range(n_scans_needed)]
    counts = [s.shape[0] for s in scans]
    maxn = max(counts)
    host = torch.zeros((n_scans_needed, maxn, 4), dtype=torch.float32).pin_memory()
    for i, s in enumerate(scans):
        host[i, :s.shape[0]] = torch.from_numpy(s)
    dev = host.to("cuda", non_blocking=False)
    torch.cuda.synchronize()
    ctx = pkg.Aloam(n_scans=64, device=local_rank, max_points=maxn + 1024)
    distinct_bytes = 16 * int(sum(counts))

    def run_stream(mode):
        """warm-up call (1 + W scans), then REPEATS timed calls of exactly K scans each on fresh stretches of the trajectory"""
        ctx.reset_odometry()
        ctx.profile_enable(False)
        base = dev if mode == "device" else host
        ptrs = [base[i].data_ptr() for i in range(n_scans_needed)]
        poses_all = [ctx.scan_stream(ptrs[:1 + W], counts[:1 + W], mode == "device")[0]]
        secs, devms, launches = [], [], 0
        for r in range(REPEATS):
            a, b = 1 + W + r * K, 1 + W + (r + 1) * K
            barrier()
            l0 = ctx.launch_count()
            t0 = time.perf_counter()
            poses, st = ctx.scan_stream(ptrs[a:b], counts[a:b], mode == "device")
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            barrier()
            secs.append(t1 - t0); devms.append(st.ms_total); launches = ctx.launch_count() - l0
            poses_all.append(poses)
        return secs, devms, launches, np.concatenate(poses_all), st

    def run_sync(mode, profile=False):
        """one synchronous aloam_scan_to_pose(_device) call per scan (latency mode); profiling covers the timed steps only"""
        ctx.reset_odometry()
        ctx.profile_enable(False)

        def step(i):
            if mode == "device":
                return ctx.scan_to_pose_device(dev[i].data_ptr(), counts[i])
            return ctx.scan_to_pose_ptr(host[i].data_ptr(), counts[i])
        for i in range(1 + W):
            step(i)
        barrier()
        if profile:
            ctx.profile_enable(True)
        dev_ms = 0.0
        t0 = time.perf_counter()
        for i in range(1 + W, 1 + W + K):
            q, t, st = step(i)
            dev_ms += st.ms_total
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        barrier()
        return t1 - t0, dev_ms, np.concatenate([q, t])

    sampler.start()
    secs_dev, devms_dev, launches, poses_dev, stats_dev = run_stream("device")
    secs_e2e, _, _, poses_e2e, _ = run_stream("host")
    sync_dev, devms_sync, pose_sync = run_sync("device")
    sync_e2e, _, _ = run_sync("host")
    clocks = sampler.stop()
    run_sync("device", profile=True)
    prof = ctx.profile_read()
    ctx.profile_enable(False)

    # max over ranks of every timed region, then the median repeat
    tt = torch.tensor(secs_dev + secs_e2e + [sync_dev, sync_e2e], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        lt = torch.tensor([launches], dtype=torch.int64, device="cuda")
        dist.all_reduce(lt, op=dist.ReduceOp.SUM)
        launches = int(lt[0])
    tt = tt.cpu().numpy()
    rep_dev, rep_e2e = tt[:REPEATS], tt[REPEATS:2 * REPEATS]
    sync_dev, sync_e2e = float(tt[-2]), float(tt[-1])
    med_dev, med_e2e = float(np.median(rep_dev)), float(np.median(rep_e2e))

    mapping = None if args.no_mapping else mapping_record(args, synth, pkg, ctx, rank, world, local_rank, dist, torch, K, W)
    batch = None if args.no_batch else batch_record(args, synth, pkg, rank, world, local_rank, dist, torch, K, W)
    # pose RMSE of the K timed scans of the first repeat against the CPU oracle on the same scans (BASELINE.json metric)
    n_chk = 1 + W + K
    oposes = None
    if rank == 0:
        import pyoracle as orc
        tot_cpu, t_ext, t_odo, oposes = cpu_odometry_sequential(orc, synth, scans[:n_chk])
    mapped = None
    if not args.no_mapped:
        if world > 1:   # every rank feeds its oracle-independent run; only rank 0 holds the oracle poses
            pass
        mapped = mapped_record(args, synth, pkg, rank, world, local_rank, dist, torch, K, W, scans, counts, dev, host, oposes)

    if rank == 0:
        feats = ctx.extract_features(scans[1 + W])
        n_raw = counts[1 + W]
        n_full = feats["full"].shape[0]
        n_q = feats["sharp"].shape[0] + feats["flat"].shape[0]
        n_m = feats["less_sharp"].shape[0] + feats["less_flat"].shape[0]
        n_out = n_q + n_m
        alg_bytes = {
            "k_classify": 16 * n_raw + n_raw,
            "k_ring_scan": 2 * 4 * 64 * ((n_raw + 1023) // 1024),
            "k_scatter": 16 * n_raw + n_raw + 16 * n_full,
            "k_ring_features": 16 * n_full + 16 * n_out + 5 * n_full,
            "k_compact": 2 * 16 * n_out,
            "k_rab_build(3 launches)": 16 * n_m + 16 * n_m + 8 * n_m,
            "k_odom_assoc": 16 * n_m + 16 * n_q + 8 * 3 * n_q + 88 * n_q,
            "k_lm_solve": 88 * (768 + 1536),
        }
        peak, peak_src = peak_hbm()
        per_kernel = {k: {"ms_per_launch": v[0] / v[1], "launches_per_step": v[1] / K, "ms_per_step": v[0] / K} for k, v in prof.items()}
        dom = max(per_kernel, key=lambda k: per_kernel[k]["ms_per_step"])
        dom_ms = per_kernel[dom]["ms_per_launch"]
        achieved = alg_bytes.get(dom, 0) / (dom_ms * 1e-3) / 1e9 if dom_ms > 0 else 0.0
        roofline = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": committed_traffic(dom), "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes.get(dom, 0),
                    "ms_per_launch": dom_ms, "per_kernel": per_kernel,
                    "note": "single ~2 MB scans are latency/occupancy bound, not HBM bound (SURVEY.md 8d): frac is expected << 1; per_kernel is "
                            "measured with CUDA events around every launch of the K timed steps of the synchronous API (launches_per_step = launches / K)"}

        tot = tot_cpu
        rm, rr, mm, mr_ = pose_rmse(poses_dev[1 + W:n_chk], oposes[1 + W:])
        rm_e, rr_e, _, _ = pose_rmse(poses_e2e[1 + W:n_chk], oposes[1 + W:])
        cpu_baseline = None
        if world == 1 and not args.no_cpu_baseline:
            cpu_baseline = {"value": (n_chk - 1) / tot, "unit": "scans/s", "cores": 1, "kind": "port",
                            "sample": "%d consecutive HDL-64 scans of the same stream, single thread; extraction %.1f ms/scan, "
                                      "odometry (kd-tree builds + 2 x (association + LM)) %.1f ms/scan" %
                                      (n_chk, 1e3 * t_ext / n_chk, 1e3 * t_odo / n_chk)}
        total_scans = K * world
        line = {"metric": "scans/sec", "value": total_scans / med_dev, "unit": "scans/s", "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": 1e3 * med_dev / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32/f64", "data": "synthetic", "config": config, "clocks": clocks,
                "timing": {"repeats": REPEATS, "statistic": "median", "ms_per_step_each_repeat": [1e3 * float(s) / K for s in rep_dev],
                           "timed_region_s_total": float(rep_dev.sum()), "device_ms_per_step": float(np.median(devms_dev)) / K},
                "workload_stats": {"points_per_scan_raw": n_raw, "points_per_scan_kept": n_full, "queries_per_scan": n_q, "targets_per_scan": n_m,
                                   "distinct_input_bytes": distinct_bytes, "inputs_larger_than_l2": bool(distinct_bytes > L2_BYTES)},
                "api": "aloam_scan_stream: K scans in one pipelined call (upload | ring binning | per-ring features | compaction + index | association + LM on five streams)",
                "sync_api": {"value": total_scans / sync_dev, "e2e": total_scans / sync_e2e, "ms_per_step": 1e3 * sync_dev / K,
                             "device_ms_per_step": devms_sync / K,
                             "note": "the live drop-in call a ROS node makes once per scan: one synchronous aloam_scan_to_pose(_device) per scan (latency mode); "
                                     "the headline value / e2e are the offline pipelined call over K scans"},
                "e2e": {"value": total_scans / med_e2e, "unit": "scans/s", "h2d_bytes_per_step": 16 * n_raw,
                        "d2h_bytes_per_step": 56 + 4 * 560 + 32, "ms_per_step": 1e3 * med_e2e / K,
                        "ms_per_step_each_repeat": [1e3 * float(s) / K for s in rep_e2e],
                        "api": "aloam_scan_stream with host pinned raw scans (H2D of every raw scan and D2H of every pose inside the timed region)"},
                "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu_baseline,
                "pose_rmse_vs_oracle_m": rm, "pose_rmse_vs_oracle_rad": rr,
                "pose_check": {"vs_oracle_max_m": mm, "vs_oracle_max_rad": mr_, "scans": K, "tolerance": 1e-4,
                               "e2e_path_rmse_vs_oracle_m": rm_e, "e2e_path_rmse_vs_oracle_rad": rr_e,
                               "device_vs_host_path_identical": bool(np.array_equal(poses_dev, poses_e2e)),
                               "t_w_stream_vs_sync_maxabs": float(np.abs(poses_dev[W + K, 4:] - pose_sync[4:]).max())},
                "mapping": mapping, "batch": batch, "mapped_stream": mapped}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, poses_dev[-K:], stats_dev)
        emit(line)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
