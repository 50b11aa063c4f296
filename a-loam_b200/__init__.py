"""aloam-b200: B200-native (sm_100a) A-LOAM per-scan registration hot path.

Python here is only a ctypes mirror of the C ABI in include/aloam_b200.h (the reference is C++; its host side is
C++ inside libaloam_b200.so).  There is no CPU fallback: importing works anywhere (so the symbol table can be
checked on a CPU box) but creating a context needs a CUDA device and fails loudly without one.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libaloam_b200.so")
_LIB = None

OK = 0
FLAG_FEW_CORRESPONDENCES, FLAG_MAP_TOO_THIN, FLAG_INITIALISED_ONLY, FLAG_CUBE_OVERFLOW = 1, 2, 4, 8
FLAG_OUTPUT_TRUNCATED = 16
MAP_SURROUND, MAP_ALL = 0, 1
BLOCK_DOUBLES = 11

EXPORTED_SYMBOLS = [
    "aloam_default_config", "aloam_create", "aloam_destroy", "aloam_strerror", "aloam_extract_features",
    "aloam_odometry_set_last", "aloam_odometry_register", "aloam_map_upload", "aloam_mapping_register",
    "aloam_voxel_filter", "aloam_scan_to_pose", "aloam_scan_to_pose_device", "aloam_reset_odometry", "aloam_knn",
    "aloam_odometry_associate", "aloam_normal_equations", "aloam_solve", "aloam_debug_features", "aloam_mapping_associate",
    "aloam_comm_unique_id", "aloam_comm_init", "aloam_comm_uses_peer_memory", "aloam_map_upload_sharded", "aloam_scan_stream", "aloam_scan_stream_batch", "aloam_scan_stream_mapped", "aloam_transform_to_end", "aloam_mapper_reset", "aloam_mapper_step", "aloam_profile_enable", "aloam_profile_read", "aloam_launch_count",
    "aloam_mapper_export", "aloam_mapper_associate_to_map", "aloam_scan_stream_mapped_registered",
]


class Config(C.Structure):
    _fields_ = [("n_scans", C.c_int), ("minimum_range", C.c_float), ("line_res", C.c_float), ("plane_res", C.c_float),
                ("outer_iters", C.c_int), ("inner_iters", C.c_int), ("huber", C.c_double), ("dist_sq_thresh", C.c_double),
                ("nearby_scan", C.c_double), ("device", C.c_int), ("max_points", C.c_int), ("max_map_points", C.c_int),
                ("max_batch", C.c_int), ("distortion", C.c_int), ("max_ring_points", C.c_int)]


class CloudView(C.Structure):
    _fields_ = [("data", C.POINTER(C.c_float)), ("n", C.c_int), ("stride_floats", C.c_int)]


class Stats(C.Structure):
    _fields_ = [("n_corner_corr", C.c_int), ("n_plane_corr", C.c_int), ("lm_iters", C.c_int), ("accepted_steps", C.c_int),
                ("flags", C.c_int), ("termination", C.c_int * 4), ("init_cost", C.c_double), ("final_cost", C.c_double),
                ("ms_total", C.c_float)]

    def as_dict(self):
        return {"n_corner_corr": self.n_corner_corr, "n_plane_corr": self.n_plane_corr, "lm_iters": self.lm_iters,
                "accepted_steps": self.accepted_steps, "flags": self.flags, "termination": list(self.termination),
                "init_cost": self.init_cost, "final_cost": self.final_cost, "ms_total": self.ms_total}


class AloamError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("aloam_b200 error %d: %s" % (code, msg))
        self.code = code


def build(force=False, verbose=False):
    from . import _build
    return _build.build(force=force, verbose=verbose)


def lib():
    """Loads libaloam_b200.so (raises if it has not been built -- there is no fallback)."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(SO_PATH):
            raise ImportError("libaloam_b200.so is missing: run `python -c 'import __graft_entry__ as g; g.build()'`")
        L = C.CDLL(SO_PATH)
        dp, fp, ip = C.POINTER(C.c_double), C.POINTER(C.c_float), C.POINTER(C.c_int)
        L.aloam_default_config.argtypes = [C.POINTER(Config), C.c_int]
        L.aloam_default_config.restype = None
        L.aloam_create.argtypes = [C.POINTER(Config), C.POINTER(C.c_void_p)]
        L.aloam_destroy.argtypes = [C.c_void_p]
        L.aloam_strerror.argtypes = [C.c_int]
        L.aloam_strerror.restype = C.c_char_p
        cv = CloudView
        L.aloam_extract_features.argtypes = [C.c_void_p, cv] + [C.POINTER(cv)] * 5
        L.aloam_odometry_set_last.argtypes = [C.c_void_p, cv, cv]
        L.aloam_odometry_register.argtypes = [C.c_void_p, cv, cv, dp, dp, C.POINTER(Stats)]
        L.aloam_map_upload.argtypes = [C.c_void_p, cv, cv]
        L.aloam_map_upload_sharded.argtypes = [C.c_void_p, cv, cv]
        L.aloam_mapping_register.argtypes = [C.c_void_p, cv, cv, dp, C.POINTER(Stats)]
        L.aloam_voxel_filter.argtypes = [C.c_void_p, cv, C.c_float, C.POINTER(cv)]
        L.aloam_mapper_reset.argtypes = [C.c_void_p]
        L.aloam_mapper_step.argtypes = [C.c_void_p, cv, cv, dp, dp, dp, dp, C.POINTER(Stats)]
        L.aloam_mapper_debug_state.argtypes = [C.c_void_p, ip, ip, ip, dp, dp, C.POINTER(C.c_longlong)]
        L.aloam_mapper_debug_cube.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(cv)]
        L.aloam_mapper_export.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_longlong, C.POINTER(C.c_longlong)]
        L.aloam_mapper_associate_to_map.argtypes = [C.c_void_p, cv, C.c_void_p]
        L.aloam_scan_stream_mapped_registered.argtypes = [C.c_void_p, C.POINTER(cv), C.c_int, C.c_int, dp, dp, C.c_void_p, C.c_longlong,
                                                          C.POINTER(C.c_longlong), C.POINTER(Stats)]
        L.aloam_scan_to_pose.argtypes = [C.c_void_p, cv, dp, dp, C.POINTER(Stats)]
        L.aloam_scan_to_pose_device.argtypes = [C.c_void_p, C.c_void_p, C.c_int, dp, dp, C.POINTER(Stats)]
        L.aloam_reset_odometry.argtypes = [C.c_void_p]
        L.aloam_scan_stream.argtypes = [C.c_void_p, C.POINTER(cv), C.c_int, C.c_int, dp, C.POINTER(Stats)]
        L.aloam_scan_stream_batch.argtypes = [C.c_void_p, C.POINTER(cv), C.c_int, C.c_int, C.c_int, dp, C.POINTER(Stats)]
        L.aloam_scan_stream_mapped.argtypes = [C.c_void_p, C.POINTER(cv), C.c_int, C.c_int, dp, dp, C.POINTER(Stats)]
        L.aloam_transform_to_end.argtypes = [C.c_void_p, cv, dp, dp, C.c_int, C.POINTER(cv)]
        L.aloam_knn.argtypes = [C.c_void_p, C.c_int, cv, C.c_int, ip, fp]
        L.aloam_odometry_associate.argtypes = [C.c_void_p, cv, cv, dp, dp, ip, ip]
        L.aloam_normal_equations.argtypes = [C.c_void_p, dp, C.c_int, dp, dp, dp, dp]
        L.aloam_solve.argtypes = [C.c_void_p, dp, C.c_int, dp, dp, dp, C.c_int, ip]
        L.aloam_debug_features.argtypes = [C.c_void_p, fp, ip, ip, ip]
        L.aloam_profile_enable.argtypes = [C.c_void_p, C.c_int]
        L.aloam_profile_read.argtypes = [C.c_void_p, dp, C.POINTER(C.c_longlong), C.POINTER(C.c_char_p), C.c_int]
        L.aloam_launch_count.argtypes = [C.c_void_p]
        L.aloam_launch_count.restype = C.c_longlong
        L.aloam_mapping_associate.argtypes = [C.c_void_p, cv, cv, dp, dp]
        L.aloam_comm_unique_id.argtypes = [C.c_char_p]
        L.aloam_comm_init.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_char_p]
        _LIB = L
    return _LIB


def _check(rc):
    if rc != 0:
        raise AloamError(rc, lib().aloam_strerror(rc).decode())


def _view(a):
    """numpy (n, 4|8) float32 -> CloudView (keeps `a` alive through the returned tuple)."""
    a = np.ascontiguousarray(a, dtype=np.float32)
    if a.ndim != 2 or a.shape[1] not in (4, 8):
        raise ValueError("clouds are (n, 4) or (n, 8) float32")
    return CloudView(a.ctypes.data_as(C.POINTER(C.c_float)), a.shape[0], a.shape[1]), a


def _out(v):
    if v.n == 0:
        return np.zeros((0, 4), np.float32)
    return np.ctypeslib.as_array(v.data, shape=(v.n, 4)).copy()


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def default_config(n_scans):
    cfg = Config()
    lib().aloam_default_config(C.byref(cfg), n_scans)
    return cfg


class Aloam:
    """One context = one caller thread = one CUDA stream on one B200 (mirrors `aloam_ctx`)."""

    def __init__(self, n_scans=64, device=0, max_points=None, **overrides):
        cfg = default_config(n_scans)
        cfg.device = device
        if max_points is not None:
            cfg.max_points = max_points
        for k, v in overrides.items():
            setattr(cfg, k, v)
        self.cfg = cfg
        self._h = C.c_void_p()
        _check(lib().aloam_create(C.byref(cfg), C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None) and self._h:
            lib().aloam_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # --- scanRegistration.cpp:129-408
    def extract_features(self, raw):
        v, keep = _view(raw)
        outs = [CloudView() for _ in range(5)]
        _check(lib().aloam_extract_features(self._h, v, *[C.byref(o) for o in outs]))
        names = ["full", "sharp", "less_sharp", "flat", "less_flat"]
        return {n: _out(o) for n, o in zip(names, outs)}

    def debug_features(self, n_full):
        curv = np.zeros(n_full, np.float32)
        label = np.zeros(n_full, np.int32)
        s = np.zeros(64, np.int32)
        e = np.zeros(64, np.int32)
        ip = C.POINTER(C.c_int)
        _check(lib().aloam_debug_features(self._h, curv.ctypes.data_as(C.POINTER(C.c_float)), label.ctypes.data_as(ip),
                                          s.ctypes.data_as(ip), e.ctypes.data_as(ip)))
        return curv, label, s[:self.cfg.n_scans], e[:self.cfg.n_scans]

    # --- laserOdometry.cpp:554-568 / :274-502
    def odometry_set_last(self, corner_last, surf_last):
        a, ka = _view(corner_last)
        b, kb = _view(surf_last)
        _check(lib().aloam_odometry_set_last(self._h, a, b))

    def odometry_register(self, sharp, flat, q, t):
        a, ka = _view(sharp)
        b, kb = _view(flat)
        q = np.array(q, np.float64)
        t = np.array(t, np.float64)
        st = Stats()
        _check(lib().aloam_odometry_register(self._h, a, b, _dp(q), _dp(t), C.byref(st)))
        return q, t, st.as_dict()

    def odometry_associate(self, sharp, flat, q, t):
        a, ka = _view(sharp)
        b, kb = _view(flat)
        cc = np.zeros((max(a.n, 1), 3), np.int32)
        pc = np.zeros((max(b.n, 1), 4), np.int32)
        ip = C.POINTER(C.c_int)
        _check(lib().aloam_odometry_associate(self._h, a, b, _dp(np.ascontiguousarray(q, np.float64)),
                                              _dp(np.ascontiguousarray(t, np.float64)), cc.ctypes.data_as(ip), pc.ctypes.data_as(ip)))
        return cc[:a.n], pc[:b.n]

    # --- laserMapping.cpp:531-559 / :554-729
    def map_upload(self, corner_map, surf_map):
        a, ka = _view(corner_map)
        b, kb = _view(surf_map)
        _check(lib().aloam_map_upload(self._h, a, b))

    def map_upload_sharded(self, corner_map, surf_map):
        """the whole submap in, this rank's shard (owned x-slabs + halo) cut out on the device and indexed"""
        a, ka = _view(corner_map)
        b, kb = _view(surf_map)
        _check(lib().aloam_map_upload_sharded(self._h, a, b))

    def map_upload_sharded_ptr(self, corner_ptr, n_corner, surf_ptr, n_surf, stride=4):
        a = CloudView(C.cast(C.c_void_p(int(corner_ptr)), C.POINTER(C.c_float)), int(n_corner), stride)
        b = CloudView(C.cast(C.c_void_p(int(surf_ptr)), C.POINTER(C.c_float)), int(n_surf), stride)
        _check(lib().aloam_map_upload_sharded(self._h, a, b))

    def map_upload_ptr(self, corner_ptr, n_corner, surf_ptr, n_surf, stride=4):
        """aloam_map_upload on raw addresses (pinned host memory or device memory; the library infers the copy kind)"""
        a = CloudView(C.cast(C.c_void_p(int(corner_ptr)), C.POINTER(C.c_float)), int(n_corner), stride)
        b = CloudView(C.cast(C.c_void_p(int(surf_ptr)), C.POINTER(C.c_float)), int(n_surf), stride)
        _check(lib().aloam_map_upload(self._h, a, b))

    # --- map cube store (laserMapping.cpp:309-550,736-801)
    def mapper_reset(self):
        _check(lib().aloam_mapper_reset(self._h))

    def mapper_step(self, corner_last, surf_last, q_wodom_curr, t_wodom_curr):
        """one alaserMapping frame -> (q_w_curr, t_w_curr, stats)"""
        a, ka = _view(corner_last)
        b, kb = _view(surf_last)
        qo = np.ascontiguousarray(q_wodom_curr, np.float64); to = np.ascontiguousarray(t_wodom_curr, np.float64)
        q = np.zeros(4); t = np.zeros(3)
        st = Stats()
        _check(lib().aloam_mapper_step(self._h, a, b, _dp(qo), _dp(to), _dp(q), _dp(t), C.byref(st)))
        return q, t, st.as_dict()

    def mapper_state(self):
        cen = (C.c_int * 3)(); nv = C.c_int(0); valid = (C.c_int * 125)(); tot = (C.c_longlong * 2)()
        q = np.zeros(4); t = np.zeros(3)
        _check(lib().aloam_mapper_debug_state(self._h, cen, C.byref(nv), valid, _dp(q), _dp(t), tot))
        return {"centre": tuple(cen), "valid": list(valid[:nv.value]), "q_wmap_wodom": q, "t_wmap_wodom": t,
                "total_corner": int(tot[0]), "total_surf": int(tot[1])}

    def mapper_cube(self, which, cube_index):
        out = CloudView()
        _check(lib().aloam_mapper_debug_cube(self._h, which, cube_index, C.byref(out)))
        return _out(out)

    # --- map outputs (laserMapping.cpp:803-848)
    def mapper_export_ptr(self, region, ptr, capacity):
        """aloam_mapper_export into caller memory at `ptr` (host or device address, room for `capacity` points); returns the
        number of points.  ptr = 0 with capacity = 0 only asks for the size."""
        n = C.c_longlong(0)
        _check(lib().aloam_mapper_export(self._h, int(region), C.c_void_p(int(ptr)) if ptr else None, int(capacity), C.byref(n)))
        return n.value

    def mapper_export(self, region):
        """/laser_cloud_surround (MAP_SURROUND) or /laser_cloud_map (MAP_ALL) as an (n, 4) float32 array"""
        n = self.mapper_export_ptr(region, 0, 0)
        out = np.zeros((n, 4), np.float32)
        if n:
            self.mapper_export_ptr(region, out.ctypes.data, n)
        return out

    def mapper_associate_to_map(self, cloud):
        """/velodyne_cloud_registered: pointAssociateToMap of `cloud` with the refined pose of the last frame -> (n, 4)"""
        v, keep = _view(cloud)
        out = np.zeros((v.n, 4), np.float32)
        _check(lib().aloam_mapper_associate_to_map(self._h, v, out.ctypes.data if v.n else None))
        return out

    def scan_stream_mapped_registered(self, ptrs, counts, device_resident, out_ptr, capacity, stride=4):
        """scan_stream_mapped, and every scan's registered full cloud written to out_ptr (device or pinned host address,
        room for `capacity` points) at offsets[k]; returns (odom poses, map poses, offsets (n + 1), stats dict)"""
        n = len(ptrs)
        views = (CloudView * n)()
        for i in range(n):
            views[i] = CloudView(C.cast(C.c_void_p(int(ptrs[i])), C.POINTER(C.c_float)), int(counts[i]), stride)
        odom = np.zeros((n, 7)); mapped = np.zeros((n, 7))
        offsets = np.zeros(n + 1, np.int64)
        st = Stats()
        _check(lib().aloam_scan_stream_mapped_registered(self._h, views, n, int(device_resident), _dp(odom), _dp(mapped),
                                                         C.c_void_p(int(out_ptr)) if out_ptr else None, int(capacity),
                                                         offsets.ctypes.data_as(C.POINTER(C.c_longlong)), C.byref(st)))
        return odom, mapped, offsets, st.as_dict()

    def mapping_register(self, corner_stack, surf_stack, x):
        a, ka = _view(corner_stack)
        b, kb = _view(surf_stack)
        x = np.array(x, np.float64)
        st = Stats()
        _check(lib().aloam_mapping_register(self._h, a, b, _dp(x), C.byref(st)))
        return x, st.as_dict()

    def mapping_associate(self, corner_stack, surf_stack, x):
        """per stack point [query, type (-1 rejected, 0 edge, 2 plane-norm), p0(3), p1(3), d, nn(5)] (corner rows first)"""
        a, ka = _view(corner_stack)
        b, kb = _view(surf_stack)
        fits = np.zeros((max(a.n + b.n, 1), 14))
        _check(lib().aloam_mapping_associate(self._h, a, b, _dp(np.ascontiguousarray(x, np.float64)), _dp(fits)))
        return fits[:a.n + b.n]

    # --- multi-GPU map sharding: rank 0 makes the id, everybody joins (ship the id with torch.distributed)
    @staticmethod
    def comm_unique_id():
        buf = C.create_string_buffer(128)
        _check(lib().aloam_comm_unique_id(buf))
        return bytes(buf.raw)

    def comm_init(self, rank, world, unique_id):
        _check(lib().aloam_comm_init(self._h, rank, world, C.create_string_buffer(bytes(unique_id), 128)))

    def comm_uses_peer_memory(self):
        lib().aloam_comm_uses_peer_memory.argtypes = [C.c_void_p]
        return bool(lib().aloam_comm_uses_peer_memory(self._h))

    def voxel_filter(self, cloud, leaf):
        a, ka = _view(cloud)
        o = CloudView()
        _check(lib().aloam_voxel_filter(self._h, a, float(leaf), C.byref(o)))
        return _out(o)

    # --- fused device-resident pipeline
    def scan_to_pose(self, raw):
        v, keep = _view(raw)
        q = np.zeros(4)
        t = np.zeros(3)
        st = Stats()
        _check(lib().aloam_scan_to_pose(self._h, v, _dp(q), _dp(t), C.byref(st)))
        return q, t, st.as_dict()

    def scan_to_pose_ptr(self, host_ptr, n, stride=4):
        """raw scan given as a host address (e.g. pinned memory owned by the caller)."""
        v = CloudView(C.cast(host_ptr, C.POINTER(C.c_float)), n, stride)
        q = np.zeros(4)
        t = np.zeros(3)
        st = Stats()
        _check(lib().aloam_scan_to_pose(self._h, v, _dp(q), _dp(t), C.byref(st)))
        return q, t, st

    def scan_to_pose_device(self, dev_ptr, n):
        q = np.zeros(4)
        t = np.zeros(3)
        st = Stats()
        _check(lib().aloam_scan_to_pose_device(self._h, C.c_void_p(dev_ptr), n, _dp(q), _dp(t), C.byref(st)))
        return q, t, st

    def scan_stream(self, ptrs, counts, device_resident, stride=4):
        """pipelined scan_to_pose over a sequence: ptrs = host (or device) addresses of the raw scans; returns (n, 7) poses"""
        n = len(ptrs)
        views = (CloudView * n)()
        for i in range(n):
            views[i] = CloudView(C.cast(C.c_void_p(int(ptrs[i])), C.POINTER(C.c_float)), int(counts[i]), stride)
        poses = np.zeros((n, 7))
        st = Stats()
        _check(lib().aloam_scan_stream(self._h, views, n, int(device_resident), _dp(poses), C.byref(st)))
        return poses, st

    def scan_stream_mapped(self, ptrs, counts, device_resident, stride=4):
        """aloam_scan_stream_mapped: odometry + scan-to-map of every scan on the device; returns (odom poses, map poses), (n, 7) each"""
        n = len(ptrs)
        views = (CloudView * n)()
        for i in range(n):
            views[i] = CloudView(C.cast(C.c_void_p(int(ptrs[i])), C.POINTER(C.c_float)), int(counts[i]), stride)
        odom = np.zeros((n, 7)); mapped = np.zeros((n, 7))
        st = Stats()
        _check(lib().aloam_scan_stream_mapped(self._h, views, n, int(device_resident), _dp(odom), _dp(mapped), C.byref(st)))
        return odom, mapped

    def scan_stream_batch(self, ptrs, counts, device_resident, stride=4):
        """aloam_scan_stream_batch: ptrs / counts are (n_scans, batch) arrays of addresses / point counts (scan-major);
        returns poses (n_scans, batch, 7).  Every kernel launch covers all `batch` trajectories of a step."""
        ptrs = np.asarray(ptrs, np.uint64)
        counts = np.asarray(counts, np.int64)
        n, b = ptrs.shape
        views = (CloudView * (n * b))()
        for k in range(n):
            for j in range(b):
                views[k * b + j] = CloudView(C.cast(C.c_void_p(int(ptrs[k, j])), C.POINTER(C.c_float)), int(counts[k, j]), stride)
        poses = np.zeros((n, b, 7))
        st = (Stats * b)()
        _check(lib().aloam_scan_stream_batch(self._h, views, n, b, int(device_resident), _dp(poses), st))
        self.last_batch_stats = [s.as_dict() for s in st]
        return poses

    def transform_to_end(self, cloud, q, t, distortion=True):
        v, keep = _view(cloud)
        o = CloudView()
        _check(lib().aloam_transform_to_end(self._h, v, _dp(np.ascontiguousarray(q, np.float64)), _dp(np.ascontiguousarray(t, np.float64)),
                                            int(distortion), C.byref(o)))
        return _out(o)

    def reset_odometry(self):
        _check(lib().aloam_reset_odometry(self._h))

    # --- measurement hooks
    def profile_enable(self, on=True):
        _check(lib().aloam_profile_enable(self._h, int(on)))

    def profile_read(self):
        """{kernel name: (total ms, launches)} measured with CUDA events on the ctx stream"""
        ms = (C.c_double * 32)()
        cnt = (C.c_longlong * 32)()
        names = (C.c_char_p * 32)()
        n = lib().aloam_profile_read(self._h, ms, cnt, names, 32)
        return {names[k].decode(): (ms[k], cnt[k]) for k in range(n) if names[k] and cnt[k] > 0}

    def launch_count(self):
        return int(lib().aloam_launch_count(self._h))

    # --- fine-grained
    def knn(self, which, queries, k):
        v, keep = _view(queries)
        idx = np.zeros((v.n, k), np.int32)
        sqd = np.zeros((v.n, k), np.float32)
        _check(lib().aloam_knn(self._h, which, v, k, idx.ctypes.data_as(C.POINTER(C.c_int)), sqd.ctypes.data_as(C.POINTER(C.c_float))))
        return idx, sqd

    def normal_equations(self, blocks, x):
        blocks = np.ascontiguousarray(blocks, np.float64).reshape(-1, BLOCK_DOUBLES)
        JtJ = np.zeros((6, 6))
        Jtr = np.zeros(6)
        cost = C.c_double(0)
        _check(lib().aloam_normal_equations(self._h, _dp(blocks), blocks.shape[0], _dp(np.ascontiguousarray(x, np.float64)),
                                            _dp(JtJ), _dp(Jtr), C.byref(cost)))
        return JtJ, Jtr, cost.value

    def solve(self, blocks, x):
        blocks = np.ascontiguousarray(blocks, np.float64).reshape(-1, BLOCK_DOUBLES)
        x = np.array(x, np.float64)
        s = np.zeros(7)
        trace = np.zeros((8, 8))
        rows = C.c_int(0)
        _check(lib().aloam_solve(self._h, _dp(blocks), blocks.shape[0], _dp(x), _dp(s), _dp(trace), 8, C.byref(rows)))
        keys = ["termination", "num_iterations", "num_successful", "num_jac_evals", "num_cost_evals", "initial_cost", "final_cost"]
        return x, dict(zip(keys, s)), trace[:rows.value]
