"""Helpers shared by tests/test_oracle_vs_reference_source.py (CPU), tests/test_gpu_vs_reference_source.py (GPU) and
tests/golden/make_reference_golden.py.  TEST INFRASTRUCTURE.

The tests compare with tests/golden/reference_source.npz: what the libraries of oracle/_ref -- the reference's own translation
units compiled unmodified against the stand-in headers of oracle/ref_shim -- computed on the tests' inputs.  The classes below
load and drive those libraries from Python; only the golden generator uses them, so the tests run wherever the repository does.
Small results (poses, counts, Jacobians) are stored as they are; clouds and work arrays as `digest`s."""
import ctypes as C
import hashlib
import os
import shutil
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_DIR = os.path.join(ROOT, "oracle", "_ref")
GOLDEN = os.path.join(ROOT, "tests", "golden", "reference_source.npz")
NCUBE = 21 * 21 * 11
TOPICS = {"full": "/velodyne_cloud_2", "sharp": "/laser_cloud_sharp", "less_sharp": "/laser_cloud_less_sharp",
          "flat": "/laser_cloud_flat", "less_flat": "/laser_cloud_less_flat"}
CLOUDS = ("full", "sharp", "less_sharp", "flat", "less_flat")


def digest(a):
    """dtype, shape and SHA-256 of the bytes: two arrays have the same digest exactly when they are equal bit for bit, so a
    bit-exact comparison with a cloud of ~100k points needs 100 bytes of golden data instead of 1.6 MB"""
    a = np.ascontiguousarray(a)
    return "%s %s %s" % (a.dtype.str, "x".join(str(d) for d in a.shape), hashlib.sha256(a.tobytes()).hexdigest())


def cube_store_digest(cubes):
    """one digest over the non-empty cubes of a store in index order (with the per-cube sizes equal, the same digest means
    every cube is equal bit for bit)"""
    return digest(np.concatenate(cubes) if cubes else np.zeros((0, 4), np.float32))


_GOLDEN = None


def golden():
    """tests/golden/reference_source.npz as a dict: key -> array, or key -> digest string (stored together as `digests`)"""
    global _GOLDEN
    if _GOLDEN is None:
        with np.load(GOLDEN, allow_pickle=False) as z:
            _GOLDEN = {k: z[k] for k in z.files if k != "digests"}
            _GOLDEN.update((k.decode(), v.decode()) for k, v in z["digests"])
    return _GOLDEN


def assert_digest(key, a, *msg):
    assert digest(a) == golden()[key], (key,) + msg


def assert_clouds(key, f, raw=None):
    """the five clouds of oracle Features `f` are bit-identical to what the reference's laserCloudHandler published under `key`"""
    if raw is not None:
        assert_digest(key + "/raw", raw, "not the scan the golden data was recorded on")
    for name in CLOUDS:
        assert_digest("%s/%s" % (key, name), getattr(f, name))


def ref_lib(name):
    """oracle/_ref/<name>: built by `make -C oracle ref REF=<checkout of the reference>` (build() does it where the sources are)"""
    path = os.path.join(REF_DIR, name)
    if not os.path.exists(path):
        raise FileNotFoundError("oracle/_ref/%s is not built: run `make -C oracle ref REF=<checkout of the reference>`" % name)
    return C.CDLL(path)


def private_copy(name, tag):
    """a private copy of a library = private file-scope state of the reference node inside this process"""
    ref_lib(name)
    path = os.path.join(tempfile.mkdtemp(prefix="ref_"), name.replace(".so", "_%s.so" % tag))
    shutil.copy(os.path.join(REF_DIR, name), path)
    return C.CDLL(path)


class RefRegistration:
    """the reference's scanRegistration node, one process-wide instance per N_SCANS (its state is file-scope globals)"""

    def __init__(self, lib, n_scans, min_range):
        self.lib = lib
        fp = C.POINTER(C.c_float); ip = C.POINTER(C.c_int)
        lib.ref_reg_init.argtypes = [C.c_int, C.c_double]
        lib.ref_reg_process.argtypes = [fp, C.c_int, C.c_int, C.c_double]
        lib.ref_reg_cloud.argtypes = [C.c_char_p, fp, C.c_int]
        lib.ref_reg_arrays.argtypes = [fp, ip, ip, C.c_int]
        lib.ref_reg_voxel_sort_mode.argtypes = [C.c_int]
        lib.ref_reg_published.argtypes = [C.c_char_p]; lib.ref_reg_published.restype = C.c_long
        lib.ref_reg_init(n_scans, float(min_range))

    def run(self, raw, sort_mode):
        raw = np.ascontiguousarray(raw, np.float32)
        self.lib.ref_reg_voxel_sort_mode(sort_mode)
        before = self.lib.ref_reg_published(b"/laser_cloud_less_flat")
        self.lib.ref_reg_process(raw.ctypes.data_as(C.POINTER(C.c_float)), raw.shape[0], raw.shape[1], 0.0)
        assert self.lib.ref_reg_published(b"/laser_cloud_less_flat") == before + 1, "the reference's handler did not publish"
        out = {}
        for k, topic in TOPICS.items():
            n = self.lib.ref_reg_cloud(topic.encode(), None, 0)
            a = np.zeros((n, 4), np.float32)
            self.lib.ref_reg_cloud(topic.encode(), a.ctypes.data_as(C.POINTER(C.c_float)), n)
            out[k] = a
        n = out["full"].shape[0]
        out["curvature"] = np.zeros(n, np.float32); out["label"] = np.zeros(n, np.int32); out["picked"] = np.zeros(n, np.int32)
        self.lib.ref_reg_arrays(out["curvature"].ctypes.data_as(C.POINTER(C.c_float)), out["label"].ctypes.data_as(C.POINTER(C.c_int)),
                                out["picked"].ctypes.data_as(C.POINTER(C.c_int)), n)
        return out


_REG = {}


def ref_registration(n_scans, min_range):
    """one copy of the library per scan-line count: N_SCANS and the publishers are set once, in the reference's main()"""
    key = (n_scans, float(min_range))
    if key not in _REG:
        _REG[key] = RefRegistration(private_copy("libref_registration.so", "%d" % n_scans), n_scans, min_range)
    return _REG[key]


class RefOdometry:
    def __init__(self, lib):
        self.lib = lib
        fp = C.POINTER(C.c_float); dp = C.POINTER(C.c_double); ip = C.POINTER(C.c_int)
        lib.ref_odom_init.argtypes = [C.c_int]
        lib.ref_odom_process.argtypes = [fp, C.c_int, fp, C.c_int, fp, C.c_int, fp, C.c_int, fp, C.c_int, C.c_double]
        lib.ref_odom_state.argtypes = [dp, dp, dp, dp, ip]
        lib.ref_odom_published_pose.argtypes = [dp, dp]; lib.ref_odom_published_pose.restype = C.c_long
        lib.ref_odom_cloud.argtypes = [C.c_char_p, fp, C.c_int]
        lib.ref_odom_transform_to_start.argtypes = [fp, fp]
        lib.ref_odom_init(1)

    def process(self, f, stamp):
        a = [np.ascontiguousarray(x, np.float32) for x in (f.sharp, f.less_sharp, f.flat, f.less_flat, f.full)]
        args = []
        for x in a:
            args += [x.ctypes.data_as(C.POINTER(C.c_float)), x.shape[0]]
        self.lib.ref_odom_process(*args, float(stamp))
        q = np.zeros(4); t = np.zeros(3); qw = np.zeros(4); tw = np.zeros(3); cnt = np.zeros(2, np.int32)
        dp = C.POINTER(C.c_double)
        self.lib.ref_odom_state(q.ctypes.data_as(dp), t.ctypes.data_as(dp), qw.ctypes.data_as(dp), tw.ctypes.data_as(dp), cnt.ctypes.data_as(C.POINTER(C.c_int)))
        pq = np.zeros(4); pt = np.zeros(3)
        n_pub = self.lib.ref_odom_published_pose(pq.ctypes.data_as(dp), pt.ctypes.data_as(dp))
        return {"q": q, "t": t, "qw": qw, "tw": tw, "counts": cnt, "pub_q": pq, "pub_t": pt, "n_pub": n_pub}

    def cloud(self, topic):
        n = self.lib.ref_odom_cloud(topic.encode(), None, 0)
        a = np.zeros((max(n, 0), 4), np.float32)
        if n > 0:
            self.lib.ref_odom_cloud(topic.encode(), a.ctypes.data_as(C.POINTER(C.c_float)), n)
        return a


class RefMapping:
    def __init__(self, lib, line_res, plane_res, sort_mode):
        self.lib = lib
        fp = C.POINTER(C.c_float); dp = C.POINTER(C.c_double); ip = C.POINTER(C.c_int)
        lib.ref_map_init.argtypes = [C.c_double, C.c_double, C.c_int]
        lib.ref_map_process.argtypes = [fp, C.c_int, fp, C.c_int, fp, C.c_int, dp, dp, C.c_double]
        lib.ref_map_state.argtypes = [dp, dp, dp, ip, ip, ip]
        lib.ref_map_cube.argtypes = [C.c_int, C.c_int, fp, C.c_int]
        lib.ref_map_cube_sizes.argtypes = [C.c_int, ip]
        lib.ref_map_published_pose.argtypes = [dp, dp]; lib.ref_map_published_pose.restype = C.c_long
        lib.ref_map_init(line_res, plane_res, sort_mode)

    def process(self, corner_last, surf_last, full, q, t, stamp):
        a = [np.ascontiguousarray(x, np.float32) for x in (corner_last, surf_last, full)]
        q = np.ascontiguousarray(q, np.float64); t = np.ascontiguousarray(t, np.float64)
        dp = C.POINTER(C.c_double); fp = C.POINTER(C.c_float)
        self.lib.ref_map_process(a[0].ctypes.data_as(fp), a[0].shape[0], a[1].ctypes.data_as(fp), a[1].shape[0], a[2].ctypes.data_as(fp), a[2].shape[0],
                                 q.ctypes.data_as(dp), t.ctypes.data_as(dp), float(stamp))
        pose = np.zeros(7); qm = np.zeros(4); tm = np.zeros(3); cen = np.zeros(3, np.int32); fr = np.zeros(1, np.int32); nv = np.zeros(1, np.int32)
        ip = C.POINTER(C.c_int)
        self.lib.ref_map_state(pose.ctypes.data_as(dp), qm.ctypes.data_as(dp), tm.ctypes.data_as(dp), cen.ctypes.data_as(ip), fr.ctypes.data_as(ip), nv.ctypes.data_as(ip))
        pq = np.zeros(4); pt = np.zeros(3)
        n_pub = self.lib.ref_map_published_pose(pq.ctypes.data_as(dp), pt.ctypes.data_as(dp))
        return {"pose": pose, "q_wmap_wodom": qm, "t_wmap_wodom": tm, "centre": tuple(int(v) for v in cen), "frames": int(fr[0]),
                "pub": np.concatenate([pq, pt]), "n_pub": n_pub}

    def sizes(self, which):
        s = np.zeros(NCUBE, np.int32)
        self.lib.ref_map_cube_sizes(which, s.ctypes.data_as(C.POINTER(C.c_int)))
        return s

    def cube(self, which, index, n):
        a = np.zeros((n, 4), np.float32)
        if n:
            self.lib.ref_map_cube(which, index, a.ctypes.data_as(C.POINTER(C.c_float)), n)
        return a
