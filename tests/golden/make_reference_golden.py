"""Records what the reference's own source files compute on the inputs of tests/test_oracle_vs_reference_source.py and
tests/test_gpu_vs_reference_source.py into reference_source.npz, so that those tests run without the reference.  Needs the
libraries of oracle/_ref (the reference's scanRegistration.cpp, laserOdometry.cpp, laserMapping.cpp and lidarFactor.hpp
compiled unmodified against oracle/ref_shim; `make -C oracle ref REF=<checkout of the reference>`).
Run from the repo root:  python tests/golden/make_reference_golden.py"""
import importlib
import os
import sys
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)
import pyoracle as orc  # noqa
import refsource as rs  # noqa
from test_oracle_vs_reference_source import SCROLL_PATH, factor_cases, scroll_clouds  # noqa
synth = importlib.import_module("a-loam_b200.synth")

G = {}


def put_clouds(key, out, raw=None):
    for name in rs.CLOUDS:
        G["%s/%s" % (key, name)] = rs.digest(out[name])
    if raw is not None:
        G[key + "/raw"] = rs.digest(raw)


def put_mapping_frames(key, frames):
    """frames: the RefMapping.process results of one run, in order"""
    for f in ("pose", "pub", "q_wmap_wodom", "t_wmap_wodom", "centre", "frames", "n_pub"):
        G["%s/%s" % (key, f)] = np.array([r[f] for r in frames])


def put_cube_stores(key, ref):
    """digests of the two cube stores after a frame; returns their per-cube sizes (2, NCUBE)"""
    sizes = np.stack([ref.sizes(w) for w in (0, 1)])
    for w in (0, 1):
        G["%s/cubes%d" % (key, w)] = rs.cube_store_digest([ref.cube(w, i, int(sizes[w, i])) for i in range(rs.NCUBE) if sizes[w, i]])
    return sizes


def scan(sensor, k, n_az):
    return synth.scan(sensor, k, n_az=n_az) if n_az else synth.scan(sensor, k)


# lidarFactor.hpp
lib = rs.ref_lib("libref_factor.so")
dp = rs.C.POINTER(rs.C.c_double)
lib.ref_factor_eval.argtypes = [rs.C.c_int, dp, rs.C.c_double, dp, dp, dp, dp, dp]
lib.ref_factor_eval.restype = rs.C.c_int
fin = np.full((12, 5, 21), np.nan); frows = np.zeros((12, 5), np.int32)
fr = np.zeros((12, 5, 3)); fjq = np.zeros((12, 5, 3, 4)); fjt = np.zeros((12, 5, 3, 3))
for seed in range(12):
    for c, (kind, pts, extra, q, t) in enumerate(factor_cases(seed)):
        a = [np.ascontiguousarray(v, np.float64).reshape(-1) for v in (pts, q, t)]
        r = np.zeros(3); jq = np.zeros(12); jt = np.zeros(9)
        f = lambda v: v.ctypes.data_as(dp)
        rows = lib.ref_factor_eval(kind, f(a[0]), float(extra), f(a[1]), f(a[2]), f(r), f(jq), f(jt))
        x = np.concatenate([[kind, extra], a[0], a[1], a[2]])
        fin[seed, c, :len(x)] = x; frows[seed, c] = rows
        fr[seed, c, :rows] = r[:rows]; fjq[seed, c, :rows] = jq[:rows * 4].reshape(rows, 4); fjt[seed, c, :rows] = jt[:rows * 3].reshape(rows, 3)
G.update({"factor/input": fin, "factor/rows": frows, "factor/r": fr, "factor/jq": fjq, "factor/jt": fjt})

# scanRegistration.cpp
lib = rs.ref_lib("libref_registration.so")
G["libm/atan_result_bytes"] = np.int32(lib.ref_reg_atan_result_bytes())
G["libm/sqrt_result_bytes"] = np.int32(lib.ref_reg_sqrt_result_bytes())
for sensor, n_az, scans in [("VLP-16", 900, 4), ("VLP-16", None, 2), ("HDL-32", None, 2), ("HDL-64", None, 2)]:
    ns, _, mr = synth.SENSORS[sensor][:3]
    ref = rs.ref_registration(ns, mr)
    for k in range(scans):
        raw = scan(sensor, k, n_az)
        got = ref.run(raw, orc.SORT_LITERAL)
        key = "reg/literal/%s/%s/%d" % (sensor, n_az, k)
        put_clouds(key, got, raw)
        core = slice(5, got["full"].shape[0] - 5)     # the reference's file-scope work arrays: entries [5, n - 5) are this scan's
        for a in ("curvature", "label", "picked"):
            G["%s/%s_core" % (key, a)] = rs.digest(got[a][core])

ns, _, mr = synth.SENSORS["VLP-16"][:3]
raw = synth.scan("VLP-16", 1, n_az=900).copy()
rng = np.random.default_rng(3)
raw[rng.integers(0, raw.shape[0], 200), rng.integers(0, 3, 200)] = np.nan
raw[rng.integers(0, raw.shape[0], 100), :3] *= 1e-3
put_clouds("reg/nan_and_close", rs.ref_registration(ns, mr).run(raw, orc.SORT_LITERAL), raw)

for sensor, n_az, scans in [("VLP-16", 900, 6), ("VLP-16", None, 4), ("HDL-32", None, 4), ("HDL-64", None, 4)]:
    ns, _, mr = synth.SENSORS[sensor][:3]
    ref = rs.ref_registration(ns, mr)
    for k in range(scans):
        raw = scan(sensor, k, n_az)
        put_clouds("reg/canonical/%s/%s/%d" % (sensor, n_az, k), ref.run(raw, orc.SORT_CANONICAL), raw)

# laserOdometry.cpp, fed with the features of the oracle (bit-identical to the reference's, see above)
for sensor, n_az, scans in [("VLP-16", 900, 6), ("HDL-64", None, 4)]:
    ns, _, mr = synth.SENSORS[sensor][:3]
    ref = rs.RefOdometry(rs.private_copy("libref_odometry.so", "%s_%d" % (sensor, scans)))
    out = []
    for k in range(scans):
        f = orc.Features(scan(sensor, k, n_az), ns, mr, mode=orc.SORT_LITERAL)
        out.append(ref.process(f, stamp=0.1 * (k + 1)))
        G["odom/%s/%d/corner_last" % (sensor, k)] = rs.digest(ref.cloud("/laser_cloud_corner_last"))
        G["odom/%s/%d/surf_last" % (sensor, k)] = rs.digest(ref.cloud("/laser_cloud_surf_last"))
    for f in ("q", "t", "qw", "tw", "counts", "pub_q", "pub_t", "n_pub"):
        G["odom/%s/%s" % (sensor, f)] = np.array([o[f] for o in out])

# laserMapping.cpp: the ring buffer scrolled by thin clouds
ref = rs.RefMapping(rs.private_copy("libref_mapping.so", "scroll"), 0.4, 0.8, orc.SORT_CANONICAL)
ident = np.array([0, 0, 0, 1.0])
frames, sizes = [], []
for k, (corner, surf) in enumerate(scroll_clouds()):
    frames.append(ref.process(corner, surf, surf, ident, np.array(SCROLL_PATH[k], float), stamp=0.1 * (k + 1)))
    sizes.append(put_cube_stores("scroll/%d" % k, ref))
    G["scroll/%d/input" % k] = rs.digest(np.concatenate([corner, surf]))
put_mapping_frames("scroll", frames)
G["scroll/cube_sizes"] = np.array(sizes, np.int32)

# laserMapping.cpp: the whole frame over a VLP-16 trajectory, fed with the oracle's features and odometry poses
ns, _, mr = synth.SENSORS["VLP-16"][:3]
for mode in ("canonical", "literal"):
    sm = orc.SORT_CANONICAL if mode == "canonical" else orc.SORT_LITERAL
    ref = rs.RefMapping(rs.private_copy("libref_mapping.so", "loop_" + mode), 0.2, 0.4, sm)
    od = orc.Odometry()
    q = np.array([0, 0, 0, 1.0]); t = np.zeros(3); qw = q.copy(); tw = t.copy()
    frames, sizes = [], []
    for k in range(6):
        f = orc.Features(synth.scan("VLP-16", k, n_az=900), ns, mr, mode=sm)
        if k > 0:
            q, t, _ = od.register(f.sharp, f.flat, q, t)
            qw, tw = orc.integrate_pose(qw, tw, q, t)
        od.set_last(f.less_sharp, f.less_flat)
        frames.append(ref.process(f.less_sharp, f.less_flat, f.full, qw, tw, stamp=0.1 * (k + 1)))
        sizes.append(put_cube_stores("loop/%s/%d" % (mode, k), ref))
    put_mapping_frames("loop/" + mode, frames)
    G["loop/%s/cube_sizes" % mode] = np.array(sizes, np.int32)

# the three nodes chained on their published topics
reg = rs.ref_registration(ns, mr)
odo = rs.RefOdometry(rs.private_copy("libref_odometry.so", "chain"))
mp = rs.RefMapping(rs.private_copy("libref_mapping.so", "chain"), 0.2, 0.4, orc.SORT_LITERAL)
chain = {"odom_q": [], "odom_t": [], "odom_pub": [], "map_pub": []}
for k in range(6):
    stamp = 0.1 * (k + 1)
    r = reg.run(synth.scan("VLP-16", k, n_az=900), orc.SORT_LITERAL)
    o = odo.process(types.SimpleNamespace(**{n: r[n] for n in rs.CLOUDS}), stamp)
    m = mp.process(odo.cloud("/laser_cloud_corner_last"), odo.cloud("/laser_cloud_surf_last"), odo.cloud("/velodyne_cloud_3"),
                   o["pub_q"], o["pub_t"], stamp)
    chain["odom_q"].append(o["qw"]); chain["odom_t"].append(o["tw"])
    chain["odom_pub"].append(np.concatenate([o["pub_q"], o["pub_t"]])); chain["map_pub"].append(m["pub"])
for f, v in chain.items():
    G["chain/" + f] = np.array(v)

digests = sorted((k, v) for k, v in G.items() if isinstance(v, str))
np.savez_compressed(rs.GOLDEN, digests=np.array(digests, dtype="S"), **{k: v for k, v in G.items() if not isinstance(v, str)})
print("written:", rs.GOLDEN, len(G), "entries,", os.path.getsize(rs.GOLDEN), "bytes")
