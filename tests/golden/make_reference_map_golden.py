"""Records what the reference's own laserMapping.cpp publishes at the end of its frames (laserMapping.cpp:803-848:
/laser_cloud_surround, /laser_cloud_map, /velodyne_cloud_registered) on the inputs of tests/test_oracle_map_outputs.py and
tests/test_gpu_map_outputs.py into reference_map_outputs.npz.  Clouds are stored as refsource.digest; poses and publish counts
as they are.

The node is compiled here, into a temporary directory, from tests/golden/ref_map_outputs.cc: oracle/ref_drivers/ref_mapping.cc
(the driver behind oracle/_ref/libref_mapping.so) with read access to the published topics added, against the same stand-in
headers and flags as `make -C oracle ref`.  Needs a checkout of the reference.
Run from the repo root:  python tests/golden/make_reference_map_golden.py [--ref <checkout of the reference>]"""
import argparse
import ctypes as C
import importlib
import os
import shutil
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)
import pyoracle as orc  # noqa
import refsource as rs  # noqa
from test_oracle_map_outputs import GOLDEN, RUNS, TOPICS, input_digest, publishes, run_frames  # noqa
synth = importlib.import_module("a-loam_b200.synth")
ORACLE = os.path.join(ROOT, "oracle")


def build_node(ref, out_dir):
    """the flags of oracle/Makefile's `ref` target (REFFLAGS) and the sources of its libref_mapping.so"""
    so = os.path.join(out_dir, "libref_map_outputs.so")
    cmd = [os.environ.get("CXX", "g++"), "-std=c++17", "-O3", "-fPIC", "-ffp-contract=off", "-fno-gnu-unique", "-w",
           "-I", os.path.join(ORACLE, "ref_shim"), "-I", ORACLE, "-I", os.path.join(ref, "include"), "-I", os.path.join(ref, "src"),
           '-DREF_LASER_MAPPING_CPP="%s"' % os.path.join(ref, "src", "laserMapping.cpp"), "-shared", "-o", so,
           os.path.join(ROOT, "tests", "golden", "ref_map_outputs.cc")] + [os.path.join(ORACLE, f) for f in ("voxelgrid.cc", "kdtree.cc", "lm.cc", "mapping.cc")]
    subprocess.check_call(cmd)
    return so


def published(lib, topic):
    """(number of messages published on `topic` so far, the last one's cloud as (n, 4) float32)"""
    n = lib.ref_map_cloud(topic.encode(), None, 0)
    a = np.zeros((max(n, 0), 4), np.float32)
    if n > 0:
        lib.ref_map_cloud(topic.encode(), a.ctypes.data_as(C.POINTER(C.c_float)), n)
    return int(lib.ref_map_published(topic.encode())), a


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ref", default=os.environ.get("REF", "/root/reference"), help="checkout of the reference")
    args = ap.parse_args()
    tmp = tempfile.mkdtemp(prefix="ref_map_outputs_")
    so = build_node(args.ref, tmp)
    G = {}
    for run, (line_res, plane_res) in RUNS.items():
        path = os.path.join(tmp, "libref_map_outputs_%s.so" % run)   # a private copy = private file-scope state of the node
        shutil.copy(so, path)
        lib = C.CDLL(path)
        lib.ref_map_cloud.argtypes = [C.c_char_p, C.POINTER(C.c_float), C.c_int]
        lib.ref_map_published.argtypes = [C.c_char_p]; lib.ref_map_published.restype = C.c_long
        ref = rs.RefMapping(lib, line_res, plane_res, orc.SORT_CANONICAL)
        poses, n_pub = [], []
        for k, (corner, surf, full, q, t) in enumerate(run_frames(run, orc, synth)):
            G["%s/%d/input" % (run, k)] = input_digest(corner, surf, full)
            before = {name: published(lib, topic)[0] for name, topic in TOPICS.items()}
            r = ref.process(corner, surf, full, q, t, stamp=0.1 * (k + 1))
            poses.append(r["pose"])
            counts = []
            for name, topic in TOPICS.items():
                n, cloud = published(lib, topic)
                counts.append(n)
                if n > before[name]:
                    assert publishes(name, k), (run, k, name)
                    G["%s/%d/%s" % (run, k, name)] = rs.digest(cloud)
                else:
                    assert not publishes(name, k), (run, k, name)
            n_pub.append(counts)
        G[run + "/pose"] = np.array(poses)
        G[run + "/n_pub"] = np.array(n_pub, np.int64)
    shutil.rmtree(tmp, ignore_errors=True)
    digests = sorted((k, v) for k, v in G.items() if isinstance(v, str))
    np.savez_compressed(GOLDEN, digests=np.array(digests, dtype="S"), **{k: v for k, v in G.items() if not isinstance(v, str)})
    print("written:", GOLDEN, len(G), "entries,", os.path.getsize(GOLDEN), "bytes")


if __name__ == "__main__":
    main()
