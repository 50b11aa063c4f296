"""CPU: the three clouds alaserMapping publishes at the end of a frame (laserMapping.cpp:803-848) -- /laser_cloud_surround
(every 5th frame), /laser_cloud_map (every 20th) and /velodyne_cloud_registered (every frame) -- built from the oracle equal
what the reference's own laserMapping.cpp published, bit for bit, on every publishing frame.  The reference side is stored in
tests/golden/reference_map_outputs.npz (tests/golden/make_reference_map_golden.py).

The inputs below are shared with tests/test_gpu_map_outputs.py and the golden generator."""
import os

import numpy as np
import pytest

from refsource import NCUBE, digest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "reference_map_outputs.npz")
TOPICS = {"surround": "/laser_cloud_surround", "map": "/laser_cloud_map", "registered": "/velodyne_cloud_registered"}
N_FRAMES = 21     # /laser_cloud_map at frames 0 and 20, /laser_cloud_surround at 0, 5, 10, 15, 20

# translations of the odometry pose: every frame moves far enough that the submap stays thin (no optimisation, so the pose is
# the odometry pose), and the path scrolls the 21 x 21 x 11 ring buffer in all six directions
SCROLL_T = [(0, 0, 0), (60, -35, 12), (130, -80, 30), (260, -170, 75), (420, -290, 140), (300, -100, 60), (-90, 40, -30),
            (-400, 380, -160), (-700, 600, -260), (-640, 610, -250), (-380, 420, -150), (-120, 230, -40), (200, -20, 70),
            (420, -200, 170), (700, -430, 280), (560, -700, 200), (300, -980, 100), (20, -1250, 0), (-260, -1000, -110),
            (-540, -760, -220), (-820, -520, -330)]
LOOP_SCANS = 21


def publishes(topic, frame):
    """the reference's cadence: frameCount % 5 (:806), % 20 (:823), every frame (:838)"""
    return {"surround": frame % 5 == 0, "map": frame % 20 == 0, "registered": True}[topic]


def scroll_frames():
    """(corner_last, surf_last, full, q_wodom, t_wodom) of the scroll run: thin seeded clouds and a separate seeded full cloud
    with non-trivial intensities, the odometry pose turning about z (and a little about x) along SCROLL_T"""
    rng = np.random.default_rng(29)
    for k, t in enumerate(SCROLL_T):
        corner = (rng.normal(size=(6, 4)) * [8, 8, 2, 0]).astype(np.float32)
        surf = (rng.normal(size=(300, 4)) * [30, 30, 3, 0]).astype(np.float32)
        full = (rng.normal(size=(1500, 4)) * [40, 40, 4, 0]).astype(np.float32)
        full[:, 3] = rng.integers(0, 16, 1500) + 0.1 * rng.random(1500).astype(np.float32)   # scanID + 0.1 * relTime
        yaw, roll = 0.25 * k, 0.05 * np.sin(k)
        q = np.array([np.sin(roll / 2) * np.cos(yaw / 2), -np.sin(roll / 2) * np.sin(yaw / 2), np.cos(roll / 2) * np.sin(yaw / 2),
                      np.cos(roll / 2) * np.cos(yaw / 2)])
        yield corner, surf, full, q, np.array(t, float)


def loop_frames(orc, synth):
    """(corner_last, surf_last, full, q_wodom, t_wodom) of the loop run: VLP-16 scans through the oracle's features and odometry"""
    ns, _, mr = synth.SENSORS["VLP-16"][:3]
    od = orc.Odometry()
    q = np.array([0, 0, 0, 1.0]); t = np.zeros(3); qw = q.copy(); tw = t.copy()
    for k in range(LOOP_SCANS):
        f = orc.Features(synth.scan("VLP-16", k, n_az=900), ns, mr, mode=orc.SORT_CANONICAL)
        if k > 0:
            q, t, _ = od.register(f.sharp, f.flat, q, t)
            qw, tw = orc.integrate_pose(qw, tw, q, t)
        od.set_last(f.less_sharp, f.less_flat)
        yield f.less_sharp, f.less_flat, f.full, qw.copy(), tw.copy()


RUNS = {"scroll": (0.4, 0.8), "loop": (0.2, 0.4)}   # (line_res, plane_res)


def run_frames(run, orc, synth):
    return scroll_frames() if run == "scroll" else loop_frames(orc, synth)


def input_digest(corner, surf, full):
    return digest(np.concatenate([corner, surf, full]))


def region_cloud(get_cube, cubes):
    """per cube the corner points, then the surf points (:811-812, :828-829); get_cube(which, index) -> (n, 4)"""
    parts = [get_cube(w, i) for i in cubes for w in (0, 1)]
    parts = [p for p in parts if p.shape[0]]
    return np.concatenate(parts) if parts else np.zeros((0, 4), np.float32)


def point_associate_to_map(cloud, q, t):
    """pointAssociateToMap (laserMapping.cpp:154-163) of every point: q_w_curr * p + t_w_curr in double, in the operation order
    of Eigen's Quaternion * Vector3 (uv = u x p; uv += uv; p + w uv + u x uv), stored as float; the intensity is kept.  numpy
    runs each operation on its own (no contraction), like the reference's x86-64 build; the test below pins it to the clouds
    the reference published"""
    c = np.ascontiguousarray(cloud, np.float32)
    p = c[:, :3].astype(np.float64)
    u = np.broadcast_to(np.asarray(q[:3], np.float64), p.shape)
    w, t = float(q[3]), np.asarray(t, np.float64)
    uv = np.cross(u, p)
    uv = uv + uv
    out = c.copy()
    out[:, :3] = (((p + w * uv) + np.cross(u, uv)) + t).astype(np.float32)
    return out


def oracle_outputs(cm, pose, full, frame):
    """the clouds the reference publishes after `frame`, built from the oracle's cube store and pose"""
    out = {"registered": point_associate_to_map(full, pose[:4], pose[4:])}
    if publishes("surround", frame):
        out["surround"] = region_cloud(cm.cube, cm.state()["valid"])
    if publishes("map", frame):
        out["map"] = region_cloud(cm.cube, range(NCUBE))
    return out


_GOLDEN = None


def golden():
    global _GOLDEN
    if _GOLDEN is None:
        with np.load(GOLDEN, allow_pickle=False) as z:
            _GOLDEN = {k: z[k] for k in z.files if k != "digests"}
            _GOLDEN.update((k.decode(), v.decode()) for k, v in z["digests"])
    return _GOLDEN


@pytest.mark.parametrize("run", ["scroll", "loop"])
def test_oracle_map_outputs_equal_the_reference(orc, synth, run):
    """oracle surround, map and registered clouds == what laserMapping.cpp published, on every publishing frame; the reference
    published exactly on its cadence"""
    G = golden()
    line_res, plane_res = RUNS[run]
    cm = orc.CubeMap()
    counts = np.zeros(3, np.int64)
    for k, (corner, surf, full, q, t) in enumerate(run_frames(run, orc, synth)):
        assert input_digest(corner, surf, full) == G["%s/%d/input" % (run, k)], "not the inputs the golden data was recorded on"
        pose, info = cm.step(corner, surf, q, t, line_res, plane_res, sort_mode=orc.SORT_CANONICAL)
        if run == "scroll":
            assert not info["optimised"], k
        assert np.array_equal(pose, G[run + "/pose"][k]), k
        for j, name in enumerate(TOPICS):
            counts[j] += publishes(name, k)
        assert np.array_equal(G[run + "/n_pub"][k], counts), (k, G[run + "/n_pub"][k])
        for name, cloud in oracle_outputs(cm, pose, full, k).items():
            assert digest(cloud) == G["%s/%d/%s" % (run, k, name)], (run, k, name, cloud.shape)
    assert counts.tolist() == [5, 2, N_FRAMES]

