"""CPU: the oracle against THE REFERENCE'S OWN SOURCE FILES, compiled unmodified against the stand-in headers of
oracle/ref_shim (ROS / PCL / Eigen / Ceres are not available to build against; see oracle/ref_shim/README.md).  What is
pinned here is the in-tree arithmetic and control flow -- a transcription error in oracle/*.cc would show up as a difference.
The third-party semantics behind the stand-ins (VoxelGrid, kd-tree, Eigen's operation order, Jets) remain restatements and are
shared by both sides of the comparison.  What the reference's sources computed on these inputs is stored in
tests/golden/reference_source.npz (tests/golden/make_reference_golden.py runs them from oracle/_ref); bit-exact comparisons of
clouds and work arrays go through their digests (refsource.digest)."""
import numpy as np
import pytest

from refsource import NCUBE, assert_clouds, assert_digest, cube_store_digest, golden

SCROLL_PATH = [(0, 0, 0), (60, -35, 12), (130, -80, 30), (260, -170, 75), (420, -290, 140), (300, -100, 60), (-90, 40, -30),
               (-400, 380, -160), (-700, 600, -260), (-640, 610, -250)]


# ------------------------------------------------------------------------------------------------ lidarFactor.hpp
def factor_cases(seed):
    """(kind, points, extra, q, t) of the residual blocks evaluated for `seed`: kind 0 edge, 1 plane (extra = s), 2 plane-norm
    (extra = d)"""
    rng = np.random.default_rng(seed)
    q = rng.normal(size=4); q /= np.linalg.norm(q)
    if seed % 3 == 0:
        q = np.array([0.01, -0.02, 0.015, 1.0]) * rng.uniform(0.5, 1.5, 4); q /= np.linalg.norm(q)   # the small rotations of odometry
    t = rng.normal(size=3)
    for s in (1.0, float(rng.uniform(0.05, 0.95))):
        cp, a, b, c = (rng.normal(size=3) * 10 for _ in range(4))
        yield 0, [cp, a, b], s, q, t
        yield 1, [cp, a, b, c], s, q, t
        if s == 1.0:
            n = rng.normal(size=3); n /= np.linalg.norm(n); d = float(rng.normal())
            yield 2, [cp, n], d, q, t


def plus_jacobian(q):
    """d Plus(q, delta) / d delta at 0 for ceres::EigenQuaternionParameterization, storage x, y, z, w"""
    x, y, z, w = q
    return np.array([[w, z, -y], [-z, w, x], [y, -x, w], [-x, -y, -z]])


@pytest.mark.parametrize("seed", range(12))
def test_the_three_cost_functions_of_lidarFactor_hpp(orc, seed):
    """residuals and Jacobians of the reference's functors (its own operator() text, through its own Create()) equal the
    oracle's: Jet autodiff and the closed form, for s = 1 (the reference build) and s != 1 (DISTORTION 1)"""
    g = golden()
    make = {0: orc.make_edge, 1: orc.make_plane, 2: orc.make_plane_norm}
    n = 0
    for c, (kind, pts, extra, q, t) in enumerate(factor_cases(seed)):
        x = np.concatenate([[kind, extra], np.reshape(pts, -1), q, t])
        assert np.array_equal(g["factor/input"][seed, c, :len(x)], x), (seed, c, "not the block the golden data was recorded on")
        rows = g["factor/rows"][seed, c]
        assert rows in (1, 3)
        r_ref, jq, jt = g["factor/r"][seed, c, :rows], g["factor/jq"][seed, c, :rows], g["factor/jt"][seed, c, :rows]
        j_ref = np.concatenate([jq @ plus_jacobian(q), jt], axis=1)            # tangent [dtheta, dt], what the solver sees
        block = make[kind](*pts, extra)
        for autodiff in (True, False):
            r_o, j_o, _ = orc.evaluate([block], np.concatenate([q, t]), huber=1e12, autodiff=autodiff)   # huber far away: no correction
            assert np.allclose(r_o, r_ref, rtol=1e-12, atol=1e-12), (kind, extra, autodiff)
            assert np.allclose(np.asarray(j_o).reshape(j_ref.shape), j_ref, rtol=1e-10, atol=1e-10), (kind, extra, autodiff)
        n += 1
    assert n == 5


# ------------------------------------------------------------------------------------------------ scanRegistration.cpp


def test_which_libm_overloads_the_reference_source_sees():
    """scanRegistration.cpp:166 calls atan / sqrt unqualified on floats: with headers that never pull <math.h>'s std overloads
    into the global namespace (GCC 5 of the reference's docker image; the oracle/_ref build) they are the C double functions,
    which is what oracle/features.cc and the CUDA kernel restate (DESIGN.md section 2, row 13)"""
    g = golden()
    assert int(g["libm/atan_result_bytes"]) == 8 and int(g["libm/sqrt_result_bytes"]) == 8


@pytest.mark.parametrize("sensor,n_az,scans", [("VLP-16", 900, 4), ("VLP-16", None, 2), ("HDL-32", None, 2), ("HDL-64", None, 2)])
def test_scan_registration_source_equals_oracle_features(orc, synth, sensor, n_az, scans):
    """every output of the reference's laserCloudHandler (its own source text, std::sort and all) is bit-identical to
    oracle/features.cc in LITERAL mode: the ring-major cloud with its ring.relTime intensities, the four feature clouds in
    publishing order, and the curvature / label / neighbour-picked work arrays"""
    ns, _, mr = synth.SENSORS[sensor][:3]
    for k in range(scans):
        raw = synth.scan(sensor, k, n_az=n_az) if n_az else synth.scan(sensor, k)
        want = orc.Features(raw, ns, mr, mode=orc.SORT_LITERAL)
        key = "reg/literal/%s/%s/%d" % (sensor, n_az, k)
        assert_clouds(key, want, raw)
        # the reference's work arrays are file-scope and only entries [5, n - 5) are written per scan (:256-268): compare those
        n = want.full.shape[0]
        core = slice(5, n - 5)
        assert_digest(key + "/curvature_core", want.curvature[core])
        assert_digest(key + "/label_core", want.label[core])
        assert_digest(key + "/picked_core", want.picked[core])


def test_scan_registration_source_with_nan_and_close_points(orc, synth):
    ns, _, mr = synth.SENSORS["VLP-16"][:3]
    raw = synth.scan("VLP-16", 1, n_az=900).copy()
    rng = np.random.default_rng(3)
    raw[rng.integers(0, raw.shape[0], 200), rng.integers(0, 3, 200)] = np.nan
    raw[rng.integers(0, raw.shape[0], 100), :3] *= 1e-3                       # inside minimum_range
    assert_clouds("reg/nan_and_close", orc.Features(raw, ns, mr, mode=orc.SORT_LITERAL), raw)


@pytest.mark.parametrize("sensor,n_az,scans", [("VLP-16", 900, 6), ("VLP-16", None, 4), ("HDL-32", None, 4), ("HDL-64", None, 4)])
def test_canonical_tie_order_changes_nothing_on_these_scans(orc, synth, sensor, n_az, scans):
    """the CUDA path defines ties by index (CANONICAL); on the synthetic scans the literal std::sort order of the reference
    source gives the same features, so GPU == oracle(CANONICAL) == reference source.  The reference side ran its own
    std::sort for the picks, canonical ties in VoxelGrid"""
    ns, _, mr = synth.SENSORS[sensor][:3]
    for k in range(scans):
        raw = synth.scan(sensor, k, n_az=n_az) if n_az else synth.scan(sensor, k)
        assert_clouds("reg/canonical/%s/%s/%d" % (sensor, n_az, k), orc.Features(raw, ns, mr, mode=orc.SORT_CANONICAL), raw)


# ------------------------------------------------------------------------------------------------ laserOdometry.cpp
@pytest.mark.parametrize("sensor,n_az,scans", [("VLP-16", 900, 6), ("HDL-64", None, 4)])
def test_laser_odometry_source_equals_oracle_odometry(orc, synth, sensor, n_az, scans):
    """the reference's laserOdometry.cpp (its own TransformToStart, correspondence search, block construction, pose
    integration and cloud swap; ceres::Solve = oracle/lm.cc behind the stand-in) run scan after scan gives bit-identical
    q_last_curr / t_last_curr, world pose and correspondence counts to oracle/odometry.cc, and republishes the clouds unchanged"""
    g = golden()
    ns, _, mr = synth.SENSORS[sensor][:3]
    ref = lambda f, k: g["odom/%s/%s" % (sensor, f)][k]
    od = orc.Odometry()
    q = np.array([0, 0, 0, 1.0]); t = np.zeros(3); qw = q.copy(); tw = t.copy()
    moved = 0.0
    for k in range(scans):
        raw = synth.scan(sensor, k, n_az=n_az) if n_az else synth.scan(sensor, k)
        f = orc.Features(raw, ns, mr, mode=orc.SORT_LITERAL)
        if k > 0:
            q, t, info = od.register(f.sharp, f.flat, q, t)
            qw, tw = orc.integrate_pose(qw, tw, q, t)
            assert ref("counts", k).tolist() == [info["corner_corr"], info["plane_corr"]], (k, ref("counts", k), info)
            moved = max(moved, float(np.abs(t).max()))
        od.set_last(f.less_sharp, f.less_flat)
        assert np.array_equal(ref("q", k), q) and np.array_equal(ref("t", k), t), (k, ref("q", k) - q, ref("t", k) - t)
        assert np.array_equal(ref("qw", k), qw) and np.array_equal(ref("tw", k), tw), k
        assert ref("n_pub", k) == k + 1 and np.array_equal(ref("pub_q", k), qw) and np.array_equal(ref("pub_t", k), tw)
        assert_digest("odom/%s/%d/corner_last" % (sensor, k), f.less_sharp)
        assert_digest("odom/%s/%d/surf_last" % (sensor, k), f.less_flat)
    assert moved > 0.05     # the trajectory moves: the comparison is not between two identities


# ------------------------------------------------------------------------------------------------ laserMapping.cpp


def _compare_cube_stores(key, k, cm):
    """all 2 x 4851 cubes after frame k: sizes, and the contents of every non-empty cube, bit for bit"""
    g = golden()
    nonempty = 0
    for which in (0, 1):
        sizes = g[key + "/cube_sizes"][k, which]
        cubes = []
        for idx in range(NCUBE):
            want = cm.cube(which, idx) if sizes[idx] or idx % 97 == 0 else None
            if want is None:
                continue
            assert want.shape[0] == sizes[idx], (key, k, which, idx, want.shape[0], sizes[idx])
            if sizes[idx]:
                nonempty += 1
                cubes.append(want)
        assert cube_store_digest(cubes) == g["%s/%d/cubes%d" % (key, k, which)], (key, k, which)
    return nonempty


def _compare_frame(key, k, pose, so):
    g = golden()
    got = lambda f: g["%s/%s" % (key, f)][k]
    assert got("frames") == k + 1 and got("n_pub") == k + 1
    assert np.array_equal(got("pose"), pose), (k, got("pose") - pose)
    assert np.array_equal(got("pub"), pose)
    assert tuple(got("centre")) == so["centre"], (k, got("centre"), so["centre"])
    assert np.array_equal(got("q_wmap_wodom"), so["q_wmap_wodom"]) and np.array_equal(got("t_wmap_wodom"), so["t_wmap_wodom"])


def scroll_clouds():
    """the thin (corner, surf) clouds of the frames along SCROLL_PATH"""
    rng = np.random.default_rng(11)
    for _ in SCROLL_PATH:
        corner = (rng.normal(size=(6, 4)) * [8, 8, 2, 0]).astype(np.float32)
        surf = (rng.normal(size=(300, 4)) * [30, 30, 3, 0]).astype(np.float32)
        yield corner, surf


def test_laser_mapping_source_ring_buffer_scrolls_like_the_oracle(orc):
    """thin clouds (no optimisation: the pose is the odometry pose) along a path that scrolls the 21 x 21 x 11 ring buffer in all
    six directions: centre indices, T_wmap_wodom and EVERY cube of the reference's laserCloudCornerArray / laserCloudSurfArray
    (laserMapping.cpp:309-505 shift loops, :736-801 insertion + per-cube VoxelGrid) equal oracle/cubemap.cc bit for bit"""
    cm = orc.CubeMap()
    ident = np.array([0, 0, 0, 1.0])
    for k, (corner, surf) in enumerate(scroll_clouds()):
        assert_digest("scroll/%d/input" % k, np.concatenate([corner, surf]), "not the clouds the golden data was recorded on")
        pose, info = cm.step(corner, surf, ident, np.array(SCROLL_PATH[k], float), 0.4, 0.8, sort_mode=orc.SORT_CANONICAL)
        assert not info["optimised"]
        _compare_frame("scroll", k, pose, cm.state())
        assert _compare_cube_stores("scroll", k, cm) >= 2


@pytest.mark.parametrize("mode", ["canonical", "literal"])
def test_laser_mapping_source_equals_oracle_mapping_loop(orc, synth, mode):
    """the whole alaserMapping frame of the reference's own source (pose hand-off, shift, submap gather, stack filters, 5-NN,
    line / plane fits, two ceres::Solve passes, transformUpdate, insertion, per-cube re-filter) over a VLP-16 trajectory equals
    oracle/cubemap.cc + mapping.cc bit for bit: refined pose, T_wmap_wodom, and every cube.  The reference ran with the VLP-16
    launch file's resolutions (0.2, 0.4)"""
    sm = orc.SORT_CANONICAL if mode == "canonical" else orc.SORT_LITERAL
    ns, _, mr = synth.SENSORS["VLP-16"][:3]
    cm = orc.CubeMap()
    od = orc.Odometry()
    q = np.array([0, 0, 0, 1.0]); t = np.zeros(3); qw = q.copy(); tw = t.copy()
    optimised = 0
    refined = 0.0
    for k in range(6):
        f = orc.Features(synth.scan("VLP-16", k, n_az=900), ns, mr, mode=sm)
        if k > 0:
            q, t, _ = od.register(f.sharp, f.flat, q, t)
            qw, tw = orc.integrate_pose(qw, tw, q, t)
        od.set_last(f.less_sharp, f.less_flat)
        pose, info = cm.step(f.less_sharp, f.less_flat, qw, tw, 0.2, 0.4, sort_mode=sm)
        optimised += int(info["optimised"])
        refined = max(refined, float(np.abs(pose[4:] - tw).max()))
        _compare_frame("loop/" + mode, k, pose, cm.state())
        assert _compare_cube_stores("loop/" + mode, k, cm) >= 2
    assert optimised >= 4 and refined > 0      # the optimisation ran and moved the pose: not a comparison of two hand-offs


# ------------------------------------------------------------------------------------------------ the three nodes chained
def test_the_three_reference_nodes_chained_equal_the_oracle_chain(orc, synth):
    """raw scans through the reference's scanRegistration -> laserOdometry -> laserMapping sources, each node fed with what the
    previous one PUBLISHED (the topics of the real pipeline), against the oracle's extract -> register -> integrate -> mapping step:
    /laser_odom_to_init and /aft_mapped_to_init equal the oracle's poses bit for bit on every frame"""
    g = golden()
    ns, _, mr = synth.SENSORS["VLP-16"][:3]
    cm = orc.CubeMap(); od = orc.Odometry()
    q = np.array([0, 0, 0, 1.0]); t = np.zeros(3); qw = q.copy(); tw = t.copy()
    drift = 0.0
    for k in range(6):
        raw = synth.scan("VLP-16", k, n_az=900)
        f = orc.Features(raw, ns, mr, mode=orc.SORT_LITERAL)
        if k > 0:
            q, t, _ = od.register(f.sharp, f.flat, q, t)
            qw, tw = orc.integrate_pose(qw, tw, q, t)
        od.set_last(f.less_sharp, f.less_flat)
        pose, info = cm.step(f.less_sharp, f.less_flat, qw, tw, 0.2, 0.4, sort_mode=orc.SORT_LITERAL)
        assert np.array_equal(g["chain/odom_pub"][k], np.concatenate([qw, tw])), k
        assert np.array_equal(g["chain/map_pub"][k], pose), (k, g["chain/map_pub"][k] - pose)
        drift = max(drift, float(np.abs(pose[4:] - tw).max()))
    assert drift > 0
