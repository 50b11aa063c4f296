"""GPU: the CUDA path against THE REFERENCE'S OWN SOURCE FILES in execution -- scanRegistration.cpp and laserOdometry.cpp compiled
unmodified against the stand-in headers of oracle/ref_shim (oracle/_ref), as recorded in tests/golden/reference_source.npz.  The
other GPU tests compare with the oracle restatement, and tests/test_oracle_vs_reference_source.py (CPU) shows the restatement
bit-identical to the reference's sources; this file closes the triangle directly.  Where only digests of the reference's clouds
are stored, the oracle's clouds stand in for them once their digests match, i.e. once they are the same bits."""
import numpy as np
import pytest

from conftest import rot_angle
from refsource import CLOUDS, assert_clouds, assert_digest, golden

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("sensor", ["VLP-16", "HDL-32", "HDL-64"])
@pytest.mark.parametrize("index", [0, 3])
def test_features_match_the_reference_source(sensor, index, aloam, orc, synth, scans):
    """aloam_extract_features vs the clouds the reference's laserCloudHandler publishes: coordinates bit-exact, ring ids equal,
    relTime fraction within the atan2f rounding of the two libm's (as against the oracle, tests/test_gpu_features.py)"""
    ns, _, mr = synth.SENSORS[sensor][:3]
    raw = scans(sensor, index)
    f = orc.Features(raw, ns, mr, mode=orc.SORT_CANONICAL)
    assert_clouds("reg/canonical/%s/None/%d" % (sensor, index), f, raw)      # f's clouds are the reference's, bit for bit
    ref = {name: getattr(f, name) for name in CLOUDS}
    c = aloam.Aloam(n_scans=ns, max_points=200000)
    got = c.extract_features(raw)
    c.close()
    for name in CLOUDS:
        g, r_ = got[name], ref[name]
        assert g.shape == r_.shape, name
        assert np.array_equal(g[:, :3], r_[:, :3]), name
        assert np.array_equal(g[:, 3].astype(np.int32), r_[:, 3].astype(np.int32)), name
        assert np.abs(g[:, 3] - r_[:, 3]).max() <= 1e-5, name


def test_odometry_poses_match_the_reference_source_chain(aloam, synth, scans):
    """aloam_scan_to_pose per scan vs the reference's scanRegistration -> laserOdometry chain (its own source for feature
    extraction, TransformToStart, correspondence search, block construction and pose integration): the north_star tolerance is
    1e-4 m / 1e-4 rad, the bar here is ten times tighter"""
    g = golden()
    ns = synth.SENSORS["VLP-16"][0]
    c = aloam.Aloam(n_scans=ns, max_points=40000)
    moved = 0.0
    for k in range(5):
        raw = scans("VLP-16", k, n_az=900)
        assert_digest("reg/canonical/VLP-16/900/%d/raw" % k, raw, "not the scan the golden data was recorded on")
        gq, gt, _ = c.scan_to_pose(raw)
        qw, tw = g["chain/odom_q"][k], g["chain/odom_t"][k]
        assert np.abs(gt - tw).max() < 1e-5 and rot_angle(gq, qw) < 1e-5, (k, gt - tw)
        moved = max(moved, float(np.abs(tw).max()))
    c.close()
    assert moved > 0.05
