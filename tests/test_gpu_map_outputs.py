"""GPU: the map outputs of laserMapping.cpp:803-848 read out of the device cube store -- aloam_mapper_export (surround / whole
map), aloam_mapper_associate_to_map (/velodyne_cloud_registered) and aloam_scan_stream_mapped_registered -- against the oracle
(bit for bit), the reference's published clouds (tests/golden/reference_map_outputs.npz) and the per-scan API."""
import ctypes as C

import numpy as np
import pytest

from refsource import NCUBE, digest
from test_oracle_map_outputs import (RUNS, golden, input_digest, loop_frames, point_associate_to_map, publishes, region_cloud,
                                     scroll_frames)

pytestmark = pytest.mark.gpu

ERR_INVALID_ARG, ERR_CAPACITY, ERR_STATE = -1, -4, -9


def export_raw(aloam, ctx, region, ptr, capacity):
    """aloam_mapper_export without the Python wrapper's raise: (return code, *n_points)"""
    n = C.c_longlong(-1)
    rc = aloam.lib().aloam_mapper_export(ctx._h, region, C.c_void_p(ptr) if ptr else None, capacity, C.byref(n))
    return rc, n.value


def cube_store_cloud(ctx, cubes):
    return region_cloud(ctx.mapper_cube, cubes)


def test_scroll_outputs_equal_the_oracle_and_the_reference(aloam, orc):
    """thin clouds, pose = odometry pose: on every frame the registered full cloud, the surround and the whole map equal the
    oracle bit for bit; on the reference's publishing frames they also equal what laserMapping.cpp published"""
    G = golden()
    line_res, plane_res = RUNS["scroll"]
    c = aloam.Aloam(n_scans=16, max_points=20000, max_map_points=200000, line_res=line_res, plane_res=plane_res)
    c.mapper_reset()
    cm = orc.CubeMap()
    for k, (corner, surf, full, q, t) in enumerate(scroll_frames()):
        assert input_digest(corner, surf, full) == G["scroll/%d/input" % k]
        pose, info = cm.step(corner, surf, q, t, line_res, plane_res, sort_mode=orc.SORT_CANONICAL)
        gq, gt, st = c.mapper_step(corner, surf, q, t)
        assert np.array_equal(np.concatenate([gq, gt]), pose), k
        got = {"registered": c.mapper_associate_to_map(full), "surround": c.mapper_export(aloam.MAP_SURROUND),
               "map": c.mapper_export(aloam.MAP_ALL)}
        want = {"registered": point_associate_to_map(full, pose[:4], pose[4:]),
                "surround": region_cloud(cm.cube, cm.state()["valid"]), "map": region_cloud(cm.cube, range(NCUBE))}
        for name in got:
            assert np.array_equal(got[name], want[name]), (k, name, got[name].shape, want[name].shape)
            if publishes(name, k):
                assert digest(got[name]) == G["scroll/%d/%s" % (k, name)], (k, name)
    c.close()


def test_loop_outputs(aloam, orc, synth):
    """VLP-16 loop with the optimisation running: the registered cloud is pointAssociateToMap with the GPU's pose
    (bit for bit) and differs from the reference's only by the difference of the two poses; the whole map and the surround are
    the cube store's cubes in the reference's order"""
    G = golden()
    line_res, plane_res = RUNS["loop"]
    c = aloam.Aloam(n_scans=16, max_points=40000, max_map_points=400000, line_res=line_res, plane_res=plane_res)
    c.mapper_reset()
    for k, (corner, surf, full, q, t) in enumerate(loop_frames(orc, synth)):
        assert input_digest(corner, surf, full) == G["loop/%d/input" % k]
        gq, gt, _ = c.mapper_step(corner, surf, q, t)
        reg = c.mapper_associate_to_map(full)
        assert np.array_equal(reg, point_associate_to_map(full, gq, gt)), k
        ref_pose = G["loop/pose"][k]
        ref_reg = point_associate_to_map(full, ref_pose[:4], ref_pose[4:])
        assert digest(ref_reg) == G["loop/%d/registered" % k]
        # against the reference's cloud: the same points, moved only by the difference of the two refined poses (the device's
        # follows the reference's to float rounding that compounds through the cube store; on a B200 the registered points of
        # frame 18 of this loop differ by up to 2 cm).  |(R1 - R2) p + t1 - t2| <= angle(q1, q2) |p| + |t1 - t2|, plus the float32 store
        assert reg.shape == ref_reg.shape
        s = 1.0 if np.dot(gq, ref_pose[:4]) >= 0 else -1.0
        angle = 4.0 * np.arcsin(min(1.0, np.linalg.norm(gq - s * ref_pose[:4]) / 2.0))
        rng = np.linalg.norm(full[:, :3].astype(np.float64), axis=1)
        bound = 1.01 * angle * rng + np.linalg.norm(gt - ref_pose[4:]) + 1e-5 + 1e-6 * (rng + np.linalg.norm(gt))
        assert (np.linalg.norm((reg[:, :3] - ref_reg[:, :3]).astype(np.float64), axis=1) <= bound).all(), k
        assert np.array_equal(reg[:, 3], ref_reg[:, 3])
    st = c.mapper_state()
    whole = c.mapper_export(aloam.MAP_ALL)
    assert whole.shape[0] == st["total_corner"] + st["total_surf"] > 0
    assert np.array_equal(whole, cube_store_cloud(c, range(NCUBE)))
    assert np.array_equal(c.mapper_export(aloam.MAP_SURROUND), cube_store_cloud(c, st["valid"]))
    c.close()


def test_export_contract(aloam, orc):
    """size query; a too-small buffer returns ERR_CAPACITY with the size, writes nothing and changes no state; device and pinned
    output equal host output; ERR_STATE before the mapper exists / before the first frame; 0 points after a reset"""
    import torch
    mk = lambda: aloam.Aloam(n_scans=16, max_points=20000, max_map_points=200000, line_res=0.4, plane_res=0.8)
    a, b = mk(), mk()
    assert export_raw(aloam, a, aloam.MAP_ALL, 0, 0)[0] == ERR_STATE
    with pytest.raises(aloam.AloamError) as e:
        a.mapper_associate_to_map(np.zeros((3, 4), np.float32))
    assert e.value.code == ERR_STATE
    a.mapper_reset()
    assert a.mapper_export(aloam.MAP_ALL).shape == (0, 4) and a.mapper_export(aloam.MAP_SURROUND).shape == (0, 4)
    with pytest.raises(aloam.AloamError) as e:
        a.mapper_associate_to_map(np.zeros((3, 4), np.float32))
    assert e.value.code == ERR_STATE
    b.mapper_reset()
    frames = list(scroll_frames())
    for corner, surf, full, q, t in frames[:4]:
        for ctx in (a, b):
            ctx.mapper_step(corner, surf, q, t)
    for region in (aloam.MAP_SURROUND, aloam.MAP_ALL):
        host = a.mapper_export(region)
        n = host.shape[0]
        assert n > 0 and export_raw(aloam, a, region, 0, 0) == (0, n)
        sentinel = np.full((n + 8, 4), -7.25, np.float32)
        assert export_raw(aloam, a, region, sentinel.ctypes.data, n - 1) == (ERR_CAPACITY, n)
        assert (sentinel == -7.25).all()
        dev = torch.full((n + 8, 4), -7.25, dtype=torch.float32, device="cuda")
        assert a.mapper_export_ptr(region, dev.data_ptr(), n + 8) == n
        d = dev.cpu().numpy()
        assert np.array_equal(d[:n], host) and (d[n:] == -7.25).all()
        pinned = torch.full((n, 4), -7.25, dtype=torch.float32).pin_memory()
        assert a.mapper_export_ptr(region, pinned.data_ptr(), n) == n
        assert np.array_equal(pinned.numpy(), host)
    # the rejected and the successful exports changed nothing: the next frame equals the control context's
    corner, surf, full, q, t = frames[4]
    pa = a.mapper_step(corner, surf, q, t)[:2]
    pb = b.mapper_step(corner, surf, q, t)[:2]
    assert all(np.array_equal(x, y) for x, y in zip(pa, pb))
    assert np.array_equal(a.mapper_export(aloam.MAP_ALL), b.mapper_export(aloam.MAP_ALL))
    assert np.array_equal(a.mapper_associate_to_map(full), b.mapper_associate_to_map(full))
    a.mapper_reset()
    assert a.mapper_export(aloam.MAP_ALL).shape == (0, 4)
    a.close(); b.close()


def _per_scan(aloam, raws, maxn):
    """scan_to_pose -> extract_features -> mapper_step -> mapper_associate_to_map, one scan at a time"""
    c = aloam.Aloam(n_scans=16, max_points=maxn + 1024, max_map_points=400000)
    c.mapper_reset()
    odom, mapped, regs = [], [], []
    for raw in raws:
        q, t, _ = c.scan_to_pose(raw)
        f = c.extract_features(raw)
        mq, mt, _ = c.mapper_step(f["less_sharp"], f["less_flat"], q, t)
        odom.append(np.concatenate([q, t])); mapped.append(np.concatenate([mq, mt]))
        regs.append(c.mapper_associate_to_map(f["full"]))
    return c, np.array(odom), np.array(mapped), regs


def test_stream_registered_equals_per_scan_path(aloam, scans):
    """6 VLP-16 scans in two calls (device raws into a device buffer, pinned host raws into a pinned host buffer): poses equal
    scan_stream_mapped, every registered cloud equals the per-scan path, offsets are the prefix sums of the cloud sizes, and the
    cube store ends up the same"""
    import torch
    raws = [scans("VLP-16", k, n_az=900) for k in range(6)]
    maxn = max(r.shape[0] for r in raws)
    ref, odom, mapped, regs = _per_scan(aloam, raws, maxn)
    plain = aloam.Aloam(n_scans=16, max_points=maxn + 1024, max_map_points=400000)
    o_plain, m_plain = plain.scan_stream_mapped([r.ctypes.data for r in raws], [r.shape[0] for r in raws], False)
    plain.close()
    c = aloam.Aloam(n_scans=16, max_points=maxn + 1024, max_map_points=400000)
    cap = sum(r.shape[0] for r in raws)
    dev_raws = [torch.from_numpy(r).cuda() for r in raws[:3]]
    dev_out = torch.full((cap, 4), -7.25, dtype=torch.float32, device="cuda")
    o1, m1, off1, st1 = c.scan_stream_mapped_registered([d.data_ptr() for d in dev_raws], [r.shape[0] for r in raws[:3]], True,
                                                         dev_out.data_ptr(), cap)
    pin_raws = [torch.from_numpy(r).pin_memory() for r in raws[3:]]
    pin_out = torch.full((cap, 4), -7.25, dtype=torch.float32).pin_memory()
    o2, m2, off2, st2 = c.scan_stream_mapped_registered([p.data_ptr() for p in pin_raws], [r.shape[0] for r in raws[3:]], False,
                                                         pin_out.data_ptr(), cap)
    assert not (st1["flags"] | st2["flags"]) & aloam.FLAG_OUTPUT_TRUNCATED
    assert np.array_equal(np.concatenate([o1, o2]), o_plain) and np.array_equal(np.concatenate([m1, m2]), m_plain)
    assert np.array_equal(o_plain, odom) and np.array_equal(m_plain, mapped)
    sizes = [r.shape[0] for r in regs]
    assert off1.tolist() == np.concatenate([[0], np.cumsum(sizes[:3])]).tolist()
    assert off2.tolist() == np.concatenate([[0], np.cumsum(sizes[3:])]).tolist()
    d, h = dev_out.cpu().numpy(), pin_out.numpy()
    for k in range(6):
        buf, off, j = (d, off1, k) if k < 3 else (h, off2, k - 3)
        assert np.array_equal(buf[off[j]:off[j + 1]], regs[k]), k
    assert (d[off1[-1]:] == -7.25).all() and (h[off2[-1]:] == -7.25).all()
    assert np.array_equal(c.mapper_export(aloam.MAP_ALL), ref.mapper_export(aloam.MAP_ALL))
    c.close(); ref.close()


def test_stream_registered_truncation_and_rejected_buffer(aloam, scans):
    """a buffer that holds three scans: scans 0-2 are written, nothing beyond, the flag is set and the poses are complete; a
    pageable buffer is rejected before any work, and the next valid call continues the trajectory as if it had never been made"""
    import torch
    raws = [scans("VLP-16", k, n_az=900) for k in range(8)]
    maxn = max(r.shape[0] for r in raws)
    ref, odom, mapped, regs = _per_scan(aloam, raws[:6], maxn)
    ref.close()
    ctrl = aloam.Aloam(n_scans=16, max_points=maxn + 1024, max_map_points=400000)
    o_ctrl, m_ctrl = ctrl.scan_stream_mapped([r.ctypes.data for r in raws], [r.shape[0] for r in raws], False)
    ctrl.close()
    c = aloam.Aloam(n_scans=16, max_points=maxn + 1024, max_map_points=400000)
    cap = sum(r.shape[0] for r in regs[:3])
    out = torch.full((cap + 4096, 4), -7.25, dtype=torch.float32, device="cuda")
    o, m, off, st = c.scan_stream_mapped_registered([r.ctypes.data for r in raws[:6]], [r.shape[0] for r in raws[:6]], False,
                                                    out.data_ptr(), cap)
    assert st["flags"] & aloam.FLAG_OUTPUT_TRUNCATED
    assert np.array_equal(o, odom) and np.array_equal(m, mapped)
    assert off[3] == cap and off[-1] > cap
    got = out.cpu().numpy()
    assert np.array_equal(got[:cap], np.concatenate(regs[:3])) and (got[cap:] == -7.25).all()
    pageable = np.zeros((100000, 4), np.float32)
    with pytest.raises(aloam.AloamError) as e:
        c.scan_stream_mapped_registered([r.ctypes.data for r in raws[6:]], [r.shape[0] for r in raws[6:]], False, pageable.ctypes.data, 100000)
    assert e.value.code == ERR_INVALID_ARG
    o, m, off, st = c.scan_stream_mapped_registered([r.ctypes.data for r in raws[6:]], [r.shape[0] for r in raws[6:]], False,
                                                    out.data_ptr(), cap + 4096)
    assert np.array_equal(o, o_ctrl[6:]) and np.array_equal(m, m_ctrl[6:])
    c.close()
