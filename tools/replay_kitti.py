#!/usr/bin/env python
"""Replay a directory of KITTI-format velodyne scans (NNNNNN.bin, float32 x,y,z,intensity -- kittiHelper.cpp:25-35)
through the device pipeline and write one lidar-odometry pose per scan.

    python tools/replay_kitti.py /data/kitti/sequences/00/velodyne --out poses.txt [--gt /data/kitti/poses/00.txt]

Output: KITTI pose lines (row-major 3x4, camera frame, first pose = identity) so the usual KITTI evaluation tools
apply.  With --gt the translation drift against the ground truth (read the way kittiHelper.cpp:97-113 reads it) is
printed.  The scans go through aloam_scan_stream in chunks: extraction, index build and odometry of consecutive scans
overlap on the device and only the poses come back.

With --map OUT.bin the scans go through aloam_scan_stream_mapped instead (odometry and scan-to-map on the device) and the
final map -- all cubes of the store, what laserMapping.cpp:823-836 publishes as /laser_cloud_map -- is written to OUT.bin
in the KITTI layout.  With --registered DIR as well, every scan's full-resolution cloud registered with its refined pose
(/velodyne_cloud_registered, :838-848) is written to DIR/NNNNNN.bin.  The pose file keeps the odometry poses."""
import argparse
import importlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def replay(scan_paths, n_scans=64, chunk=256, minimum_range=None, device=0, map_out=None, registered_dir=None, max_map_points=600000):
    """-> (n, 7) world poses (q xyzw, t) in the lidar frame of the first scan.  map_out: also run the scan-to-map stage and
    write the final map there; registered_dir: and every scan's registered full cloud"""
    import torch
    pkg = importlib.import_module("a-loam_b200")
    io = importlib.import_module("a-loam_b200.io")
    sizes = [os.path.getsize(p) // 16 for p in scan_paths]
    kw = {} if minimum_range is None else {"minimum_range": minimum_range}
    if map_out:
        kw["max_map_points"] = max_map_points
    ctx = pkg.Aloam(n_scans=n_scans, device=device, max_points=max(sizes) + 1024, **kw)
    poses = []
    for c0 in range(0, len(scan_paths), chunk):
        paths = scan_paths[c0:c0 + chunk]
        cnt = sizes[c0:c0 + chunk]
        host = torch.zeros((len(paths), max(cnt), 4), dtype=torch.float32).pin_memory()
        for i, p in enumerate(paths):
            host[i, :cnt[i]] = torch.from_numpy(io.read_kitti_bin(p))
        ptrs = [host[i].data_ptr() for i in range(len(paths))]
        if not map_out:
            p, _ = ctx.scan_stream(ptrs, cnt, False)
        elif not registered_dir:
            p, _ = ctx.scan_stream_mapped(ptrs, cnt, False)
        else:
            out = torch.empty((sum(cnt), 4), dtype=torch.float32).pin_memory()   # a full cloud is never larger than its scan
            p, _, off, _ = ctx.scan_stream_mapped_registered(ptrs, cnt, False, out.data_ptr(), out.shape[0])
            reg = out.numpy()
            for i, path in enumerate(paths):
                io.write_kitti_bin(os.path.join(registered_dir, os.path.basename(path)), reg[off[i]:off[i + 1]])
        poses.append(p)
    if map_out:
        io.write_kitti_bin(map_out, ctx.mapper_export(pkg.MAP_ALL))
    ctx.close()
    return np.concatenate(poses)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("velodyne_dir")
    ap.add_argument("--out", default="poses_aloam_b200.txt")
    ap.add_argument("--gt", default=None, help="KITTI poses file of the sequence")
    ap.add_argument("--beams", type=int, default=64)
    ap.add_argument("--limit", type=int, default=0)
    ap.add_argument("--map", default=None, metavar="OUT.bin", help="run the scan-to-map stage too and write the final map here")
    ap.add_argument("--registered", default=None, metavar="DIR", help="with --map: write every scan's registered full cloud to DIR")
    args = ap.parse_args()
    if args.registered and not args.map:
        sys.exit("--registered needs --map")
    if args.registered:
        os.makedirs(args.registered, exist_ok=True)
    io = importlib.import_module("a-loam_b200.io")
    paths = sorted(os.path.join(args.velodyne_dir, f) for f in os.listdir(args.velodyne_dir) if f.endswith(".bin"))
    if args.limit:
        paths = paths[:args.limit]
    if not paths:
        sys.exit("no .bin scans in " + args.velodyne_dir)
    poses = replay(paths, n_scans=args.beams, map_out=args.map, registered_dir=args.registered)
    with open(args.out, "w") as f:
        for p in poses:
            f.write(" ".join("%.9e" % v for v in io.lidar_pose_to_kitti(p[:4], p[4:]).reshape(-1)) + "\n")
    print("%d poses -> %s" % (len(poses), args.out))
    if args.map:
        print("map -> %s" % args.map)
    if args.gt:
        lines = [l for l in open(args.gt).read().splitlines() if l.strip()][:len(poses)]
        gt = [io.kitti_pose_to_lidar(io.parse_kitti_pose(l)) for l in lines]
        q0, t0 = gt[0]
        # express the ground truth relative to its first pose (our world frame is the first scan's lidar frame)
        R0 = io.lidar_pose_to_kitti(q0, np.zeros(3))[:, :3]
        err = [np.linalg.norm(poses[i][4:] - (io.lidar_pose_to_kitti(*gt[i])[:, 3] - io.lidar_pose_to_kitti(q0, t0)[:, 3])) for i in range(len(gt))]
        print("translation difference to ground truth: median %.3f m, final %.3f m over %d scans" % (np.median(err), err[-1], len(err)))


if __name__ == "__main__":
    main()
