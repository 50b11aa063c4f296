/* aloam_b200.h -- C ABI of the B200-native A-LOAM per-scan registration hot path.
 *
 * The reference (HKUST-Aerial-Robotics/A-LOAM) has NO library / plugin / FFI boundary: the hot path is inline
 * code in three ROS node `main`s.  This header creates the boundary at exactly the seam between the node shells
 * (topic I/O, queues, publishing -- unchanged, stay in the ROS nodes) and the per-scan algorithms (replaced).
 * Each entry point names the reference code it replaces (file:line into the reference tree).  INTEGRATION.md
 * shows the call a maintainer adds at each site.
 *
 * Conventions
 *   - plain C99 types, no exceptions cross the boundary; every call returns 0 (ALOAM_OK) or a negative error.
 *   - points are 4 floats x,y,z,intensity (pcl::PointXYZI's meaningful fields, include/aloam_velodyne/common.h:43);
 *     `stride_floats` = 4 for packed arrays, 8 for PCL's 32-byte PointXYZI, so a pcl::PointCloud's storage can be
 *     passed without repacking.  intensity = scanID + 0.1*relTime exactly as scanRegistration.cpp:239.
 *   - quaternions are Eigen/Ceres parameter order x,y,z,w; poses are caller-owned in/out arrays exactly like
 *     para_q/para_t (laserOdometry.cpp:97-98) and parameters[7] (laserMapping.cpp:110).
 *   - inputs are borrowed for the duration of the call; output views point into ctx-owned pinned host memory and
 *     stay valid until the next call on the same ctx.  One ctx per calling thread (each reference node calls from
 *     exactly one thread); a ctx is not thread-safe; calls are synchronous.
 *   - soft conditions mirror the reference and are NOT errors: < 10 correspondences (laserOdometry.cpp:488-491)
 *     sets ALOAM_FLAG_FEW_CORRESPONDENCES; a thin map (corner <= 10 or surf <= 50, laserMapping.cpp:554,730-733)
 *     skips the optimisation, leaves the pose unchanged and sets ALOAM_FLAG_MAP_TOO_THIN.
 *   - there is NO CPU fallback: if the CUDA device or kernels are unavailable aloam_create fails.
 */
#ifndef ALOAM_B200_H_
#define ALOAM_B200_H_

#ifdef __cplusplus
extern "C" {
#endif

#define ALOAM_OK 0
#define ALOAM_ERR_INVALID_ARG (-1)
#define ALOAM_ERR_UNSUPPORTED_SCANS (-2) /* scanRegistration.cpp:472-476: only 16, 32 or 64 scan lines */
#define ALOAM_ERR_EMPTY_CLOUD (-3)       /* no point survives the NaN / minimum-range filter */
#define ALOAM_ERR_CAPACITY (-4)          /* more points than the ctx was created for */
#define ALOAM_ERR_CUDA (-5)
#define ALOAM_ERR_NO_DEVICE (-6)
#define ALOAM_ERR_RING_TOO_LARGE (-7)    /* a single ring holds more than ALOAM_MAX_RING_POINTS returns */
#define ALOAM_ERR_NOT_RING_MAJOR (-8)    /* "last" cloud not in ascending ring order (laserOdometry.cpp:312-361 relies on it) */
#define ALOAM_ERR_STATE (-9)             /* call sequence error, e.g. register before set_last */
#define ALOAM_ERR_COMM (-10)

#define ALOAM_MAX_RING_POINTS 4096
#define ALOAM_MAX_BATCH 16

#define ALOAM_FLAG_FEW_CORRESPONDENCES 1
#define ALOAM_FLAG_MAP_TOO_THIN 2
#define ALOAM_FLAG_INITIALISED_ONLY 4 /* first frame: laserOdometry.cpp:267-271 */
#define ALOAM_FLAG_CUBE_OVERFLOW 8    /* map cube store: a cube slab (16 k corner / 64 k surf points) or the slab pool was full; the overflow was dropped */
#define ALOAM_FLAG_OUTPUT_TRUNCATED 16 /* aloam_scan_stream_mapped_registered: the registered clouds did not all fit the caller's buffer */

#define ALOAM_MAP_SURROUND 0 /* aloam_mapper_export: the valid cubes of the last frame, laserCloudSurroundInd (laserMapping.cpp:806-814) */
#define ALOAM_MAP_ALL 1      /* aloam_mapper_export: all 21 x 21 x 11 cubes in index order (laserMapping.cpp:823-830) */

typedef struct aloam_ctx aloam_ctx;

/* The constants of the hot path (SURVEY.md section 5 "config / flags").  aloam_default_config fills the values
 * of launch/aloam_velodyne_{VLP_16,HDL_32,HDL_64}.launch:3-13 for n_scans = 16 / 32 / 64. */
typedef struct aloam_config {
  int n_scans;           /* scan_line                       scanRegistration.cpp:466 */
  float minimum_range;   /* minimum_range                   scanRegistration.cpp:468 */
  float line_res;        /* mapping_line_resolution         laserMapping.cpp:902-906 */
  float plane_res;       /* mapping_plane_resolution */
  int outer_iters;       /* 2   laserOdometry.cpp:278, laserMapping.cpp:562 */
  int inner_iters;       /* 4   options.max_num_iterations, laserOdometry.cpp:496 */
  double huber;          /* 0.1 HuberLoss, laserOdometry.cpp:284 */
  double dist_sq_thresh; /* 25  DISTANCE_SQ_THRESHOLD, laserOdometry.cpp:65 */
  double nearby_scan;    /* 2.5 NEARBY_SCAN, laserOdometry.cpp:66 */
  int device;            /* CUDA device ordinal */
  int max_points;        /* capacity of one raw scan (reference: 400000 static arrays, scanRegistration.cpp:66-69) */
  int max_map_points;    /* capacity of the uploaded submap, per cloud type (0 = mapping not used) */
  int max_batch;         /* trajectories a context can advance in lockstep (aloam_scan_stream_batch); 1..ALOAM_MAX_BATCH, default 1 */
  int distortion;        /* 0 (reference build) or 1: #define DISTORTION of laserOdometry.cpp:59 -- per-point interpolation ratio
                            s = (intensity - int(intensity)) / SCAN_PERIOD in TransformToStart (:113-118) and in the
                            residual blocks (:376-379, 470-473; slerp inside the functors, lidarFactor.hpp:27-33) */
  int max_ring_points;   /* capacity of one scan ring, multiple of 32, <= ALOAM_MAX_RING_POINTS (default).  Smaller rings take
                            less shared memory per ring CTA, so more of them are resident per SM (batched streams) */
} aloam_config;

typedef struct aloam_cloud_view {
  const float* data;
  int n;
  int stride_floats; /* 4 or 8 */
} aloam_cloud_view;

typedef struct aloam_stats {
  int n_corner_corr, n_plane_corr; /* residual blocks built in the LAST outer iteration */
  int lm_iters;                    /* sum of trust-region iterations over the outer iterations */
  int accepted_steps;
  int flags;
  int termination[4];              /* per outer iteration: 0 max-iters 1 gradient 2 parameter 3 function 4 empty 5 failure */
  double init_cost, final_cost;    /* of the last outer iteration */
  float ms_total;                  /* device time of the call, CUDA events */
} aloam_stats;

void aloam_default_config(aloam_config* cfg, int n_scans);
int aloam_create(const aloam_config* cfg, aloam_ctx** out);
int aloam_destroy(aloam_ctx* ctx);
const char* aloam_strerror(int code);

/* ---- feature extraction: replaces scanRegistration.cpp:129-408 (body of laserCloudHandler between fromROSMsg
 * and the five toROSMsg/publish calls at :413-441).  raw = the PointXYZ cloud in arrival order. */
int aloam_extract_features(aloam_ctx* ctx, aloam_cloud_view raw, aloam_cloud_view* full,
                           aloam_cloud_view* sharp, aloam_cloud_view* less_sharp, aloam_cloud_view* flat,
                           aloam_cloud_view* less_flat);

/* ---- scan-to-scan odometry.
 * aloam_odometry_set_last replaces laserOdometry.cpp:554-568 (swap in the less-sharp / less-flat clouds and
 * rebuild kdtreeCornerLast / kdtreeSurfLast).  aloam_odometry_register replaces :274-502 (the two
 * association + ceres::Solve rounds); q_last_curr/t_last_curr are para_q/para_t, warm-started by the caller. */
int aloam_odometry_set_last(aloam_ctx* ctx, aloam_cloud_view corner_last, aloam_cloud_view surf_last);
int aloam_odometry_register(aloam_ctx* ctx, aloam_cloud_view sharp, aloam_cloud_view flat,
                            double q_last_curr[4], double t_last_curr[3], aloam_stats* stats);

/* ---- scan-to-map refinement.
 * aloam_map_upload replaces laserMapping.cpp:531-539 + :558-559 (the gathered 5x5x3-cube submap and the two
 * kd-tree builds).  aloam_mapping_register replaces :554-729; the stacks are the voxel-filtered current
 * corner / surf clouds of :542-550 (use aloam_voxel_filter for those), q_t_w_curr = parameters[7].
 * Input views of aloam_map_upload / aloam_odometry_* / aloam_mapping_* may point to host memory (pageable or pinned)
 * or to device memory: the copy kind is inferred from the address (unified virtual addressing). */
int aloam_map_upload(aloam_ctx* ctx, aloam_cloud_view corner_map, aloam_cloud_view surf_map);
int aloam_mapping_register(aloam_ctx* ctx, aloam_cloud_view corner_stack, aloam_cloud_view surf_stack,
                           double q_t_w_curr[7], aloam_stats* stats);
/* pcl::VoxelGrid<PointXYZI> with a cubic leaf: laserMapping.cpp:543-549 (scan stacks), scanRegistration.cpp:401-405 */
int aloam_voxel_filter(aloam_ctx* ctx, aloam_cloud_view in, float leaf, aloam_cloud_view* out);

/* ---- fused, device-resident pipeline (SURVEY.md 8f-2): one raw scan in, world pose out; the feature clouds
 * and the "last" clouds never leave the GPU.  Equivalent to extract_features -> odometry_register ->
 * pose integration (laserOdometry.cpp:504-505) -> odometry_set_last, with the reference's warm start.
 * First call only initialises (laserOdometry.cpp:267-271).  q_w_curr/t_w_curr are outputs. */
int aloam_scan_to_pose(aloam_ctx* ctx, aloam_cloud_view raw, double q_w_curr[4], double t_w_curr[3],
                       aloam_stats* stats);
/* same, raw scan already in device memory (4-float packed points); used for HBM-resident measurements */
int aloam_scan_to_pose_device(aloam_ctx* ctx, const float* d_raw_xyzi, int n, double q_w_curr[4],
                              double t_w_curr[3], aloam_stats* stats);
/* pipelined form for a sequence of scans: upload, ring binning, per-ring feature extraction, compaction + index build
 * and association + LM of consecutive scans overlap on five CUDA streams (the overlap the reference gets from its three
 * ROS processes); results identical to calling aloam_scan_to_pose once per scan, in any interleaving with it.  device_resident != 0: raws[k].data are device pointers (stride 4).
 * poses: n_scans x 7 doubles (q_w xyzw, t_w). */
int aloam_scan_stream(aloam_ctx* ctx, const aloam_cloud_view* raws, int n_scans, int device_resident, double* poses,
                      aloam_stats* stats_last);
/* batched form (BASELINE configs[4], SURVEY.md 8b "aloam_*_batch"): `batch` independent trajectories advance in lockstep and
 * SHARE every kernel launch (ring CTAs of all trajectories in one grid, one LM cluster per trajectory, ...), so one
 * context and one host thread fill the GPU.  raws: n_scans x batch views, scan-major (raws[k * batch + b] = scan k of
 * trajectory b); poses: n_scans x batch x 7 doubles in the same order; stats_last: `batch` entries or NULL.  Every
 * trajectory keeps the reference's warm-start chain (laserOdometry.cpp:97-98,504-505) and its result is bit-identical to
 * running it alone through aloam_scan_stream.  batch <= cfg.max_batch; all trajectories of a context share the frame
 * counter (the first scan of a fresh / reset context only initialises, laserOdometry.cpp:267-271). */
int aloam_scan_stream_batch(aloam_ctx* ctx, const aloam_cloud_view* raws, int n_scans, int batch, int device_resident,
                            double* poses, aloam_stats* stats_last);
/* the whole pipeline of the three reference nodes in one call (SURVEY.md 8 f-2): as aloam_scan_stream, and every scan's
 * less-sharp / less-flat clouds and odometry pose are handed ON THE DEVICE to the scan-to-map stage (one aloam_mapper_step
 * per scan, on its own stream, overlapping the odometry of the following scans) -- what the reference ships over
 * /laser_cloud_corner_last, /laser_cloud_surf_last and /laser_odom_to_init (laserOdometry.cpp:570-591 ->
 * laserMapping.cpp:278-288, 142-152).  odom_poses / map_poses: n_scans x 7 doubles (q xyzw, t): laser_odom_to_init and
 * aft_mapped_to_init.  Identical to calling aloam_scan_to_pose + aloam_mapper_step per scan.  Needs cfg.max_map_points > 0.
 * After aloam_comm_init (every rank fed the same scans) the scan-to-map stage is sharded: each rank keeps the whole cube store,
 * indexes and searches only its x-slabs of the gathered submap, and the ranks meet in the all-reduce of the normal equations;
 * all ranks return the same poses (equal to a single-GPU run to rounding of the summation order). */
int aloam_scan_stream_mapped(aloam_ctx* ctx, const aloam_cloud_view* raws, int n_scans, int device_resident, double* odom_poses,
                             double* map_poses, aloam_stats* stats_last);
int aloam_reset_odometry(aloam_ctx* ctx); /* forget pose, warm start and "last" clouds (all trajectories) */

/* TransformToEnd of laserOdometry.cpp:133-148 on a whole cloud: undistort every point to the sweep start with its own
 * interpolation ratio, then carry it to the sweep end with (q_last_curr, t_last_curr); the intensity keeps only the scan id.
 * (Dead code in the reference -- its call sites sit under `if (0)`, :533-552 -- provided because the DISTORTION build
 * is where it belongs.)  distortion != 0 uses the per-point ratio, 0 uses s = 1.  out: view into ctx-owned pinned memory. */
int aloam_transform_to_end(aloam_ctx* ctx, aloam_cloud_view in, const double q_last_curr[4], const double t_last_curr[3],
                           int distortion, aloam_cloud_view* out);

/* ---- fine-grained entry points (tests; or to keep Ceres in the loop) */
/* exact k-NN replacing pcl::KdTreeFLANN::nearestKSearch: which = 0 corner_last, 1 surf_last (laserOdometry.cpp:302,390),
 * 2 corner_map, 3 surf_map (laserMapping.cpp:582,648).  idx/sqdist: queries.n x k, ascending (dist, index). */
int aloam_knn(aloam_ctx* ctx, int which, aloam_cloud_view queries, int k, int* idx, float* sqdist);
/* association of laserOdometry.cpp:299-483 at pose (q,t): corner_corr n_sharp x 3 (a,b,valid), plane_corr n_flat x 4 (a,b,c,valid) */
int aloam_odometry_associate(aloam_ctx* ctx, aloam_cloud_view sharp, aloam_cloud_view flat, const double q[4],
                             const double t[3], int* corner_corr, int* plane_corr);
/* residual blocks are 11 doubles [type(0 edge,1 plane,2 plane-norm), cp(3), a(3), b(3), s]; for type 1 b is the unit
 * normal LidarPlaneFactor precomputes (lidarFactor.hpp:64-65), for type 2 a is the unit normal and s = negative_OA_dot_norm.
 * For types 0 and 1 s is the functor's interpolation ratio (1.0 in the reference build; any value in [0, 1] is evaluated with the
 * slerp of lidarFactor.hpp:27-33 and its analytic Jacobian).  include/lidarFactor.hpp packs these records (PackBlock).
 * JtJ (6x6 row-major), Jtr (6) in the tangent [dtheta(3), dt(3)] with Huber(0.1) applied, cost = sum 0.5 rho. */
int aloam_normal_equations(aloam_ctx* ctx, const double* blocks, int n_blocks, const double x[7], double JtJ[36],
                           double Jtr[6], double* cost);
/* Ceres-equivalent trust-region solve on the device (replaces ceres::Solve at laserOdometry.cpp:494-499,
 * laserMapping.cpp:712-720).  trace: up to max_trace rows of 8 doubles, may be NULL. */
int aloam_solve(aloam_ctx* ctx, const double* blocks, int n_blocks, double x[7], double summary7[7], double* trace,
                int max_trace, int* trace_rows);
/* last extract_features call: per-point curvature (scanRegistration.cpp:262), label (:303,309,355), ring start/end */
int aloam_debug_features(aloam_ctx* ctx, float* curvature, int* label, int* scan_start, int* scan_end);

/* association + fits of laserMapping.cpp:577-687 at pose x (tests): fits = (n_corner + n_surf) x 14 doubles
 * [query, type (-1 rejected, 0 edge, 2 plane-norm), p0(3), p1(3), d, nn(5)], corner rows first */
int aloam_mapping_associate(aloam_ctx* ctx, aloam_cloud_view corner_stack, aloam_cloud_view surf_stack,
                            const double x[7], double* fits);

/* ---- map cube store + the mapping loop around it (laserMapping.cpp:74-108,142-163,309-550,736-801; SURVEY.md 8 f-1).
 * The 21 x 21 x 11 ring buffer of 50 m cubes lives in device memory: a pool of fixed-capacity slabs (1024 per cloud type,
 * 16 k corner / 64 k surf points each, 1.3 GB, created on first use) handed to cubes on their first insertion.
 * aloam_mapper_step is one frame of alaserMapping's process(), entirely on the device with one synchronisation at the end:
 * pose hand-off from the odometry (transformAssociateToMap), ring-buffer shift, gather of the <= 75 valid cubes (device
 * to device), stack filters at line_res / plane_res, optimisation against the gathered submap (skipped while it is thinner
 * than 10 corner / 50 surf points), transformUpdate, insertion of the registered stacks and per-cube VoxelGrid of the valid
 * cubes.  corner_last / surf_last are the less-sharp / less-flat clouds of the scan (what /laser_cloud_corner_last and
 * /laser_cloud_surf_last carry); the odometry pose is q_wodom_curr / t_wodom_curr; the refined pose is returned.
 * The call never fails half-way: a full cube slab, an exhausted pool or a submap beyond cfg.max_map_points drop the
 * overflow and set ALOAM_FLAG_CUBE_OVERFLOW in stats->flags; argument errors are reported before any state changes.
 * cfg.max_map_points must be > 0. */
int aloam_mapper_reset(aloam_ctx* ctx);
int aloam_mapper_step(aloam_ctx* ctx, aloam_cloud_view corner_last, aloam_cloud_view surf_last,
                      const double q_wodom_curr[4], const double t_wodom_curr[3], double q_w_curr[4], double t_w_curr[3],
                      aloam_stats* stats);
/* inspection (tests): ring-buffer centre offsets, valid cube indices of the last step (i + 21 j + 441 k), the map-to-
 * odometry transform, total stored points per type; and the points of one cube (which: 0 corner, 1 surf; host view,
 * valid until the next call) */
int aloam_mapper_debug_state(aloam_ctx* ctx, int centre[3], int* n_valid, int valid[125], double q_wmap_wodom[4],
                             double t_wmap_wodom[3], long long totals[2]);
int aloam_mapper_debug_cube(aloam_ctx* ctx, int which, int cube_index, aloam_cloud_view* out);

/* ---- map outputs: the three clouds alaserMapping publishes at the end of a frame (laserMapping.cpp:803-848).  Outputs are
 * packed stride-4 points in caller-owned memory (a map has no fixed upper size, so there is no ctx-owned output view).
 * aloam_mapper_export: /laser_cloud_surround (region ALOAM_MAP_SURROUND, published by the reference every 5th frame) or
 * /laser_cloud_map (ALOAM_MAP_ALL, every 20th frame) -- per cube the corner points, then the surf points, in the reference's
 * order; the store as it is after the last frame's insertion and per-cube VoxelGrid.  Publish cadence is the caller's choice.
 * out == NULL with capacity_points == 0 is a size query.  A result larger than capacity_points returns ALOAM_ERR_CAPACITY with
 * the required size in *n_points and writes nothing.  out may be host (pageable or pinned) or device memory.
 * ALOAM_ERR_STATE before the mapper exists; 0 points after aloam_mapper_reset.
 * aloam_mapper_associate_to_map: /velodyne_cloud_registered -- pointAssociateToMap (:154-163) of a whole cloud (the full-
 * resolution /velodyne_cloud_3) with the refined pose of the last frame; the intensity is kept.  in: stride 4 or 8, host or
 * device, n <= cfg.max_points; out: in.n points, host or device.  ALOAM_ERR_STATE before the first frame since a reset.
 * aloam_scan_stream_mapped_registered: aloam_scan_stream_mapped, and every scan's ring-major full cloud (what /velodyne_cloud_2
 * and, unchanged, /velodyne_cloud_3 carry) registered with the scan's refined pose and written to registered[offsets[k] ...].
 * offsets (n_scans + 1) are the prefix sums of the cloud sizes and are always filled.  Scans that end beyond capacity_points
 * are not written (the buffer holds a prefix of whole scans) and ALOAM_FLAG_OUTPUT_TRUNCATED is set in stats_last->flags;
 * the poses are complete either way.  registered must be device memory or page-locked host memory (written by a kernel);
 * pageable memory is ALOAM_ERR_INVALID_ARG, reported before any work is issued. */
int aloam_mapper_export(aloam_ctx* ctx, int region, float* out, long long capacity_points, long long* n_points);
int aloam_mapper_associate_to_map(aloam_ctx* ctx, aloam_cloud_view in, float* out);
int aloam_scan_stream_mapped_registered(aloam_ctx* ctx, const aloam_cloud_view* raws, int n_scans, int device_resident,
                                        double* odom_poses, double* map_poses, float* registered, long long capacity_points,
                                        long long* offsets, aloam_stats* stats_last);

/* ---- multi-GPU scan-to-map (one process per GPU).  Rank 0 creates the 128-byte id and ships it to the others;
 * after aloam_comm_init each rank uploads only ITS shard of the submap (x-slabs of aloam_shard_slab_cells() cells of
 * 1.00001 m, owner = slab mod world, plus one cell of halo) and aloam_mapping_register fits only the stack points
 * whose cell the rank owns; the ranks meet in one ncclAllReduce of the 6x6 / 6x1 normal equations per evaluation and
 * return the identical pose. */
int aloam_comm_unique_id(char out128[128]);
int aloam_comm_init(aloam_ctx* ctx, int rank, int world, const char id128[128]);
int aloam_shard_slab_cells(void);
/* as aloam_map_upload, for a rank that holds the WHOLE submap (host or device memory): the rank's shard -- its x-slabs plus the
 * one-cell halo -- is cut out on the device (stable compaction), then indexed.  cfg.max_map_points must hold the shard. */
int aloam_map_upload_sharded(aloam_ctx* ctx, aloam_cloud_view corner_map, aloam_cloud_view surf_map);
/* 1 when the ranks exchange the normal equations through NVLink peer memory INSIDE the LM kernel (one launch per solve; CUDA IPC
 * mailboxes set up by aloam_comm_init), 0 when they use ncclAllReduce between per-evaluation kernels (no peer access, or the
 * environment variable ALOAM_NO_PEER is set -- kept for A/B measurements). */
int aloam_comm_uses_peer_memory(aloam_ctx* ctx);

/* ---- measurement hooks (bench.py): per-kernel CUDA-event timing on the ctx stream, and a launch counter */
int aloam_profile_enable(aloam_ctx* ctx, int on);
int aloam_profile_read(aloam_ctx* ctx, double* ms_sum, long long* count, const char** names, int capacity);
long long aloam_launch_count(aloam_ctx* ctx);
int aloam_debug_lm_cycles(aloam_ctx* ctx, long long* out, int outer_iters); /* SM cycles: [solve, evaluation passes] per outer iteration */

#ifdef __cplusplus
}
#endif
#endif /* ALOAM_B200_H_ */
