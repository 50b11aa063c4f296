// Internal: the context object behind the C ABI and the helpers shared by capi.cu, mapping.cu, cubemap.cu, comm.cu.
#pragma once
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>
#include "../../include/aloam_b200.h"
#include "kernels.h"

using namespace aloam;

namespace {

constexpr int kMaxSharpPerRing = 12, kMaxLessSharpPerRing = 120, kMaxFlatPerRing = 24;
constexpr int kFusedSharpSlots = 64 * kMaxSharpPerRing;  // 768
constexpr int kFusedFlatSlots = 64 * kMaxFlatPerRing;    // 1536
constexpr int kMaxQueries = ALOAM_MAX_QUERIES;         // API-path capacity for sharp / flat query clouds
constexpr int kProfSlots = 192;                        // kernel launches timed per profile window (one API call)
constexpr int kFeatSlots = 4;                          // feature-set ring of the fused / stream paths
constexpr int kApiLast = kFeatSlots, kApiCur = kFeatSlots + 1;   // feature sets of the per-stage entry points (set_last / extract, register): never the ring's
constexpr int kMaxStreamScans = 4096;                  // scans x lanes per aloam_scan_stream(_batch) call

struct FeatBuf {
  Pt4 *sharp = nullptr, *less_sharp = nullptr, *flat = nullptr, *less_flat = nullptr;
  int* counts = nullptr;           // [4] n_sharp, n_less_sharp, n_flat, n_less_flat (device)
  int *rs_ls = nullptr, *rs_lf = nullptr;  // ring_start tables [65+]
  RabIndex g_ls = {}, g_lf = {};           // (azimuth bucket x ring) indices over less_sharp / less_flat
};

// Everything one trajectory owns on the device.  A context has cfg.max_batch of them; the single-trajectory entry points
// use lane 0, aloam_scan_stream_batch drives lanes 0 .. batch-1 in lockstep with shared launches.
struct Lane {
  float* d_raw[2] = {nullptr, nullptr};          // raw-scan staging, double-buffered by scan parity
  int8_t* d_ring = nullptr;
  int *d_hist = nullptr, *d_offsets = nullptr, *d_scan_start = nullptr, *d_scan_end = nullptr;
  int* d_ring_start[2] = {nullptr, nullptr};
  ScanScalars* d_sc = nullptr;                   // [3]: scan k uses slot k%3 and re-arms the next
  Pt4* d_full[2] = {nullptr, nullptr};           // ring-major cloud, double-buffered for the pipelined stream call
  // per-ring staging sets: in the stream call k_compact(k) runs on the index stream while k_ring_features(k+1) fills the other set
  Pt4 *st_sharp[2] = {}, *st_less_sharp[2] = {}, *st_flat[2] = {}, *st_less_flat[2] = {};
  int* st_counts[2] = {};
  FeatBuf feat[kFeatSlots + 2];                  // [0, kFeatSlots): ring of feature sets (odometry k reads sets k-1 and k while extraction runs ahead) ; kApiLast, kApiCur
  BlockRec* d_blocks = nullptr;
  int* d_corr = nullptr;
  double *d_pose = nullptr, *d_world = nullptr;  // para_q/para_t (laserOdometry.cpp:97-98) and q_w_curr/t_w_curr (:93-94)
  LmSummary* d_summary = nullptr;                // [4]
};

}  // namespace

struct aloam_ctx {
  aloam_config cfg;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  int max_points = 0, nblocks_max = 0, max_ring = ALOAM_MAX_RING, n_lanes = 1;
  std::vector<Lane> lanes;
  float* d_curv = nullptr;         // debug outputs of the last extraction (lane 0 only)
  int8_t* d_label = nullptr;
  int* d_scan_nfull = nullptr;     // [kMaxStreamScans] ring-major cloud size of every (scan, lane) of a stream call
  double *d_out28 = nullptr, *d_packed = nullptr;
  double* d_api_pose = nullptr;    // [8] pose of the per-stage entry points (odometry_register, solve, ...): not the warm start of the fused pipeline
  int* d_err = nullptr;
  Pt4* d_query = nullptr;
  int* d_knn_idx = nullptr;
  float* d_knn_d = nullptr;
  // multi-GPU sharding of the map (spatial slabs + halo, SURVEY.md 8e): this process's rank / world and its communicator
  int shard_rank = 0, shard_count = 1;
  void* comm = nullptr;          // ncclComm_t when shard_count > 1 (comm.cu)
  void* peer = nullptr;          // peer-memory exchange of the sharded LM (comm.cu), when enabled
  double* d_lm_tot = nullptr;    // [64] all-reduced normal equations of one evaluation (sharded LM)
  void* d_lm_state = nullptr;    // device-resident trust-region state (sharded LM)
  void* mapper = nullptr;        // map cube store (cubemap.cu), created on first use
  // scan-to-map: uploaded submap (corner, surf) with hash grids, stack queries, fit debug records
  MapCloud map_corner = {}, map_surf = {};
  Pt4* d_map_pts[2] = {nullptr, nullptr};   // staging for maps handed in as host views (device views are indexed in place)
  int max_map = 0, map_slots = 0;
  int map_n[2] = {0, 0};          // points indexed on this rank (corner, surf)
  int map_global_n[2] = {0, 0};   // size of the whole submap (== map_n unless the map is sharded over ranks)
  bool have_map = false;
  Pt4 *d_stack_corner = nullptr, *d_stack_surf = nullptr;
  int* d_stack_counts = nullptr;  // [4] {n_corner, n_surf, total} of the stacks being registered
  float4* d_nbr = nullptr;        // [queries][5] neighbours found by k_map_knn5 (x, y, z, index bits)
  double* d_map_pose = nullptr;   // [7] scan-to-map pose being refined (parameters[7], laserMapping.cpp:110)
  double* d_fits = nullptr;       // [queries][14] debug / test records of the line / plane fits
  BlockRec* d_map_blocks = nullptr;
  LmSummary* d_map_summary = nullptr;   // [4] summaries of the scan-to-map solves
  // general voxel filter (voxel.cu): radix-sort ping-pong buffers, histograms, small scalars
  unsigned* d_vox_keys[2] = {nullptr, nullptr};
  int* d_vox_vals[2] = {nullptr, nullptr};
  int *d_vox_hist = nullptr, *d_vox_offs = nullptr, *d_vox_misc = nullptr;
  // pipelined scan stream: ring binning on s_exa, per-ring features on s_ext, compaction + index on s_idx, association + LM
  // on `stream`, host->device copies of the raw scans on s_h2d, scan-to-map on s_map; all chained by events
  cudaStream_t s_ext = nullptr, s_exa = nullptr, s_idx = nullptr, s_h2d = nullptr, s_map = nullptr;
  cudaEvent_t ev_feat[kFeatSlots] = {}, ev_idx[kFeatSlots] = {}, ev_odo[kFeatSlots] = {}, ev_mapdone[kFeatSlots] = {}, ev_h2d[2] = {}, ev_rawfree[2] = {},
              ev_a[2] = {}, ev_b[2] = {}, ev_cmp[2] = {};
  double* h_poses = nullptr;     // pinned [kMaxStreamScans][7]
  double* d_poses = nullptr;     // device [kMaxStreamScans][7]: per-(scan, lane) world poses of a stream call (one D2H at the end)
  double* d_map_poses = nullptr; // device [kMaxStreamScans][7]: map-refined poses (aloam_scan_stream_mapped)
  int* h_scan_nfull = nullptr;   // pinned [kMaxStreamScans]
  // aloam_scan_stream_mapped_registered, created on its first call: every scan's ring-major cloud is copied out of the
  // double-buffered d_full into a per-feature-slot buffer in stage C, then put through pointAssociateToMap with the scan's
  // refined pose on s_reg, behind that scan's mapping step (the s_map chain is not lengthened)
  Pt4* d_reg_full[kFeatSlots] = {};
  long long* d_reg_off = nullptr;   // [kMaxStreamScans + 1] running prefix of the cloud sizes of the current call
  cudaStream_t s_reg = nullptr;
  cudaEvent_t ev_regcopy[kFeatSlots] = {}, ev_regdone[kFeatSlots] = {}, ev_fullfree[2] = {};
  // pinned host mirrors
  Pt4* h_out[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
  Pt4* h_vox_out = nullptr;     // result of aloam_voxel_filter (never aliases the feature views)
  int* h_ints = nullptr;        // scratch ints (counts etc.)
  double* h_dbl = nullptr;      // scratch doubles
  LmSummary* h_summary = nullptr;   // [n_lanes][4]
  ScanScalars* h_sc = nullptr;      // [n_lanes][3]
  // per-kernel profiler (bench.py roofline leg) + cumulative launch counter
  bool prof_on = false;
  cudaEvent_t prof_ev[2 * kProfSlots] = {};
  int prof_kid[kProfSlots] = {};
  int prof_n = 0;
  double prof_ms[ALOAM_N_KERNEL_IDS] = {};
  long long prof_cnt[ALOAM_N_KERNEL_IDS] = {};
  long long launches = 0;
  // state (all lanes advance in lockstep)
  int parity = 0;         // ScanScalars slot of the next scan
  int frame = 0;          // fused pipeline: scans seen
  int cur = 0;            // fused pipeline: feat[] slot of the most recent scan
  bool have_last = false; // API path: set_last called
  int last_n_full = 0;
};

namespace {

enum { KID_CLASSIFY = 0, KID_RING_SCAN, KID_SCATTER, KID_RING_FEATURES, KID_COMPACT, KID_GRID_BUILD, KID_ODOM_ASSOC, KID_LM_SOLVE,
       KID_RING_OFFSETS, KID_KNN_LAST, KID_PACK_BLOCKS, KID_MAP_GRID, KID_MAP_KNN5, KID_VOXEL, KID_MAP_KNN, KID_MAP_FIT, KID_CUBES, KID_LM_SHARD,
       KID_MAP_OUTPUT };
const char* const kKernelNames[ALOAM_N_KERNEL_IDS] = {"k_classify", "k_ring_scan", "k_scatter", "k_ring_features", "k_compact",
    "k_rab_build(3 launches)", "k_odom_assoc", "k_lm_solve", "k_ring_offsets", "k_knn_last", "k_pack_blocks", "k_map_grid(4 launches)", "k_map_knn5",
    "k_voxel", "k_map_knn", "k_map_fit", "k_cube_store", "k_lm_shard", "k_map_outputs"};

inline void prof_begin(aloam_ctx* c, int kid) {
  ++c->launches;
  if (c->prof_on && c->prof_n < kProfSlots) { cudaEventRecord(c->prof_ev[2 * c->prof_n], c->stream); c->prof_kid[c->prof_n] = kid; }
}
inline void prof_end(aloam_ctx* c) {
  if (c->prof_on && c->prof_n < kProfSlots) { cudaEventRecord(c->prof_ev[2 * c->prof_n + 1], c->stream); ++c->prof_n; }
}
// call after the stream has been synchronised
inline void prof_collect(aloam_ctx* c) {
  for (int i = 0; i < c->prof_n; ++i) {
    float ms = 0;
    if (cudaEventElapsedTime(&ms, c->prof_ev[2 * i], c->prof_ev[2 * i + 1]) == cudaSuccess) { c->prof_ms[c->prof_kid[i]] += ms; ++c->prof_cnt[c->prof_kid[i]]; }
  }
  c->prof_n = 0;
}
#define LAUNCH(c, kid, kernel, grid, block, smem, ...) \
  do { prof_begin(c, kid); kernel<<<grid, block, smem, (c)->stream>>>(__VA_ARGS__); prof_end(c); } while (0)

// launch with an optional programmatic dependency on the previous kernel of the stream (PDL): the grid may become resident
// while its predecessor is still running and blocks in pdl_wait() (common.cuh) until the predecessor has completed and flushed.
template <typename K, typename... Args>
void launch_ex(aloam_ctx* c, int kid, K kernel, dim3 grid, dim3 block, size_t smem, int cluster, bool pdl, Args... args) {
  prof_begin(c, kid);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = c->stream;
  cudaLaunchAttribute at[2];
  int na = 0;
  if (cluster > 1) { at[na].id = cudaLaunchAttributeClusterDimension; at[na].val.clusterDim.x = cluster; at[na].val.clusterDim.y = 1; at[na].val.clusterDim.z = 1; ++na; }
  if (pdl && !c->prof_on) { at[na].id = cudaLaunchAttributeProgrammaticStreamSerialization; at[na].val.programmaticStreamSerializationAllowed = 1; ++na; }
  cfg.attrs = at; cfg.numAttrs = na;
  cudaLaunchKernelEx(&cfg, kernel, args...);
  prof_end(c);
}

#define LAUNCH_PDL(c, kid, kernel, grid, block, smem, ...) launch_ex(c, kid, kernel, dim3(grid), dim3(block), smem, 1, true, __VA_ARGS__)

// the LM kernel runs as one thread-block cluster per trajectory (distributed-shared-memory reduction, see lm.cu)
constexpr int kLmCluster = 8;
// general = false: all blocks have s == 1 and there is no peer exchange (the reference-build odometry, scan-to-map on one GPU)
inline void launch_lm_batch(aloam_ctx* c, bool pdl, const Batch<LmArgs>& args, int lanes, const LmParams& lp, int mode, int integrate, bool general = false,
                            const PeerX* px = nullptr) {
  if (!general && !px) {
    launch_ex(c, KID_LM_SOLVE, k_lm_solve, dim3(kLmCluster, lanes), dim3(ALOAM_LM_THREADS), lm_dynamic_smem_bytes(), kLmCluster, pdl, args, lp, mode, integrate);
    return;
  }
  PeerX none = {};
  launch_ex(c, KID_LM_SOLVE, k_lm_solve_x, dim3(kLmCluster, lanes), dim3(ALOAM_LM_THREADS), lm_dynamic_smem_bytes(), kLmCluster, pdl, args, lp, mode, integrate,
            px ? *px : none);
}
// single solve: blocks, n (device pointer or host value), pose in / out
inline void launch_lm(aloam_ctx* c, bool pdl, const BlockRec* blocks, const int* n_ptr, int n_host, double* x7, const LmParams& lp, LmSummary* summary,
                      int mode, double* out28, double* world7, int integrate, bool general = false) {
  Batch<LmArgs> b = {};
  b.a[0] = LmArgs{blocks, n_ptr, n_host, x7, summary, out28, world7};
  launch_lm_batch(c, pdl, b, 1, lp, mode, integrate, general);
}

}  // namespace
// sharded LM (comm.cu): per evaluation one kernel for the local blocks, one exchange of 32 doubles, one step kernel
void launch_lm_sharded(aloam_ctx* c, const aloam::BlockRec* blocks, const int* d_n, double* pose, const aloam::LmParams& lp, aloam::LmSummary* summary);
void vox_seg_filter(aloam_ctx* c, const aloam::SegFilter& f, aloam::SegBuffers& b, int S_upper, int n_upper, int per_seg_upper);
int vox_seg_alloc(aloam::SegBuffers& b, size_t cap);
void vox_seg_free(aloam::SegBuffers& b);
int mapper_step_device(aloam_ctx* c, const Pt4* d_corner_last, const int* d_nc, int n_upper_c, const Pt4* d_surf_last, const int* d_ns, int n_upper_s,
                       const double* d_odom7, double* d_out7);
// map outputs (cubemap.cu), on c->stream.  Stage C of the registered stream: copy scan k's ring-major cloud (size *d_n) to
// dst and advance the running offsets off[k + 1] = off[k] + *d_n.  Then, behind the scan's mapping step: pointAssociateToMap
// of those points with pose x7 into out[off[k] ...] when off[k + 1] <= capacity (n_upper bounds *d_n).
void map_out_stage_full(aloam_ctx* c, const Pt4* full, const int* d_n, int n_upper, int k, Pt4* dst, long long* off);
void map_out_register(aloam_ctx* c, const Pt4* src, const int* d_n, int n_upper, const long long* off_k, long long capacity, const double* x7, Pt4* out);
void map_index_build(aloam_ctx* c, const Pt4* d_corner, const Pt4* d_surf, int n_upper);
int map_shard_index_device(aloam_ctx* c, const Pt4* sub_corner, const int* n_corner, const Pt4* sub_surf, const int* n_surf, int n_upper, int* err_word);
void map_register_device(aloam_ctx* c, const Pt4* d_corner_stack, const Pt4* d_surf_stack, const int* d_counts3, int nq_upper, double* d_pose, bool want_fits);
namespace {

LmParams lm_params(const aloam_config& c) {
  LmParams p;
  p.max_iters = c.inner_iters; p.huber_a = c.huber;
  p.initial_radius = 1e4; p.max_radius = 1e16; p.min_radius = 1e-32;
  p.min_relative_decrease = 1e-3; p.min_lm_diagonal = 1e-6; p.max_lm_diagonal = 1e32;
  p.function_tolerance = 1e-6; p.gradient_tolerance = 1e-10; p.parameter_tolerance = 1e-8;
  p.max_invalid = 5;
  return p;
}

template <typename T> cudaError_t dalloc(T** p, size_t n) { return cudaMalloc((void**)p, n * sizeof(T)); }
template <typename T> cudaError_t halloc(T** p, size_t n) { return cudaMallocHost((void**)p, n * sizeof(T)); }

int upload_cloud(aloam_ctx* c, aloam_cloud_view v, Pt4* dst, int capacity) {
  if (v.n < 0 || (v.n > 0 && !v.data) || (v.stride_floats != 4 && v.stride_floats != 8 && v.n > 0)) return ALOAM_ERR_INVALID_ARG;
  if (v.n > capacity) return ALOAM_ERR_CAPACITY;
  if (v.n == 0) return ALOAM_OK;
  if (v.stride_floats == 4) {
    CUDA_CHECK_RET(cudaMemcpyAsync(dst, v.data, (size_t)v.n * 16, cudaMemcpyDefault, c->stream));   // host or device source
  } else {
    CUDA_CHECK_RET(cudaMemcpy2DAsync(dst, 16, v.data, (size_t)v.stride_floats * 4, 16, v.n, cudaMemcpyDefault, c->stream));
  }
  return ALOAM_OK;
}

LastCloud last_corner(const FeatBuf& f) { return LastCloud{f.less_sharp, f.counts + 1, f.g_ls}; }
LastCloud last_surf(const FeatBuf& f) { return LastCloud{f.less_flat, f.counts + 3, f.g_lf}; }

void fill_stats_from(const LmSummary* h_summary, aloam_stats* st, int outer, int flags, float ms) {
  if (!st) return;
  std::memset(st, 0, sizeof(*st));
  st->flags = flags;
  st->ms_total = ms;
  for (int it = 0; it < outer && it < 4; ++it) {
    const LmSummary& s = h_summary[it];
    st->lm_iters += s.num_iterations;
    st->accepted_steps += s.num_successful;
    st->termination[it] = s.termination;
    if (it == outer - 1) {
      st->n_corner_corr = s.n_edge; st->n_plane_corr = s.n_plane;
      st->init_cost = s.initial_cost; st->final_cost = s.final_cost;
      if (s.n_edge + s.n_plane < 10) st->flags |= ALOAM_FLAG_FEW_CORRESPONDENCES;
    }
  }
}
inline void fill_stats(aloam_ctx* c, aloam_stats* st, int outer, int flags, float ms) { fill_stats_from(c->h_summary, st, outer, flags, ms); }

int check_view(const aloam_cloud_view& v) {
  if (v.n < 0) return ALOAM_ERR_INVALID_ARG;
  if (v.n > 0 && (!v.data || (v.stride_floats != 4 && v.stride_floats != 8))) return ALOAM_ERR_INVALID_ARG;
  return ALOAM_OK;
}

}  // namespace
