// Host side of the C ABI (include/aloam_b200.h): context, device buffers, kernel sequencing.
// The reference's host code around the hot path is C++ (the ROS node bodies), so this layer is C++ too.
// No CPU fallback: every entry point runs the sm_100a kernels or returns an error.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <chrono>
#include <cstring>
#include <new>
#include <vector>
#include "../../include/aloam_b200.h"
#include "kernels.h"

#include "ctx.h"

extern "C" {

void aloam_map_free_impl(aloam_ctx* c);
void aloam_comm_free_impl(aloam_ctx* c);
void aloam_mapper_free_impl(aloam_ctx* c);
int aloam_map_knn_impl(aloam_ctx* c, int which, aloam_cloud_view queries, int k, int* idx, float* sqdist);

void aloam_default_config(aloam_config* cfg, int n_scans) {
  if (!cfg) return;
  std::memset(cfg, 0, sizeof(*cfg));
  cfg->n_scans = n_scans;
  // launch/aloam_velodyne_VLP_16.launch:3-13, ..._HDL_32.launch:3-13, ..._HDL_64.launch:3-13
  if (n_scans == 64) { cfg->minimum_range = 5.0f; cfg->line_res = 0.4f; cfg->plane_res = 0.8f; }
  else { cfg->minimum_range = 0.3f; cfg->line_res = 0.2f; cfg->plane_res = 0.4f; }
  cfg->outer_iters = 2; cfg->inner_iters = 4; cfg->huber = 0.1;
  cfg->dist_sq_thresh = 25.0; cfg->nearby_scan = 2.5;
  cfg->device = 0; cfg->max_points = 400000; cfg->max_map_points = 0;
  cfg->max_batch = 1; cfg->distortion = 0; cfg->max_ring_points = ALOAM_MAX_RING_POINTS;
}

const char* aloam_strerror(int code) {
  switch (code) {
    case ALOAM_OK: return "ok";
    case ALOAM_ERR_INVALID_ARG: return "invalid argument";
    case ALOAM_ERR_UNSUPPORTED_SCANS: return "only 16, 32 or 64 scan lines are supported";
    case ALOAM_ERR_EMPTY_CLOUD: return "no point survives the NaN / minimum-range filter";
    case ALOAM_ERR_CAPACITY: return "cloud larger than the context capacity";
    case ALOAM_ERR_CUDA: return "CUDA error";
    case ALOAM_ERR_NO_DEVICE: return "no CUDA device";
    case ALOAM_ERR_RING_TOO_LARGE: return "a ring holds more than cfg.max_ring_points returns";
    case ALOAM_ERR_NOT_RING_MAJOR: return "cloud is not in ascending ring order";
    case ALOAM_ERR_STATE: return "call sequence error";
    case ALOAM_ERR_COMM: return "communicator error";
    default: return "unknown error";
  }
}

static void free_lane(Lane& L) {
  void* dev[] = {L.d_raw[0], L.d_raw[1], L.d_ring, L.d_hist, L.d_offsets, L.d_scan_start, L.d_scan_end, L.d_ring_start[0], L.d_ring_start[1], L.d_sc,
                 L.d_full[0], L.d_full[1], L.st_sharp[0], L.st_sharp[1], L.st_less_sharp[0], L.st_less_sharp[1], L.st_flat[0], L.st_flat[1],
                 L.st_less_flat[0], L.st_less_flat[1], L.st_counts[0], L.st_counts[1], L.d_blocks, L.d_corr, L.d_pose, L.d_world, L.d_summary};
  for (void* p : dev) if (p) cudaFree(p);
  for (FeatBuf& f : L.feat) {
    void* fp[] = {f.sharp, f.less_sharp, f.flat, f.less_flat, f.counts, f.rs_ls, f.rs_lf};
    for (void* p : fp) if (p) cudaFree(p);
    for (RabIndex* g : {&f.g_ls, &f.g_lf}) {
      void* gp[] = {g->cnt, g->start, g->cell_of, g->rank_of, g->gpts};
      for (void* p : gp) if (p) cudaFree(p);
    }
  }
}

int aloam_destroy(aloam_ctx* c) {
  if (!c) return ALOAM_OK;
  cudaSetDevice(c->cfg.device);
  cudaStream_t* side[] = {&c->s_ext, &c->s_h2d, &c->s_exa, &c->s_idx, &c->s_map};
  if (c->stream) cudaStreamSynchronize(c->stream);
  for (cudaStream_t* s : side) if (*s) { cudaStreamSynchronize(*s); cudaStreamDestroy(*s); }
  for (cudaEvent_t e : c->ev_idx) if (e) cudaEventDestroy(e);
  for (cudaEvent_t e : c->ev_a) if (e) cudaEventDestroy(e);
  for (cudaEvent_t e : c->ev_b) if (e) cudaEventDestroy(e);
  for (cudaEvent_t e : c->ev_cmp) if (e) cudaEventDestroy(e);
  for (cudaEvent_t e : c->ev_feat) if (e) cudaEventDestroy(e);
  for (cudaEvent_t e : c->ev_odo) if (e) cudaEventDestroy(e);
  for (cudaEvent_t e : c->ev_mapdone) if (e) cudaEventDestroy(e);
  for (cudaEvent_t e : c->ev_h2d) if (e) cudaEventDestroy(e);
  for (cudaEvent_t e : c->ev_rawfree) if (e) cudaEventDestroy(e);
  if (c->s_reg) { cudaStreamSynchronize(c->s_reg); cudaStreamDestroy(c->s_reg); }
  for (cudaEvent_t e : c->ev_regcopy) if (e) cudaEventDestroy(e);
  for (cudaEvent_t e : c->ev_regdone) if (e) cudaEventDestroy(e);
  for (cudaEvent_t e : c->ev_fullfree) if (e) cudaEventDestroy(e);
  for (Pt4* p : c->d_reg_full) if (p) cudaFree(p);
  if (c->d_reg_off) cudaFree(c->d_reg_off);
  if (c->h_poses) cudaFreeHost(c->h_poses);
  if (c->h_scan_nfull) cudaFreeHost(c->h_scan_nfull);
  for (Lane& L : c->lanes) free_lane(L);
  void* dev[] = {c->d_poses, c->d_map_poses, c->d_scan_nfull, c->d_curv, c->d_label, c->d_out28, c->d_api_pose, c->d_packed, c->d_err, c->d_query, c->d_knn_idx, c->d_knn_d};
  for (void* p : dev) if (p) cudaFree(p);
  aloam_map_free_impl(c);
  { void* vp[] = {c->d_vox_keys[0], c->d_vox_keys[1], c->d_vox_vals[0], c->d_vox_vals[1], c->d_vox_hist, c->d_vox_offs, c->d_vox_misc}; for (void* p : vp) if (p) cudaFree(p); }
  aloam_comm_free_impl(c);
  aloam_mapper_free_impl(c);
  for (Pt4* p : c->h_out) if (p) cudaFreeHost(p);
  if (c->h_vox_out) cudaFreeHost(c->h_vox_out);
  if (c->h_ints) cudaFreeHost(c->h_ints);
  if (c->h_dbl) cudaFreeHost(c->h_dbl);
  if (c->h_summary) cudaFreeHost(c->h_summary);
  if (c->h_sc) cudaFreeHost(c->h_sc);
  for (cudaEvent_t e : c->prof_ev) if (e) cudaEventDestroy(e);
  if (c->ev0) cudaEventDestroy(c->ev0);
  if (c->ev1) cudaEventDestroy(c->ev1);
  if (c->stream) cudaStreamDestroy(c->stream);
  delete c;
  return ALOAM_OK;
}

int aloam_mapper_reset(aloam_ctx* c);

int aloam_reset_odometry(aloam_ctx* c) {
  if (!c) return ALOAM_ERR_INVALID_ARG;
  CUDA_CHECK_RET(cudaSetDevice(c->cfg.device));
  const double ident[7] = {0, 0, 0, 1, 0, 0, 0};
  for (Lane& L : c->lanes) {
    CUDA_CHECK_RET(cudaMemcpyAsync(L.d_pose, ident, sizeof(ident), cudaMemcpyHostToDevice, c->stream));
    CUDA_CHECK_RET(cudaMemcpyAsync(L.d_world, ident, sizeof(ident), cudaMemcpyHostToDevice, c->stream));
  }
  CUDA_CHECK_RET(cudaStreamSynchronize(c->stream));
  if (c->s_idx) CUDA_CHECK_RET(cudaStreamSynchronize(c->s_idx));   // an index build of the last synchronous call may still be running
  c->frame = 0; c->cur = 0; c->have_last = false;
  return ALOAM_OK;
}

int aloam_create(const aloam_config* cfg_in, aloam_ctx** out) {
  if (!cfg_in || !out) return ALOAM_ERR_INVALID_ARG;
  *out = nullptr;
  aloam_config cfg = *cfg_in;
  if (cfg.max_batch == 0) cfg.max_batch = 1;                                  // zero-initialised tail of an older caller
  if (cfg.max_ring_points == 0) cfg.max_ring_points = ALOAM_MAX_RING_POINTS;
  if (cfg.n_scans != 16 && cfg.n_scans != 32 && cfg.n_scans != 64) return ALOAM_ERR_UNSUPPORTED_SCANS;
  if (cfg.max_points <= 0 || cfg.outer_iters < 1 || cfg.outer_iters > 4 || cfg.inner_iters < 0) return ALOAM_ERR_INVALID_ARG;
  if (cfg.max_batch < 1 || cfg.max_batch > ALOAM_MAX_BATCH) return ALOAM_ERR_INVALID_ARG;
  if (cfg.max_ring_points < 64 || cfg.max_ring_points > ALOAM_MAX_RING_POINTS || cfg.max_ring_points % 32) return ALOAM_ERR_INVALID_ARG;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) return ALOAM_ERR_NO_DEVICE;
  if (cfg.device < 0 || cfg.device >= ndev) return ALOAM_ERR_INVALID_ARG;
  CUDA_CHECK_RET(cudaSetDevice(cfg.device));
  aloam_ctx* c = new (std::nothrow) aloam_ctx();
  if (!c) return ALOAM_ERR_INVALID_ARG;
  c->cfg = cfg;
  c->max_points = cfg.max_points;
  c->max_ring = cfg.max_ring_points;
  c->n_lanes = cfg.max_batch;
  c->nblocks_max = (c->max_points + 1023) / 1024;
  const size_t mp = (size_t)c->max_points;
  const size_t mr = (size_t)c->max_ring;
#define TRY(e) do { if ((e) != cudaSuccess) { fprintf(stderr, "[aloam_b200] %s failed: %s\n", #e, cudaGetErrorString(cudaGetLastError())); aloam_destroy(c); return ALOAM_ERR_CUDA; } } while (0)
  TRY(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  TRY(cudaEventCreate(&c->ev0)); TRY(cudaEventCreate(&c->ev1));
  for (cudaEvent_t& e : c->prof_ev) TRY(cudaEventCreate(&e));
  for (cudaStream_t* s : {&c->s_ext, &c->s_h2d, &c->s_exa, &c->s_idx, &c->s_map}) TRY(cudaStreamCreateWithFlags(s, cudaStreamNonBlocking));
  for (cudaEvent_t& e : c->ev_idx) TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  for (cudaEvent_t& e : c->ev_a) TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  for (cudaEvent_t& e : c->ev_b) TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  for (cudaEvent_t& e : c->ev_cmp) TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  for (cudaEvent_t& e : c->ev_feat) TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  for (cudaEvent_t& e : c->ev_odo) TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  for (cudaEvent_t& e : c->ev_mapdone) TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  for (cudaEvent_t& e : c->ev_h2d) TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  for (cudaEvent_t& e : c->ev_rawfree) TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  TRY(halloc(&c->h_poses, (size_t)kMaxStreamScans * 14)); TRY(dalloc(&c->d_poses, (size_t)kMaxStreamScans * 7)); TRY(dalloc(&c->d_map_poses, (size_t)kMaxStreamScans * 7));
  TRY(halloc(&c->h_scan_nfull, (size_t)kMaxStreamScans)); TRY(dalloc(&c->d_scan_nfull, (size_t)kMaxStreamScans));
  TRY(dalloc(&c->d_curv, mp)); TRY(dalloc(&c->d_label, mp));
  c->lanes.resize(c->n_lanes);
  ScanScalars init[3];
  for (ScanScalars& s : init) { s.first_valid = INT32_MAX; s.last_valid = -1; s.half_idx = INT32_MAX; s.n_full = 0; s.start_ori = 0; s.end_ori = 0; s.error = 0; s.pad = 0; }
  for (Lane& L : c->lanes) {
    for (int b = 0; b < 2; ++b) {
      TRY(dalloc(&L.d_raw[b], mp * 8)); TRY(dalloc(&L.d_full[b], mp)); TRY(dalloc(&L.d_ring_start[b], 72));
      TRY(dalloc(&L.st_sharp[b], 64 * kMaxSharpPerRing)); TRY(dalloc(&L.st_less_sharp[b], 64 * kMaxLessSharpPerRing));
      TRY(dalloc(&L.st_flat[b], 64 * kMaxFlatPerRing)); TRY(dalloc(&L.st_less_flat[b], (size_t)64 * mr));
      TRY(dalloc(&L.st_counts[b], 64 * 4));
    }
    TRY(dalloc(&L.d_ring, mp));
    TRY(dalloc(&L.d_hist, (size_t)c->nblocks_max * 64)); TRY(dalloc(&L.d_offsets, (size_t)c->nblocks_max * 64));
    TRY(dalloc(&L.d_scan_start, 64)); TRY(dalloc(&L.d_scan_end, 64));
    TRY(dalloc(&L.d_sc, 3));
    TRY(cudaMemcpy(L.d_sc, init, sizeof(init), cudaMemcpyHostToDevice));
    for (FeatBuf& f : L.feat) {
      TRY(dalloc(&f.sharp, kMaxQueries)); TRY(dalloc(&f.flat, kMaxQueries));
      TRY(dalloc(&f.less_sharp, mp)); TRY(dalloc(&f.less_flat, mp));
      TRY(dalloc(&f.counts, 4)); TRY(dalloc(&f.rs_ls, 72)); TRY(dalloc(&f.rs_lf, 72));
      for (RabIndex* g : {&f.g_ls, &f.g_lf}) {
        TRY(dalloc(&g->cnt, (size_t)ALOAM_NB * 64)); TRY(dalloc(&g->start, (size_t)ALOAM_NB * 64 + 8));
        TRY(dalloc(&g->cell_of, mp)); TRY(dalloc(&g->rank_of, mp)); TRY(dalloc(&g->gpts, mp));
        TRY(cudaMemset(g->cnt, 0, (size_t)ALOAM_NB * 64 * 4)); TRY(cudaMemset(g->start, 0, ((size_t)ALOAM_NB * 64 + 8) * 4));
      }
      TRY(cudaMemset(f.counts, 0, 16)); TRY(cudaMemset(f.rs_ls, 0, 72 * 4)); TRY(cudaMemset(f.rs_lf, 0, 72 * 4));
    }
    TRY(dalloc(&L.d_blocks, (size_t)2 * kMaxQueries)); TRY(dalloc(&L.d_corr, (size_t)2 * kMaxQueries * 4));
    TRY(dalloc(&L.d_pose, 8)); TRY(dalloc(&L.d_world, 8)); TRY(dalloc(&L.d_summary, 4));
  }
  TRY(dalloc(&c->d_out28, 32)); TRY(dalloc(&c->d_api_pose, 8));
  TRY(dalloc(&c->d_packed, (size_t)2 * kMaxQueries * 11));
  TRY(dalloc(&c->d_err, 4));
  TRY(dalloc(&c->d_query, mp)); TRY(dalloc(&c->d_knn_idx, mp)); TRY(dalloc(&c->d_knn_d, mp));
  for (int k = 0; k < 5; ++k) TRY(halloc(&c->h_out[k], k == 0 || k == 4 ? mp : (size_t)kMaxQueries));
  TRY(halloc(&c->h_ints, 4096)); TRY(halloc(&c->h_dbl, 4096));
  TRY(halloc(&c->h_summary, (size_t)4 * c->n_lanes)); TRY(halloc(&c->h_sc, (size_t)3 * c->n_lanes));
  TRY(cudaMemset(c->d_err, 0, 16));
  // function attributes are process-wide: always opt in to the largest ring capacity, whatever this context uses
  TRY(cudaFuncSetAttribute(k_ring_features, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ring_features_smem_bytes(ALOAM_MAX_RING, true)));
  TRY(cudaFuncSetAttribute(k_ring_features_batch, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ring_features_smem_bytes(ALOAM_MAX_RING, false)));
  TRY(cudaFuncSetAttribute(k_lm_solve, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lm_dynamic_smem_bytes()));
  TRY(cudaFuncSetAttribute(k_lm_solve_x, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lm_dynamic_smem_bytes()));
  TRY(cudaFuncSetAttribute(k_lm_eval_shard, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lm_dynamic_smem_bytes()));
#undef TRY
  int rc = aloam_reset_odometry(c);
  if (rc != ALOAM_OK) { aloam_destroy(c); return rc; }
  *out = c;
  return ALOAM_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------ kernel sequencing
namespace {

// Feature extraction is issued in two halves so that the pipelined stream call can run them on different streams:
//   A  ring binning   (k_classify, k_ring_scan, k_scatter)  raw scan -> ring-major cloud `full[buf]`, ring_start[buf]
//   B  per-ring work  (k_ring_features, k_compact)          full[buf] -> the four feature clouds of feat[slot]
// Every launch covers lanes 0 .. nb-1.  `sc_slot` (returned by A, consumed by B) is the ScanScalars parity slot of this scan;
// nfull_out (device, nb ints, may be null) receives the ring-major cloud sizes.
int run_features_a(aloam_ctx* c, int nb, const float* const* d_raw, const int* n, int stride, int buf, int* sc_slot, int* nfull_out) {
  int nmax = 0;
  for (int l = 0; l < nb; ++l) nmax = std::max(nmax, n[l]);
  const int blocks = (nmax + 1023) / 1024;
  const float thres = c->cfg.minimum_range;
  Batch<ClassifyArgs> ca = {}; Batch<RingScanArgs> ra = {}; Batch<ScatterArgs> sa = {};
  for (int l = 0; l < nb; ++l) {
    Lane& L = c->lanes[l];
    ScanScalars* sc = L.d_sc + c->parity;
    ScanScalars* sc_next = L.d_sc + (c->parity + 1) % 3;
    ca.a[l] = ClassifyArgs{d_raw[l], n[l], stride, L.d_ring, L.d_hist, sc};
    ra.a[l] = RingScanArgs{d_raw[l], stride, (n[l] + 1023) / 1024, L.d_hist, L.d_offsets, L.d_ring_start[buf], L.d_scan_start, L.d_scan_end, sc, sc_next,
                           nfull_out ? nfull_out + l : nullptr};
    sa.a[l] = ScatterArgs{d_raw[l], n[l], stride, L.d_ring, L.d_offsets, sc, L.d_full[buf]};
  }
  LAUNCH(c, KID_CLASSIFY, k_classify, dim3(blocks, nb), 256, 0, ca, c->cfg.n_scans, thres * thres);
  launch_ex(c, KID_RING_SCAN, k_ring_scan, dim3(nb), dim3(1024), 0, 1, true, ra, c->cfg.n_scans);
  launch_ex(c, KID_SCATTER, k_scatter, dim3(blocks, nb), dim3(256), 0, 1, true, sa);
  *sc_slot = c->parity;
  c->parity = (c->parity + 1) % 3;
  CUDA_CHECK_RET(cudaGetLastError());
  return ALOAM_OK;
}
// B1: per-ring kernel -> staging set `buf` ; B2: ring-ordered concatenation of the staging set into feat[slot]
int run_features_b1(aloam_ctx* c, int nb, int buf, int sc_slot) {
  Batch<RingFeatArgs> fa = {};
  for (int l = 0; l < nb; ++l) {
    Lane& L = c->lanes[l];
    fa.a[l] = RingFeatArgs{L.d_full[buf], L.d_ring_start[buf], L.st_sharp[buf], L.st_less_sharp[buf], L.st_flat[buf], L.st_less_flat[buf], L.st_counts[buf],
                           l == 0 ? c->d_curv : nullptr, l == 0 ? c->d_label : nullptr, L.d_sc + sc_slot};
  }
  // one trajectory: a cluster of two CTAs per ring (picks | voxel sort, see features.cu) ; a batch: one CTA per ring and trajectory
  if (nb == 1) launch_ex(c, KID_RING_FEATURES, k_ring_features, dim3(2 * c->cfg.n_scans, 1), dim3(512), ring_features_smem_bytes(c->max_ring, true), 2, false, fa, c->cfg.n_scans, 0.2f, c->max_ring);
  else LAUNCH(c, KID_RING_FEATURES, k_ring_features_batch, dim3(c->cfg.n_scans, nb), 256, ring_features_smem_bytes(c->max_ring, false), fa, c->cfg.n_scans, 0.2f, c->max_ring);
  CUDA_CHECK_RET(cudaGetLastError());
  return ALOAM_OK;
}
int run_features_b2(aloam_ctx* c, int nb, int buf, int slot, bool pdl) {
  Batch<CompactArgs> ka = {};
  for (int l = 0; l < nb; ++l) {
    Lane& L = c->lanes[l];
    FeatBuf& out = L.feat[slot];
    ka.a[l] = CompactArgs{L.st_sharp[buf], L.st_less_sharp[buf], L.st_flat[buf], L.st_less_flat[buf], L.st_counts[buf], out.sharp, out.less_sharp, out.flat,
                          out.less_flat, out.counts, out.rs_ls, out.rs_lf};
  }
  launch_ex(c, KID_COMPACT, k_compact, dim3(c->cfg.n_scans, nb), dim3(128), 0, 1, pdl, ka, c->cfg.n_scans, c->max_ring);
  CUDA_CHECK_RET(cudaGetLastError());
  return ALOAM_OK;
}
int run_features(aloam_ctx* c, int nb, const float* const* d_raw, const int* n, int stride, int slot) {
  int sc = 0;
  int rc = run_features_a(c, nb, d_raw, n, stride, 0, &sc, nullptr);
  if (rc) return rc;
  rc = run_features_b1(c, nb, 0, sc);
  if (rc) return rc;
  return run_features_b2(c, nb, 0, slot, true);
}

// index over the two "last" clouds of feat[slot]: count -> scan -> fill (n_ls / n_lf = host upper bounds on the cloud sizes)
void run_grid_build(aloam_ctx* c, int nb, int slot, int n_ls, int n_lf) {
  const int pb = (std::max(std::max(n_ls, n_lf), 1) + 255) / 256;
  Batch<RabArgs> ga = {};
  for (int l = 0; l < nb; ++l) {
    FeatBuf& f = c->lanes[l].feat[slot];
    ga.a[l] = RabArgs{f.g_ls, f.less_sharp, f.counts + 1, f.g_lf, f.less_flat, f.counts + 3};
  }
  LAUNCH(c, KID_GRID_BUILD, k_rab_count, dim3(pb, 2, nb), 256, 0, ga);
  launch_ex(c, KID_GRID_BUILD, k_rab_scan, dim3(2, nb), dim3(1024), 0, 1, true, ga);
  launch_ex(c, KID_GRID_BUILD, k_rab_fill, dim3(pb, 2, nb), dim3(256), 0, 1, true, ga);
}

// outer_iters x (association + LM) ; feat[cur] supplies sharp/flat, feat[last] the targets ; pose in lane.d_pose
// pose_slots (device, lane-major 7 doubles each, may be null): the integrated world pose is also written there by the last solve
void run_register(aloam_ctx* c, int nb, int cur, int last, int sharp_slots, int flat_slots, bool integrate, bool want_corr, double* pose_slots,
                  double* pose_override = nullptr /* lane 0: solve for this pose instead of the lane's warm start */) {
  OdomParams op{c->cfg.dist_sq_thresh, c->cfg.nearby_scan, c->cfg.distortion};
  const LmParams lp = lm_params(c->cfg);
  const int slots = sharp_slots + flat_slots;
  for (int it = 0; it < c->cfg.outer_iters; ++it) {
    const bool last_it = it == c->cfg.outer_iters - 1;
    Batch<AssocArgs> aa = {}; Batch<LmArgs> la = {};
    for (int l = 0; l < nb; ++l) {
      Lane& L = c->lanes[l];
      const FeatBuf& fc = L.feat[cur];
      const FeatBuf& fl = L.feat[last];
      double* pose = (l == 0 && pose_override) ? pose_override : L.d_pose;
      aa.a[l] = AssocArgs{fc.sharp, fc.flat, fc.counts, last_corner(fl), last_surf(fl), pose, L.d_blocks, want_corr ? L.d_corr : nullptr};
      la.a[l] = LmArgs{L.d_blocks, nullptr, slots, pose, L.d_summary + (it & 3), (integrate && last_it && pose_slots) ? pose_slots + (size_t)l * 7 : nullptr, L.d_world};
    }
    // within one call the chain association -> LM -> association -> LM is launched with programmatic dependencies
    if (slots > 0) launch_ex(c, KID_ODOM_ASSOC, k_odom_assoc, dim3((slots + 7) / 8, nb), dim3(256), 0, 1, it > 0, aa, op, sharp_slots);
    launch_lm_batch(c, slots > 0, la, nb, lp, 0, (integrate && last_it) ? 1 : 0, c->cfg.distortion != 0);
  }
}

// restores the main stream on every exit of a function that re-points c->stream at the side streams
struct StreamGuard {
  aloam_ctx* c; cudaStream_t main;
  explicit StreamGuard(aloam_ctx* ctx) : c(ctx), main(ctx->stream) {}
  ~StreamGuard() { c->stream = main; }
};

void sync_all_streams(aloam_ctx* c) {
  cudaStream_t ss[] = {c->stream, c->s_ext, c->s_exa, c->s_idx, c->s_h2d, c->s_map, c->s_reg};
  for (cudaStream_t s : ss) if (s) cudaStreamSynchronize(s);
}

}  // namespace

extern "C" {

// ------------------------------------------------------------------------------------------------ feature extraction
int aloam_extract_features(aloam_ctx* c, aloam_cloud_view raw, aloam_cloud_view* full, aloam_cloud_view* sharp,
                           aloam_cloud_view* less_sharp, aloam_cloud_view* flat, aloam_cloud_view* less_flat) {
  if (!c || !full || !sharp || !less_sharp || !flat || !less_flat) return ALOAM_ERR_INVALID_ARG;
  int rc = check_view(raw);
  if (rc) return rc;
  if (raw.n == 0) return ALOAM_ERR_EMPTY_CLOUD;
  if (raw.n > c->max_points) return ALOAM_ERR_CAPACITY;
  CUDA_CHECK_RET(cudaSetDevice(c->cfg.device));
  Lane& L = c->lanes[0];
  CUDA_CHECK_RET(cudaMemcpyAsync(L.d_raw[0], raw.data, (size_t)raw.n * raw.stride_floats * 4, cudaMemcpyHostToDevice, c->stream));
  FeatBuf& f = L.feat[kApiCur];
  const int slot = c->parity;
  const float* rp = L.d_raw[0];
  rc = run_features(c, 1, &rp, &raw.n, raw.stride_floats, kApiCur);
  if (rc) return rc;
  CUDA_CHECK_RET(cudaMemcpyAsync(c->h_ints, f.counts, 16, cudaMemcpyDeviceToHost, c->stream));
  CUDA_CHECK_RET(cudaMemcpyAsync(c->h_sc, L.d_sc + slot, sizeof(ScanScalars), cudaMemcpyDeviceToHost, c->stream));
  CUDA_CHECK_RET(cudaStreamSynchronize(c->stream));
  if (c->h_sc->error) {
    int e = c->h_sc->error;
    CUDA_CHECK_RET(cudaMemset(&(L.d_sc + slot)->error, 0, 4));
    return e;
  }
  const int n_full = c->h_sc->n_full;
  c->last_n_full = n_full;
  if (c->h_sc->first_valid == INT32_MAX) return ALOAM_ERR_EMPTY_CLOUD;
  const int n[5] = {n_full, c->h_ints[0], c->h_ints[1], c->h_ints[2], c->h_ints[3]};
  const Pt4* src[5] = {L.d_full[0], f.sharp, f.less_sharp, f.flat, f.less_flat};
  for (int k = 0; k < 5; ++k)
    if (n[k] > 0) CUDA_CHECK_RET(cudaMemcpyAsync(c->h_out[k], src[k], (size_t)n[k] * 16, cudaMemcpyDeviceToHost, c->stream));
  CUDA_CHECK_RET(cudaStreamSynchronize(c->stream));
  aloam_cloud_view* outs[5] = {full, sharp, less_sharp, flat, less_flat};
  for (int k = 0; k < 5; ++k) { outs[k]->data = reinterpret_cast<const float*>(c->h_out[k]); outs[k]->n = n[k]; outs[k]->stride_floats = 4; }
  return ALOAM_OK;
}

int aloam_debug_features(aloam_ctx* c, float* curvature, int* label, int* scan_start, int* scan_end) {
  if (!c) return ALOAM_ERR_INVALID_ARG;
  CUDA_CHECK_RET(cudaSetDevice(c->cfg.device));
  const int n = c->last_n_full;
  if (curvature && n > 0) CUDA_CHECK_RET(cudaMemcpy(curvature, c->d_curv, (size_t)n * 4, cudaMemcpyDeviceToHost));
  if (label && n > 0) {
    std::vector<int8_t> tmp(n);
    CUDA_CHECK_RET(cudaMemcpy(tmp.data(), c->d_label, (size_t)n, cudaMemcpyDeviceToHost));
    for (int i = 0; i < n; ++i) label[i] = tmp[i];
  }
  if (scan_start) CUDA_CHECK_RET(cudaMemcpy(scan_start, c->lanes[0].d_scan_start, (size_t)c->cfg.n_scans * 4, cudaMemcpyDeviceToHost));
  if (scan_end) CUDA_CHECK_RET(cudaMemcpy(scan_end, c->lanes[0].d_scan_end, (size_t)c->cfg.n_scans * 4, cudaMemcpyDeviceToHost));
  return ALOAM_OK;
}

// ------------------------------------------------------------------------------------------------ odometry (API path)
int aloam_odometry_set_last(aloam_ctx* c, aloam_cloud_view corner_last, aloam_cloud_view surf_last) {
  if (!c) return ALOAM_ERR_INVALID_ARG;
  int rc = check_view(corner_last); if (rc) return rc;
  rc = check_view(surf_last); if (rc) return rc;
  CUDA_CHECK_RET(cudaSetDevice(c->cfg.device));
  FeatBuf& f = c->lanes[0].feat[kApiLast];
  rc = upload_cloud(c, corner_last, f.less_sharp, c->max_points); if (rc) return rc;
  rc = upload_cloud(c, surf_last, f.less_flat, c->max_points); if (rc) return rc;
  c->h_ints[0] = 0; c->h_ints[1] = corner_last.n; c->h_ints[2] = 0; c->h_ints[3] = surf_last.n;
  CUDA_CHECK_RET(cudaMemcpyAsync(f.counts, c->h_ints, 16, cudaMemcpyHostToDevice, c->stream));
  CUDA_CHECK_RET(cudaMemsetAsync(f.rs_ls, 0, 72 * 4, c->stream));
  CUDA_CHECK_RET(cudaMemsetAsync(f.rs_lf, 0, 72 * 4, c->stream));
  CUDA_CHECK_RET(cudaMemsetAsync(c->d_err, 0, 4, c->stream));
  if (corner_last.n > 0) LAUNCH(c, KID_RING_OFFSETS, k_ring_offsets, (corner_last.n + 255) / 256, 256, 0, f.less_sharp, corner_last.n, f.rs_ls, c->d_err);
  if (surf_last.n > 0) LAUNCH(c, KID_RING_OFFSETS, k_ring_offsets, (surf_last.n + 255) / 256, 256, 0, f.less_flat, surf_last.n, f.rs_lf, c->d_err);
  run_grid_build(c, 1, kApiLast, corner_last.n, surf_last.n);
  CUDA_CHECK_RET(cudaMemcpyAsync(c->h_ints + 8, c->d_err, 4, cudaMemcpyDeviceToHost, c->stream));
  CUDA_CHECK_RET(cudaStreamSynchronize(c->stream));
  CUDA_CHECK_RET(cudaGetLastError());
  if (c->h_ints[8]) return ALOAM_ERR_NOT_RING_MAJOR;
  c->have_last = true;
  return ALOAM_OK;
}

static int upload_queries(aloam_ctx* c, aloam_cloud_view sharp, aloam_cloud_view flat, FeatBuf& f) {
  int rc = check_view(sharp); if (rc) return rc;
  rc = check_view(flat); if (rc) return rc;
  rc = upload_cloud(c, sharp, f.sharp, kMaxQueries); if (rc) return rc;
  rc = upload_cloud(c, flat, f.flat, kMaxQueries); if (rc) return rc;
  c->h_ints[16] = sharp.n; c->h_ints[17] = 0; c->h_ints[18] = flat.n; c->h_ints[19] = 0;
  CUDA_CHECK_RET(cudaMemcpyAsync(f.counts, c->h_ints + 16, 16, cudaMemcpyHostToDevice, c->stream));
  return ALOAM_OK;
}

int aloam_odometry_register(aloam_ctx* c, aloam_cloud_view sharp, aloam_cloud_view flat, double q[4], double t[3],
                            aloam_stats* stats) {
  if (!c || !q || !t) return ALOAM_ERR_INVALID_ARG;
  if (!c->have_last) return ALOAM_ERR_STATE;
  CUDA_CHECK_RET(cudaSetDevice(c->cfg.device));
  Lane& L = c->lanes[0];
  int rc = upload_queries(c, sharp, flat, L.feat[kApiCur]); if (rc) return rc;
  for (int k = 0; k < 4; ++k) c->h_dbl[k] = q[k];
  for (int k = 0; k < 3; ++k) c->h_dbl[4 + k] = t[k];
  CUDA_CHECK_RET(cudaEventRecord(c->ev0, c->stream));
  CUDA_CHECK_RET(cudaMemcpyAsync(c->d_api_pose, c->h_dbl, 56, cudaMemcpyHostToDevice, c->stream));
  run_register(c, 1, kApiCur, kApiLast, sharp.n, flat.n, false, false, nullptr, c->d_api_pose);
  CUDA_CHECK_RET(cudaMemcpyAsync(c->h_dbl + 8, c->d_api_pose, 56, cudaMemcpyDeviceToHost, c->stream));
  CUDA_CHECK_RET(cudaMemcpyAsync(c->h_summary, L.d_summary, sizeof(LmSummary) * 4, cudaMemcpyDeviceToHost, c->stream));
  CUDA_CHECK_RET(cudaEventRecord(c->ev1, c->stream));
  CUDA_CHECK_RET(cudaStreamSynchronize(c->stream));
  CUDA_CHECK_RET(cudaGetLastError());
  prof_collect(c);
  for (int k = 0; k < 4; ++k) q[k] = c->h_dbl[8 + k];
  for (int k = 0; k < 3; ++k) t[k] = c->h_dbl[12 + k];
  float ms = 0; cudaEventElapsedTime(&ms, c->ev0, c->ev1);
  fill_stats(c, stats, c->cfg.outer_iters, 0, ms);
  return ALOAM_OK;
}

int aloam_odometry_associate(aloam_ctx* c, aloam_cloud_view sharp, aloam_cloud_view flat, const double q[4], const double t[3],
                             int* corner_corr, int* plane_corr) {
  if (!c || !q || !t) return ALOAM_ERR_INVALID_ARG;
  if (!c->have_last) return ALOAM_ERR_STATE;
  CUDA_CHECK_RET(cudaSetDevice(c->cfg.device));
  Lane& L = c->lanes[0];
  FeatBuf& cur = L.feat[kApiCur];
  int rc = upload_queries(c, sharp, flat, cur); if (rc) return rc;
  for (int k = 0; k < 4; ++k) c->h_dbl[k] = q[k];
  for (int k = 0; k < 3; ++k) c->h_dbl[4 + k] = t[k];
  CUDA_CHECK_RET(cudaMemcpyAsync(c->d_api_pose, c->h_dbl, 56, cudaMemcpyHostToDevice, c->stream));
  OdomParams op{c->cfg.dist_sq_thresh, c->cfg.nearby_scan, c->cfg.distortion};
  const int slots = sharp.n + flat.n;
  if (slots > 0) {
    Batch<AssocArgs> aa = {};
    aa.a[0] = AssocArgs{cur.sharp, cur.flat, cur.counts, last_corner(L.feat[kApiLast]), last_surf(L.feat[kApiLast]), c->d_api_pose, L.d_blocks, L.d_corr};
    LAUNCH(c, KID_ODOM_ASSOC, k_odom_assoc, dim3((slots + 7) / 8, 1), 256, 0, aa, op, sharp.n);
  }
  std::vector<int> h((size_t)slots * 4 + 4);
  if (slots > 0) CUDA_CHECK_RET(cudaMemcpyAsync(h.data(), L.d_corr, (size_t)slots * 16, cudaMemcpyDeviceToHost, c->stream));
  CUDA_CHECK_RET(cudaStreamSynchronize(c->stream));
  CUDA_CHECK_RET(cudaGetLastError());
  for (int i = 0; i < sharp.n && corner_corr; ++i) { corner_corr[3 * i] = h[4 * i]; corner_corr[3 * i + 1] = h[4 * i + 1]; corner_corr[3 * i + 2] = h[4 * i + 3]; }
  for (int i = 0; i < flat.n && plane_corr; ++i) {
    const int* s = &h[4 * (size_t)(sharp.n + i)];
    plane_corr[4 * i] = s[0]; plane_corr[4 * i + 1] = s[1]; plane_corr[4 * i + 2] = s[2]; plane_corr[4 * i + 3] = s[3];
  }
  return ALOAM_OK;
}

// ------------------------------------------------------------------------------------------------ fused pipeline
static int scan_to_pose_impl(aloam_ctx* c, const float* d_raw, int n, int stride, double q_w[4], double t_w[3], aloam_stats* stats) {
  Lane& L = c->lanes[0];
  const int cur = c->frame % kFeatSlots, last = (c->frame + kFeatSlots - 1) % kFeatSlots;
  const int slot = c->parity;
  int rc = run_features(c, 1, &d_raw, &n, stride, cur);
  if (rc) return rc;
  int flags = 0;
  // The search index over this scan's less-sharp / less-flat clouds (what replaces the kd-tree rebuild, laserOdometry.cpp:567-568)
  // is needed by the NEXT scan only: it is built on the index stream while this scan's association + LM run on the main stream, and
  // the call returns the pose without waiting for it (the next call, or aloam_scan_stream, waits on ev_idx).
  {
    StreamGuard guard(c);
    CUDA_CHECK_RET(cudaEventRecord(c->ev_feat[cur], c->stream));
    CUDA_CHECK_RET(cudaStreamWaitEvent(c->s_idx, c->ev_feat[cur], 0));
    if (!c->prof_on) c->stream = c->s_idx;   // (the per-kernel profiler times everything on one stream)
    run_grid_build(c, 1, cur, 64 * kMaxLessSharpPerRing, std::min(n, c->max_points));
    CUDA_CHECK_RET(cudaEventRecord(c->ev_idx[cur], c->stream));
  }
  if (c->frame == 0) {
    flags |= ALOAM_FLAG_INITIALISED_ONLY;  // laserOdometry.cpp:267-271
  } else {
    CUDA_CHECK_RET(cudaStreamWaitEvent(c->stream, c->ev_idx[last], 0));   // the previous scan's index (built during the previous call)
    run_register(c, 1, cur, last, kFusedSharpSlots, kFusedFlatSlots, true, false, nullptr);
  }
  CUDA_CHECK_RET(cudaEventRecord(c->ev_odo[cur], c->stream));
  CUDA_CHECK_RET(cudaMemcpyAsync(c->h_dbl + 16, L.d_world, 56, cudaMemcpyDeviceToHost, c->stream));
  CUDA_CHECK_RET(cudaMemcpyAsync(c->h_summary, L.d_summary, sizeof(LmSummary) * 4, cudaMemcpyDeviceToHost, c->stream));
  CUDA_CHECK_RET(cudaMemcpyAsync(c->h_sc, L.d_sc + slot, sizeof(ScanScalars), cudaMemcpyDeviceToHost, c->stream));
  CUDA_CHECK_RET(cudaEventRecord(c->ev1, c->stream));
  CUDA_CHECK_RET(cudaStreamSynchronize(c->stream));
  CUDA_CHECK_RET(cudaGetLastError());
  prof_collect(c);
  if (c->h_sc->error) {
    int e = c->h_sc->error;
    CUDA_CHECK_RET(cudaMemset(&(L.d_sc + slot)->error, 0, 4));
    return e;
  }
  if (c->h_sc->first_valid == INT32_MAX) return ALOAM_ERR_EMPTY_CLOUD;
  c->last_n_full = c->h_sc->n_full;
  for (int k = 0; k < 4; ++k) q_w[k] = c->h_dbl[16 + k];
  for (int k = 0; k < 3; ++k) t_w[k] = c->h_dbl[20 + k];
  float ms = 0; cudaEventElapsedTime(&ms, c->ev0, c->ev1);
  if (c->frame == 0) { if (stats) { std::memset(stats, 0, sizeof(*stats)); stats->flags = flags; stats->ms_total = ms; } }
  else fill_stats(c, stats, c->cfg.outer_iters, flags, ms);
  c->cur = cur;
  c->frame++;
  return ALOAM_OK;
}

int aloam_scan_to_pose(aloam_ctx* c, aloam_cloud_view raw, double q_w[4], double t_w[3], aloam_stats* stats) {
  if (!c || !q_w || !t_w) return ALOAM_ERR_INVALID_ARG;
  int rc = check_view(raw); if (rc) return rc;
  if (raw.n == 0) return ALOAM_ERR_EMPTY_CLOUD;
  if (raw.n > c->max_points) return ALOAM_ERR_CAPACITY;
  CUDA_CHECK_RET(cudaSetDevice(c->cfg.device));
  CUDA_CHECK_RET(cudaEventRecord(c->ev0, c->stream));
  CUDA_CHECK_RET(cudaMemcpyAsync(c->lanes[0].d_raw[0], raw.data, (size_t)raw.n * raw.stride_floats * 4, cudaMemcpyHostToDevice, c->stream));
  return scan_to_pose_impl(c, c->lanes[0].d_raw[0], raw.n, raw.stride_floats, q_w, t_w, stats);
}

int aloam_scan_to_pose_device(aloam_ctx* c, const float* d_raw, int n, double q_w[4], double t_w[3], aloam_stats* stats) {
  if (!c || !q_w || !t_w || !d_raw) return ALOAM_ERR_INVALID_ARG;
  if (n <= 0) return ALOAM_ERR_EMPTY_CLOUD;
  if (n > c->max_points) return ALOAM_ERR_CAPACITY;
  CUDA_CHECK_RET(cudaSetDevice(c->cfg.device));
  CUDA_CHECK_RET(cudaEventRecord(c->ev0, c->stream));
  return scan_to_pose_impl(c, d_raw, n, 4, q_w, t_w, stats);
}

// registered full-resolution clouds of aloam_scan_stream_mapped_registered
struct RegisteredOut {
  float* points;         // device or page-locked host memory
  long long capacity;    // in points
  long long* offsets;    // [n_scans + 1], host
};

// the stream buffers of the registered clouds, created on first use (contexts that never ask for them do not grow)
static int ensure_registered_buffers(aloam_ctx* c) {
  if (c->s_reg) return ALOAM_OK;
  bool ok = dalloc(&c->d_reg_off, (size_t)kMaxStreamScans + 1) == cudaSuccess;
  for (Pt4*& p : c->d_reg_full) ok = ok && dalloc(&p, (size_t)c->max_points) == cudaSuccess;
  for (cudaEvent_t& e : c->ev_regcopy) ok = ok && cudaEventCreateWithFlags(&e, cudaEventDisableTiming) == cudaSuccess;
  for (cudaEvent_t& e : c->ev_regdone) ok = ok && cudaEventCreateWithFlags(&e, cudaEventDisableTiming) == cudaSuccess;
  for (cudaEvent_t& e : c->ev_fullfree) ok = ok && cudaEventCreateWithFlags(&e, cudaEventDisableTiming) == cudaSuccess;
  ok = ok && cudaStreamCreateWithFlags(&c->s_reg, cudaStreamNonBlocking) == cudaSuccess;
  if (!ok) {   // keep nothing half-built: the next call tries again
    cudaGetLastError();
    if (c->s_reg) cudaStreamDestroy(c->s_reg);
    c->s_reg = nullptr;
    for (cudaEvent_t* es : {c->ev_regcopy, c->ev_regdone}) for (int i = 0; i < kFeatSlots; ++i) { if (es[i]) cudaEventDestroy(es[i]); es[i] = nullptr; }
    for (cudaEvent_t& e : c->ev_fullfree) { if (e) cudaEventDestroy(e); e = nullptr; }
    for (Pt4*& p : c->d_reg_full) { if (p) cudaFree(p); p = nullptr; }
    if (c->d_reg_off) cudaFree(c->d_reg_off);
    c->d_reg_off = nullptr;
    return ALOAM_ERR_CUDA;
  }
  return ALOAM_OK;
}

// Pipelined form of aloam_scan_to_pose for a sequence of scans of `nb` trajectories in lockstep: ring binning of scan k+1
// (s_exa), per-ring extraction (s_ext), compaction + index build (s_idx) run concurrently with association + LM of scan k
// (main stream) and the host->device copies of scan k+2 (s_h2d) -- the overlap the reference gets from its three ROS
// processes.  Every launch covers all nb trajectories.  Results are identical to calling aloam_scan_to_pose once per scan
// and trajectory.  raws / poses are scan-major: entry k * nb + b.
static int scan_stream_impl(aloam_ctx* c, const aloam_cloud_view* raws, int n_scans, int nb, int device_resident, double* poses, aloam_stats* stats_last,
                            double* map_poses = nullptr, const RegisteredOut* reg = nullptr) {
  if (map_poses && (nb != 1 || !c || c->cfg.max_map_points <= 0)) return ALOAM_ERR_INVALID_ARG;
  if (reg && (!map_poses || !reg->points || !reg->offsets || reg->capacity < 0)) return ALOAM_ERR_INVALID_ARG;
  if (!c || !raws || !poses || n_scans < 1 || nb < 1 || nb > c->n_lanes || (long long)n_scans * nb > kMaxStreamScans) return ALOAM_ERR_INVALID_ARG;
  for (int k = 0; k < n_scans * nb; ++k) {
    int rc = check_view(raws[k]); if (rc) return rc;
    if (raws[k].n == 0) return ALOAM_ERR_EMPTY_CLOUD;
    if (raws[k].n > c->max_points) return ALOAM_ERR_CAPACITY;
    if (device_resident && raws[k].stride_floats != 4) return ALOAM_ERR_INVALID_ARG;
    if (raws[k].stride_floats != raws[k - k % nb].stride_floats) return ALOAM_ERR_INVALID_ARG;   // one stride per step
  }
  CUDA_CHECK_RET(cudaSetDevice(c->cfg.device));
  Pt4* reg_out = nullptr;
  if (reg) {
    // the clouds are written by a kernel: device memory of this context's GPU, or page-locked host memory it can address
    cudaPointerAttributes pa;
    if (cudaPointerGetAttributes(&pa, reg->points) != cudaSuccess) { cudaGetLastError(); return ALOAM_ERR_INVALID_ARG; }
    const bool dev = (pa.type == cudaMemoryTypeDevice || pa.type == cudaMemoryTypeManaged) && pa.device == c->cfg.device;
    if (!(dev || pa.type == cudaMemoryTypeHost) || !pa.devicePointer) return ALOAM_ERR_INVALID_ARG;
    reg_out = static_cast<Pt4*>(pa.devicePointer);
    int rc = ensure_registered_buffers(c); if (rc) return rc;
  }
  if (map_poses && !c->mapper) { int rc = aloam_mapper_reset(c); if (rc) return rc; }   // creates the cube store
  StreamGuard guard(c);
  cudaStream_t s_main = c->stream;
  const auto host_t0 = std::chrono::steady_clock::now();
  // on any failure: drain everything, clear the sticky device errors and forget the odometry state (a partially issued
  // pipeline cannot be rolled back scan by scan)
  auto fail = [&](int code) {
    sync_all_streams(c);
    cudaGetLastError();
    for (Lane& L : c->lanes) for (int b = 0; b < 3; ++b) cudaMemset(&(L.d_sc + b)->error, 0, 4);
    c->stream = s_main;
    aloam_reset_odometry(c);
    return code;
  };
#define STREAM_TRY(expr) do { cudaError_t _e = (expr); if (_e != cudaSuccess) { fprintf(stderr, "[aloam_b200] CUDA error %s at %s:%d\n", cudaGetErrorName(_e), __FILE__, __LINE__); return fail(ALOAM_ERR_CUDA); } } while (0)
  STREAM_TRY(cudaEventRecord(c->ev0, s_main));
  // everything issued on the main stream before this call (reset, earlier calls) is ordered before the side streams.
  // Waiting on an event that was never recorded, or whose work finished in an earlier call, is a no-op -- so the
  // per-scan waits below need no "first iterations" special cases.
  for (cudaStream_t s : {c->s_h2d, c->s_exa, c->s_ext, c->s_idx, c->s_map}) STREAM_TRY(cudaStreamWaitEvent(s, c->ev0, 0));
  if (reg) STREAM_TRY(cudaStreamWaitEvent(c->s_reg, c->ev0, 0));
  const float* d_raw[ALOAM_MAX_BATCH];
  int ns[ALOAM_MAX_BATCH];
  for (int k = 0; k < n_scans; ++k) {
    const int f = c->frame;                 // global frame number of this step
    const int b = k & 1;                    // raw / ring-major double buffer
    const int cur = f % kFeatSlots, last = (f + kFeatSlots - 1) % kFeatSlots;
    const aloam_cloud_view* rv = raws + (size_t)k * nb;
    int nmax = 0;
    for (int l = 0; l < nb; ++l) { ns[l] = rv[l].n; nmax = std::max(nmax, rv[l].n); }
    if (device_resident) {
      for (int l = 0; l < nb; ++l) d_raw[l] = rv[l].data;
    } else {
      STREAM_TRY(cudaStreamWaitEvent(c->s_h2d, c->ev_rawfree[b], 0));   // stage A of scan k-2 has consumed the buffers
      for (int l = 0; l < nb; ++l) {
        STREAM_TRY(cudaMemcpyAsync(c->lanes[l].d_raw[b], rv[l].data, (size_t)rv[l].n * rv[l].stride_floats * 4, cudaMemcpyHostToDevice, c->s_h2d));
        d_raw[l] = c->lanes[l].d_raw[b];
      }
      STREAM_TRY(cudaEventRecord(c->ev_h2d[b], c->s_h2d));
      STREAM_TRY(cudaStreamWaitEvent(c->s_exa, c->ev_h2d[b], 0));
    }
    // ---- stage A (ring binning) on s_exa: needs full[b] free, i.e. stage B of scan k-2 done
    STREAM_TRY(cudaStreamWaitEvent(c->s_exa, c->ev_b[b], 0));
    if (reg) STREAM_TRY(cudaStreamWaitEvent(c->s_exa, c->ev_fullfree[b], 0));   // stage C of scan k-2 has copied full[b] out
    c->stream = c->s_exa;
    int sc_slot = 0;
    int rc = run_features_a(c, nb, d_raw, ns, device_resident ? 4 : rv[0].stride_floats, b, &sc_slot, c->d_scan_nfull + (size_t)k * nb);
    if (rc) return fail(rc);
    if (!device_resident) STREAM_TRY(cudaEventRecord(c->ev_rawfree[b], c->s_exa));
    STREAM_TRY(cudaEventRecord(c->ev_a[b], c->s_exa));
    // ---- stage B (k_ring_features, the longest kernel) on s_ext: needs stage A of this scan and the staging set b free
    //      (its previous content was consumed by the compaction of scan k-2)
    c->stream = c->s_ext;
    STREAM_TRY(cudaStreamWaitEvent(c->s_ext, c->ev_a[b], 0));
    STREAM_TRY(cudaStreamWaitEvent(c->s_ext, c->ev_cmp[b], 0));
    rc = run_features_b1(c, nb, b, sc_slot);
    if (rc) return fail(rc);
    STREAM_TRY(cudaEventRecord(c->ev_b[b], c->s_ext));
    // ---- stage C on s_idx: ring-ordered compaction into feat[f % kFeatSlots] -- that slot was last read by the odometry
    //      of frame f - (kFeatSlots - 1) as its "last" clouds -- then the search index over its less-sharp / less-flat
    //      clouds, which only the NEXT scan's odometry needs
    c->stream = c->s_idx;
    STREAM_TRY(cudaStreamWaitEvent(c->s_idx, c->ev_b[b], 0));
    STREAM_TRY(cudaStreamWaitEvent(c->s_idx, c->ev_odo[(f + 1) % kFeatSlots], 0));
    STREAM_TRY(cudaStreamWaitEvent(c->s_idx, c->ev_mapdone[cur], 0));   // the scan-to-map stage of frame f - kFeatSlots has read this slot
    rc = run_features_b2(c, nb, b, cur, false);
    if (rc) return fail(rc);
    STREAM_TRY(cudaEventRecord(c->ev_cmp[b], c->s_idx));
    STREAM_TRY(cudaEventRecord(c->ev_feat[cur], c->s_idx));
    run_grid_build(c, nb, cur, 64 * kMaxLessSharpPerRing, std::min(nmax, c->max_points));
    STREAM_TRY(cudaEventRecord(c->ev_idx[cur], c->s_idx));
    if (reg) {
      // the ring-major cloud outlives full[b] (stage A of scan k+2 overwrites it) in slot `cur`, free once the registered cloud
      // of frame f - kFeatSlots has been written
      STREAM_TRY(cudaStreamWaitEvent(c->s_idx, c->ev_regdone[cur], 0));
      map_out_stage_full(c, c->lanes[0].d_full[b], c->d_scan_nfull + k, nmax, k, c->d_reg_full[cur], c->d_reg_off);
      STREAM_TRY(cudaEventRecord(c->ev_fullfree[b], c->s_idx));
      STREAM_TRY(cudaEventRecord(c->ev_regcopy[cur], c->s_idx));
    }
    c->stream = s_main;
    // ---- association + LM on the main stream: this scan's sharp / flat points, the previous scan's clouds + index
    STREAM_TRY(cudaStreamWaitEvent(s_main, c->ev_feat[cur], 0));
    STREAM_TRY(cudaStreamWaitEvent(s_main, c->ev_idx[last], 0));
    // the last solve of the scan writes the integrated world pose into its slot of d_poses (no copy on the critical chain)
    double* slots = c->d_poses + (size_t)k * nb * 7;
    if (f > 0) run_register(c, nb, cur, last, kFusedSharpSlots, kFusedFlatSlots, true, false, slots);
    else for (int l = 0; l < nb; ++l) STREAM_TRY(cudaMemcpyAsync(slots + (size_t)l * 7, c->lanes[l].d_world, 56, cudaMemcpyDeviceToDevice, s_main));
    STREAM_TRY(cudaEventRecord(c->ev_odo[cur], s_main));
    if (map_poses) {
      // ---- scan-to-map on s_map (laserMapping.cpp process()): the scan's less-sharp / less-flat clouds and its odometry pose go
      //      to the mapping stage on the device -- what the reference ships through /laser_cloud_corner_last, /laser_cloud_surf_last
      //      and /laser_odom_to_init (laserOdometry.cpp:570-591 -> laserMapping.cpp:278-288) never leaves HBM
      STREAM_TRY(cudaStreamWaitEvent(c->s_map, c->ev_odo[cur], 0));
      c->stream = c->s_map;
      const FeatBuf& fc = c->lanes[0].feat[cur];
      rc = mapper_step_device(c, fc.less_sharp, fc.counts + 1, 64 * kMaxLessSharpPerRing, fc.less_flat, fc.counts + 3, std::min(nmax, c->max_points),
                              c->d_poses + (size_t)k * 7, c->d_map_poses + (size_t)k * 7);
      if (rc) return fail(rc);
      STREAM_TRY(cudaEventRecord(c->ev_mapdone[cur], c->s_map));
      if (reg) {
        // /velodyne_cloud_registered (laserMapping.cpp:838-848) with this frame's refined pose, beside the next frames' mapping
        STREAM_TRY(cudaStreamWaitEvent(c->s_reg, c->ev_mapdone[cur], 0));
        STREAM_TRY(cudaStreamWaitEvent(c->s_reg, c->ev_regcopy[cur], 0));
        c->stream = c->s_reg;
        map_out_register(c, c->d_reg_full[cur], c->d_scan_nfull + k, nmax, c->d_reg_off + k, reg->capacity, c->d_map_poses + (size_t)k * 7, reg_out);
        STREAM_TRY(cudaEventRecord(c->ev_regdone[cur], c->s_reg));
      }
      c->stream = s_main;
    }
    c->cur = cur;
    c->frame++;
  }
  if (getenv("ALOAM_DEBUG_TIMING")) fprintf(stderr, "[aloam_b200] scan_stream: host issued %d x %d scans in %.1f us (%.1f us / step)\n", n_scans, nb,
      std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - host_t0).count(),
      std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - host_t0).count() / n_scans);
  const size_t total = (size_t)n_scans * nb;
  STREAM_TRY(cudaMemcpyAsync(c->h_poses, c->d_poses, total * 56, cudaMemcpyDeviceToHost, s_main));
  if (map_poses) {
    STREAM_TRY(cudaStreamWaitEvent(s_main, c->ev_mapdone[c->cur], 0));
    STREAM_TRY(cudaMemcpyAsync(c->h_poses + (size_t)kMaxStreamScans * 7, c->d_map_poses, total * 56, cudaMemcpyDeviceToHost, s_main));
  }
  for (int l = 0; l < nb; ++l) {
    STREAM_TRY(cudaMemcpyAsync(c->h_summary + 4 * l, c->lanes[l].d_summary, sizeof(LmSummary) * 4, cudaMemcpyDeviceToHost, s_main));
    STREAM_TRY(cudaMemcpyAsync(c->h_sc + 3 * l, c->lanes[l].d_sc, 3 * sizeof(ScanScalars), cudaMemcpyDeviceToHost, s_main));
  }
  STREAM_TRY(cudaEventRecord(c->ev1, s_main));
  STREAM_TRY(cudaStreamSynchronize(s_main));
  // the ring-binning stream has produced every n_full by now (the odometry of the last scan depends on it)
  STREAM_TRY(cudaMemcpyAsync(c->h_scan_nfull, c->d_scan_nfull, total * 4, cudaMemcpyDeviceToHost, s_main));
  sync_all_streams(c);
  STREAM_TRY(cudaGetLastError());
#undef STREAM_TRY
  prof_collect(c);
  for (int l = 0; l < nb; ++l)
    for (int b = 0; b < 3; ++b)
      if (c->h_sc[3 * l + b].error) return fail(c->h_sc[3 * l + b].error);
  for (size_t i = 0; i < total; ++i)
    if (c->h_scan_nfull[i] <= 0) return fail(ALOAM_ERR_EMPTY_CLOUD);   // scanRegistration.cpp:136-137 left nothing of this scan
  std::memcpy(poses, c->h_poses, total * 56);
  if (map_poses) std::memcpy(map_poses, c->h_poses + (size_t)kMaxStreamScans * 7, total * 56);
  float ms = 0; cudaEventElapsedTime(&ms, c->ev0, c->ev1);
  if (stats_last) {
    for (int l = 0; l < nb; ++l) {
      if (c->frame <= 1) { std::memset(&stats_last[l], 0, sizeof(aloam_stats)); stats_last[l].flags = ALOAM_FLAG_INITIALISED_ONLY; stats_last[l].ms_total = ms; }
      else fill_stats_from(c->h_summary + 4 * l, &stats_last[l], c->cfg.outer_iters, 0, ms);
    }
  }
  if (reg) {   // the same prefix sum the device ran; scans that end beyond the capacity were not written
    reg->offsets[0] = 0;
    for (int k = 0; k < n_scans; ++k) reg->offsets[k + 1] = reg->offsets[k] + c->h_scan_nfull[k];
    if (reg->offsets[n_scans] > reg->capacity && stats_last) stats_last->flags |= ALOAM_FLAG_OUTPUT_TRUNCATED;
  }
  return ALOAM_OK;
}

int aloam_scan_stream(aloam_ctx* c, const aloam_cloud_view* raws, int n_scans, int device_resident, double* poses, aloam_stats* stats_last) {
  return scan_stream_impl(c, raws, n_scans, 1, device_resident, poses, stats_last);
}

int aloam_scan_stream_mapped(aloam_ctx* c, const aloam_cloud_view* raws, int n_scans, int device_resident, double* odom_poses, double* map_poses,
                             aloam_stats* stats_last) {
  if (!map_poses) return ALOAM_ERR_INVALID_ARG;
  return scan_stream_impl(c, raws, n_scans, 1, device_resident, odom_poses, stats_last, map_poses);
}

int aloam_scan_stream_mapped_registered(aloam_ctx* c, const aloam_cloud_view* raws, int n_scans, int device_resident, double* odom_poses, double* map_poses,
                                        float* registered, long long capacity_points, long long* offsets, aloam_stats* stats_last) {
  if (!map_poses) return ALOAM_ERR_INVALID_ARG;
  const RegisteredOut reg{registered, capacity_points, offsets};
  return scan_stream_impl(c, raws, n_scans, 1, device_resident, odom_poses, stats_last, map_poses, &reg);
}

int aloam_scan_stream_batch(aloam_ctx* c, const aloam_cloud_view* raws, int n_scans, int batch, int device_resident, double* poses,
                            aloam_stats* stats_last) {
  return scan_stream_impl(c, raws, n_scans, batch, device_resident, poses, stats_last);
}

// ------------------------------------------------------------------------------------------------ fine-grained
int aloam_knn(aloam_ctx* c, int which, aloam_cloud_view queries, int k, int* idx, float* sqdist) {
  if (!c || !idx || !sqdist || k < 1) return ALOAM_ERR_INVALID_ARG;
  int rc = check_view(queries); if (rc) return rc;
  CUDA_CHECK_RET(cudaSetDevice(c->cfg.device));
  if (which == 0 || which == 1) {
    if (!c->have_last) return ALOAM_ERR_STATE;
    if (k != 1) return ALOAM_ERR_INVALID_ARG;  // the reference only asks for k = 1 on these trees (laserOdometry.cpp:302,390)
    rc = upload_cloud(c, queries, c->d_query, c->max_points); if (rc) return rc;
    if (queries.n > 0) {
      const FeatBuf& f0 = c->lanes[0].feat[kApiLast];
      LastCloud L = which == 0 ? last_corner(f0) : last_surf(f0);
      LAUNCH(c, KID_KNN_LAST, k_knn_last, (queries.n + 7) / 8, 256, 0, L, c->d_query, queries.n, c->d_knn_idx, c->d_knn_d);
      CUDA_CHECK_RET(cudaMemcpyAsync(idx, c->d_knn_idx, (size_t)queries.n * 4, cudaMemcpyDeviceToHost, c->stream));
      CUDA_CHECK_RET(cudaMemcpyAsync(sqdist, c->d_knn_d, (size_t)queries.n * 4, cudaMemcpyDeviceToHost, c->stream));
    }
    CUDA_CHECK_RET(cudaStreamSynchronize(c->stream));
    CUDA_CHECK_RET(cudaGetLastError());
    return ALOAM_OK;
  }
  if (which == 2 || which == 3) return aloam_map_knn_impl(c, which, queries, k, idx, sqdist);
  return ALOAM_ERR_INVALID_ARG;
}

int aloam_transform_to_end(aloam_ctx* c, aloam_cloud_view in, const double q[4], const double t[3], int distortion, aloam_cloud_view* out) {
  if (!c || !q || !t || !out) return ALOAM_ERR_INVALID_ARG;
  int rc = check_view(in); if (rc) return rc;
  if (in.n > c->max_points) return ALOAM_ERR_CAPACITY;
  CUDA_CHECK_RET(cudaSetDevice(c->cfg.device));
  out->data = reinterpret_cast<const float*>(c->h_out[0]); out->n = in.n; out->stride_floats = 4;
  if (in.n == 0) return ALOAM_OK;
  rc = upload_cloud(c, in, c->d_query, c->max_points); if (rc) return rc;
  for (int k = 0; k < 4; ++k) c->h_dbl[k] = q[k];
  for (int k = 0; k < 3; ++k) c->h_dbl[4 + k] = t[k];
  CUDA_CHECK_RET(cudaMemcpyAsync(c->d_out28, c->h_dbl, 56, cudaMemcpyHostToDevice, c->stream));
  Pt4* d_out = c->lanes[0].d_full[0];
  LAUNCH(c, KID_KNN_LAST, k_transform_to_end, (in.n + 255) / 256, 256, 0, c->d_query, in.n, c->d_out28, distortion, d_out);
  CUDA_CHECK_RET(cudaMemcpyAsync(c->h_out[0], d_out, (size_t)in.n * 16, cudaMemcpyDeviceToHost, c->stream));
  CUDA_CHECK_RET(cudaStreamSynchronize(c->stream));
  CUDA_CHECK_RET(cudaGetLastError());
  return ALOAM_OK;
}

static int run_lm_api(aloam_ctx* c, const double* blocks, int n_blocks, const double x[7], int mode) {
  if (n_blocks < 0 || n_blocks > 2 * kMaxQueries) return ALOAM_ERR_CAPACITY;
  Lane& L = c->lanes[0];
  if (n_blocks > 0) {
    CUDA_CHECK_RET(cudaMemcpyAsync(c->d_packed, blocks, (size_t)n_blocks * 11 * 8, cudaMemcpyHostToDevice, c->stream));
    LAUNCH(c, KID_PACK_BLOCKS, k_pack_blocks, (n_blocks + 255) / 256, 256, 0, c->d_packed, n_blocks, L.d_blocks);
  }
  for (int k = 0; k < 7; ++k) c->h_dbl[k] = x[k];
  CUDA_CHECK_RET(cudaMemcpyAsync(c->d_api_pose, c->h_dbl, 56, cudaMemcpyHostToDevice, c->stream));
  launch_lm(c, false, (const BlockRec*)L.d_blocks, (const int*)nullptr, n_blocks, c->d_api_pose, lm_params(c->cfg), L.d_summary, mode,
            c->d_out28, (double*)nullptr, 0, true /* blocks from the caller may carry any interpolation ratio */);
  CUDA_CHECK_RET(cudaMemcpyAsync(c->h_dbl + 8, c->d_api_pose, 56, cudaMemcpyDeviceToHost, c->stream));
  CUDA_CHECK_RET(cudaMemcpyAsync(c->h_dbl + 32, c->d_out28, 28 * 8, cudaMemcpyDeviceToHost, c->stream));
  CUDA_CHECK_RET(cudaMemcpyAsync(c->h_summary, L.d_summary, sizeof(LmSummary), cudaMemcpyDeviceToHost, c->stream));
  CUDA_CHECK_RET(cudaStreamSynchronize(c->stream));
  CUDA_CHECK_RET(cudaGetLastError());
  return ALOAM_OK;
}

int aloam_normal_equations(aloam_ctx* c, const double* blocks, int n_blocks, const double x[7], double JtJ[36], double Jtr[6],
                           double* cost) {
  if (!c || !x || !JtJ || !Jtr || (n_blocks > 0 && !blocks)) return ALOAM_ERR_INVALID_ARG;
  CUDA_CHECK_RET(cudaSetDevice(c->cfg.device));
  int rc = run_lm_api(c, blocks, n_blocks, x, 1);
  if (rc) return rc;
  const double* o = c->h_dbl + 32;
  int k = 0;
  for (int a = 0; a < 6; ++a)
    for (int b = a; b < 6; ++b) { JtJ[6 * a + b] = o[k]; JtJ[6 * b + a] = o[k]; ++k; }
  for (int a = 0; a < 6; ++a) Jtr[a] = o[21 + a];
  if (cost) *cost = o[27];
  return ALOAM_OK;
}

int aloam_solve(aloam_ctx* c, const double* blocks, int n_blocks, double x[7], double summary7[7], double* trace, int max_trace,
                int* trace_rows) {
  if (!c || !x || (n_blocks > 0 && !blocks)) return ALOAM_ERR_INVALID_ARG;
  CUDA_CHECK_RET(cudaSetDevice(c->cfg.device));
  int rc = run_lm_api(c, blocks, n_blocks, x, 0);
  if (rc) return rc;
  for (int k = 0; k < 7; ++k) x[k] = c->h_dbl[8 + k];
  const LmSummary& s = c->h_summary[0];
  if (summary7) {
    summary7[0] = s.termination; summary7[1] = s.num_iterations; summary7[2] = s.num_successful; summary7[3] = s.num_jac_evals;
    summary7[4] = 0; summary7[5] = s.initial_cost; summary7[6] = s.final_cost;
  }
  int rows = 0;
  if (trace)
    for (; rows < s.trace_rows && rows < max_trace; ++rows) std::memcpy(trace + (size_t)rows * 8, s.trace[rows], 64);
  if (trace_rows) *trace_rows = rows;
  return ALOAM_OK;
}

// ------------------------------------------------------------------------------------------------ profiling hooks
int aloam_profile_enable(aloam_ctx* c, int on) {
  if (!c) return ALOAM_ERR_INVALID_ARG;
  c->prof_on = on != 0;
  c->prof_n = 0;
  for (int k = 0; k < ALOAM_N_KERNEL_IDS; ++k) { c->prof_ms[k] = 0; c->prof_cnt[k] = 0; }
  return ALOAM_OK;
}
int aloam_profile_read(aloam_ctx* c, double* ms_sum, long long* count, const char** names, int capacity) {
  if (!c) return ALOAM_ERR_INVALID_ARG;
  int n = capacity < ALOAM_N_KERNEL_IDS ? capacity : ALOAM_N_KERNEL_IDS;
  for (int k = 0; k < n; ++k) { if (ms_sum) ms_sum[k] = c->prof_ms[k]; if (count) count[k] = c->prof_cnt[k]; if (names) names[k] = kKernelNames[k]; }
  return n;
}
long long aloam_launch_count(aloam_ctx* c) { return c ? c->launches : 0; }
// SM-clock cycle counts of the LM solves of the last register / scan_to_pose call: out[5*it] = whole solve, [5*it+1] = evaluation passes, ...
int aloam_debug_lm_cycles(aloam_ctx* c, long long* out, int outer) {
  if (!c || !out) return ALOAM_ERR_INVALID_ARG;
  for (int it = 0; it < outer && it < 4; ++it) { const LmSummary& s = c->h_summary[it]; out[5 * it] = s.cyc_total; out[5 * it + 1] = s.cyc_eval; out[5 * it + 2] = s.cyc_chol; out[5 * it + 3] = s.cyc_plus; out[5 * it + 4] = s.cyc_grad; }
  return ALOAM_OK;
}
// out == NULL arms the time stamps of k_ring_features (they are off by default), otherwise reads them (65 x 8 + 12 values) and disarms
int aloam_debug_feature_cycles(aloam_ctx* c, long long* out64x8) {
  if (!c) return ALOAM_ERR_INVALID_ARG;
  cudaSetDevice(c->cfg.device);
  if (!out64x8) { features_debug_enable(1); return ALOAM_OK; }
  features_debug_cycles(out64x8);
  features_debug_enable(0);
  return ALOAM_OK;
}

// ------------------------------------------------------------------------------------------------ mapping (mapping.cu)
int aloam_map_upload_impl(aloam_ctx* c, aloam_cloud_view corner_map, aloam_cloud_view surf_map);
int aloam_mapping_register_impl(aloam_ctx* c, aloam_cloud_view corner_stack, aloam_cloud_view surf_stack, double x[7], aloam_stats* stats);
int aloam_voxel_filter_impl(aloam_ctx* c, aloam_cloud_view in, float leaf, aloam_cloud_view* out);

int aloam_map_upload(aloam_ctx* c, aloam_cloud_view corner_map, aloam_cloud_view surf_map) { return aloam_map_upload_impl(c, corner_map, surf_map); }
int aloam_mapping_register(aloam_ctx* c, aloam_cloud_view corner_stack, aloam_cloud_view surf_stack, double x[7], aloam_stats* stats) {
  return aloam_mapping_register_impl(c, corner_stack, surf_stack, x, stats);
}
int aloam_voxel_filter(aloam_ctx* c, aloam_cloud_view in, float leaf, aloam_cloud_view* out) { return aloam_voxel_filter_impl(c, in, leaf, out); }

}  // extern "C"
