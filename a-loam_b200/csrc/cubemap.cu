// Map cube store of alaserMapping and the per-frame loop around it -- replaces laserMapping.cpp:74-108 (state),
// :142-163 (pose hand-off, pointAssociateToMap), :309-550 (centre cube, ring-buffer shift, 75-cube gather, stack
// filters) and :736-801 (insertion, per-cube VoxelGrid).  SURVEY.md section 8 f-1 / f-2.
//
// Second version: the WHOLE frame runs on the device without a host synchronisation, so it can sit at the end of the scan
// stream (aloam_scan_stream_mapped) or behind the host API (aloam_mapper_step, one sync at the end to return the pose):
//   * state (T_wmap_wodom, centre offsets, cube -> slab table, per-slab counts, slab free list) lives in device memory;
//   * k_mapper_begin : transformAssociateToMap, centre cube, ring-buffer shift (the reference rotates 4851 smart pointers;
//                      here one CTA permutes the cube -> slab table, one thread per line of cubes, and returns the slabs
//                      of the cubes that scroll out to the free list), valid-cube list in the reference's i, j, k order;
//   * k_mapper_gather: the <= 75 valid cubes device-to-device into the submap, then the hash-grid build of mapping.cu;
//   * the two scan-stack filters as ONE segmented VoxelGrid (voxel.cu), the registration of mapping.cu on device views;
//   * k_mapper_update: transformUpdate, refined pose out;
//   * k_cube_ids / k_cube_insert: pointAssociateToMap + cube of the stored point, then a STABLE append (push_back order =
//                      stack order): one CTA walks the stack in chunks, warps take turns, __match_any groups the lanes of a
//                      cube and the group leader advances the cube's running end (allocating a slab from the free list
//                      for a cube that was empty) -- O(n) instead of the O(n^2 / 256) rank search of the first version;
//   * the per-cube re-filter of the valid cubes as ONE segmented VoxelGrid over up to 150 segments, in place.
// Slabs are a POOL (1024 per cloud type, 16 k corner / 64 k surf points each: 1.3 GB) handed out on the device on first
// insertion, not 4851 x 2 slabs (6.4 GB) up front.  A full slab or an exhausted pool drops the overflow and raises
// ALOAM_FLAG_CUBE_OVERFLOW instead of failing the frame (the reference grows its cubes without bound between re-filters).
#include <climits>
#include "common.cuh"
#include "ctx.h"

extern "C" {
void aloam_mapper_free_impl(aloam_ctx* c);
int aloam_map_upload_impl(aloam_ctx* c, aloam_cloud_view corner_map, aloam_cloud_view surf_map);
}

namespace {

constexpr int CW = 21, CH = 21, CD = 11, NCUBE = CW * CH * CD;   // laserCloudWidth / Height / Depth (:77-82)
constexpr int kMaxValid = 128;
constexpr int kPool = 1024;                                      // physical slabs per cloud type

struct MapperState {
  double q_wmap_wodom[4], t_wmap_wodom[3];   // :116-117
  double x[7];                               // parameters[7] of this frame: q_w_curr (xyzw), t_w_curr
  double q_wodom[4], t_wodom[3];             // odometry pose of this frame
  int cen[3];                                // laserCloudCenWidth / Height / Depth (:74-76)
  int ctr[3];                                // centerCubeI / J / K after the shift
  int n_valid;
  int valid[kMaxValid];                      // laserCloudValidInd (i + 21 j + 441 k) in the reference's loop order
  int sub_off[2][kMaxValid + 1];
  int n_sub[2];                              // gathered submap sizes (corner, surf)
  int stack_counts[4];                       // filtered stack sizes: corner, surf, total used by the registration, raw total
  int in_counts[2];                          // sizes of the incoming less-sharp / less-flat clouds (host API path)
  int flags;                                 // ALOAM_FLAG_* of this frame
  int err;                                   // bit 0: voxel index range, bit 1: slab overflow, bit 2: pool exhausted, bit 3: submap capacity
  int frames;
  int zero, sink;                            // always 0 (count of a cube without a slab) ; write-only dummy
  int free_top;                              // slabs [free_top, kPool) of free_list are free ... per type
  int free_top2;
  int slab_of[2][NCUBE];                     // cube -> slab of that type, -1 = none
  int cnt[2][kPool];                         // points per slab
  int free_list[2][kPool];
};

struct Mapper {
  int cap[2] = {0, 0};
  Pt4* d_pts[2] = {nullptr, nullptr};       // [kPool * cap] slabs
  Pt4* d_sub[2] = {nullptr, nullptr};       // gathered submap
  Pt4* d_in[2] = {nullptr, nullptr};        // host API: uploaded less-sharp / less-flat clouds
  Pt4* d_world = nullptr;                   // insertion scratch: transformed stack points
  int* d_cube = nullptr;                    //                    their cube index (-1 = outside the ring buffer)
  MapperState* d_state = nullptr;
  MapperState* h_state = nullptr;           // pinned mirror (debug / host API read-back)
  SegDesc* d_segs = nullptr;                // [ALOAM_MAX_SEGS]
  int* d_nseg = nullptr;
  int *d_off = nullptr, *d_rank0 = nullptr, *d_bbox = nullptr, *d_total = nullptr;
  SegBuffers buf;
  double* d_pose_io = nullptr;              // [14] host API: odometry pose in, refined pose out
  int max_sub = 0;
  cudaStream_t s_aux = nullptr;             // the stack filters run here, beside the submap gather + index build
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  int* d_seg_off = nullptr;                 // [2 * NCUBE + 1] aloam_mapper_export: segment offsets, then the total
  Pt4* d_export = nullptr;                  // aloam_mapper_export to host memory: grow-only staging
  size_t export_cap = 0;
  bool stepped = false;                     // a frame has run since the last reset (MapperState::x is a refined pose)
};

// ---- Eigen-order quaternion helpers (operation order of Eigen::Quaternion: the pose hand-off is compared bit for bit)
struct Qd { double x, y, z, w; };
__host__ __device__ inline Qd qmul(const Qd& a, const Qd& b) {
  Qd r;
  r.w = a.w * b.w - a.x * b.x - a.y * b.y - a.z * b.z;
  r.x = a.w * b.x + a.x * b.w + a.y * b.z - a.z * b.y;
  r.y = a.w * b.y + a.y * b.w + a.z * b.x - a.x * b.z;
  r.z = a.w * b.z + a.z * b.w + a.x * b.y - a.y * b.x;
  return r;
}
__host__ __device__ inline Qd qinv(const Qd& a) {
  const double n2 = a.x * a.x + a.y * a.y + a.z * a.z + a.w * a.w;
  return Qd{-a.x / n2, -a.y / n2, -a.z / n2, a.w / n2};
}
__host__ __device__ inline void qrot(const Qd& q, const double v[3], double o[3]) {
  double uv[3] = {q.y * v[2] - q.z * v[1], q.z * v[0] - q.x * v[2], q.x * v[1] - q.y * v[0]};
  uv[0] = uv[0] + uv[0]; uv[1] = uv[1] + uv[1]; uv[2] = uv[2] + uv[2];
  const double c2[3] = {q.y * uv[2] - q.z * uv[1], q.z * uv[0] - q.x * uv[2], q.x * uv[1] - q.y * uv[0]};
  o[0] = v[0] + q.w * uv[0] + c2[0]; o[1] = v[1] + q.w * uv[1] + c2[1]; o[2] = v[2] + q.w * uv[2] + c2[2];
}

// int((v + 25.0) / 50.0) + centre, minus one when v + 25.0 < 0   (:314-325, :741-750)
__host__ __device__ inline int cube_coord(double v, int centre) {
  int c = int((v + 25.0) / 50.0) + centre;
  if (v + 25.0 < 0) c--;
  return c;
}
__host__ __device__ inline int cube_index(int i, int j, int k) { return i + CW * j + CW * CH * k; }

// :327-509 -- one step of the ring buffer along `axis` for the line (u, v) of this thread; towards_high: every cube moves one
// index up, the top cube wraps to index 0 and is emptied (its slabs go back to the free lists)
__device__ void rotate_line(MapperState* S, int axis, bool towards_high, int u, int v) {
  const int n[3] = {CW, CH, CD};
  const int a = axis, b = (axis + 1) % 3, cc = (axis + 2) % 3;
  auto at = [&](int t) { int ijk[3]; ijk[a] = t; ijk[b] = u; ijk[cc] = v; return cube_index(ijk[0], ijk[1], ijk[2]); };
#pragma unroll
  for (int ty = 0; ty < 2; ++ty) {
    int* so = S->slab_of[ty];
    int wrapped;
    if (towards_high) {
      wrapped = so[at(n[a] - 1)];
      for (int t = n[a] - 1; t >= 1; --t) so[at(t)] = so[at(t - 1)];
      so[at(0)] = -1;
    } else {
      wrapped = so[at(0)];
      for (int t = 0; t < n[a] - 1; ++t) so[at(t)] = so[at(t + 1)];
      so[at(n[a] - 1)] = -1;
    }
    if (wrapped >= 0) {
      S->cnt[ty][wrapped] = 0;
      const int slot = atomicSub(ty == 0 ? &S->free_top : &S->free_top2, 1) - 1;   // push
      S->free_list[ty][slot] = wrapped;
    }
  }
}

// transformAssociateToMap (:142-146), centre cube + shift (:314-509), valid cubes (:511-529), gather offsets
__global__ void __launch_bounds__(1024) k_mapper_begin(MapperState* S, const double* __restrict__ odom7, int max_sub) {
  pdl_launch_dependents();
  pdl_wait();   // may have been launched with a programmatic dependency on the previous kernel of the stream
  __shared__ int s_ctr[3], s_cen[3];
  const int tid = threadIdx.x;
  if (tid == 0) {
    const Qd qm{S->q_wmap_wodom[0], S->q_wmap_wodom[1], S->q_wmap_wodom[2], S->q_wmap_wodom[3]};
    const Qd qo{odom7[0], odom7[1], odom7[2], odom7[3]};
    const double to[3] = {odom7[4], odom7[5], odom7[6]};
    const Qd q0 = qmul(qm, qo);
    double r[3]; qrot(qm, to, r);
    S->x[0] = q0.x; S->x[1] = q0.y; S->x[2] = q0.z; S->x[3] = q0.w;
    S->x[4] = r[0] + S->t_wmap_wodom[0]; S->x[5] = r[1] + S->t_wmap_wodom[1]; S->x[6] = r[2] + S->t_wmap_wodom[2];
    S->q_wodom[0] = qo.x; S->q_wodom[1] = qo.y; S->q_wodom[2] = qo.z; S->q_wodom[3] = qo.w;
    S->t_wodom[0] = to[0]; S->t_wodom[1] = to[1]; S->t_wodom[2] = to[2];
    for (int a = 0; a < 3; ++a) { s_cen[a] = S->cen[a]; s_ctr[a] = cube_coord(S->x[4 + a], S->cen[a]); }
    S->flags = 0;
  }
  __syncthreads();
  const int dims[3] = {CW, CH, CD};
  for (int a = 0; a < 3; ++a) {
    const int nb = dims[(a + 1) % 3], nc = dims[(a + 2) % 3];
    for (;;) {   // :327-416 pattern: shift up while the centre is within 3 cubes of the low edge
      const int ctr = s_ctr[a];
      __syncthreads();
      if (!(ctr < 3)) break;
      if (tid < nb * nc) rotate_line(S, a, true, tid % nb, tid / nb);
      __syncthreads();
      if (tid == 0) { s_ctr[a]++; s_cen[a]++; }
      __syncthreads();
    }
    for (;;) {   // shift down while it is within 3 cubes of the high edge
      const int ctr = s_ctr[a];
      __syncthreads();
      if (!(ctr >= dims[a] - 3)) break;
      if (tid < nb * nc) rotate_line(S, a, false, tid % nb, tid / nb);
      __syncthreads();
      if (tid == 0) { s_ctr[a]--; s_cen[a]--; }
      __syncthreads();
    }
  }
  __shared__ int s_valid[kMaxValid], s_n[2][kMaxValid], s_nv;
  if (tid == 0) {
    for (int a = 0; a < 3; ++a) { S->cen[a] = s_cen[a]; S->ctr[a] = s_ctr[a]; }
    int nv = 0;
    for (int i = s_ctr[0] - 2; i <= s_ctr[0] + 2; ++i)
      for (int j = s_ctr[1] - 2; j <= s_ctr[1] + 2; ++j)
        for (int k = s_ctr[2] - 1; k <= s_ctr[2] + 1; ++k)
          if (i >= 0 && i < CW && j >= 0 && j < CH && k >= 0 && k < CD) s_valid[nv++] = cube_index(i, j, k);
    s_nv = nv;
    S->n_valid = nv;
  }
  __syncthreads();
  const int nv = s_nv;
  if (tid < 2 * nv) {   // the counts of the valid cubes, all loads in flight at once
    const int ty = tid >= nv, v = ty ? tid - nv : tid;
    const int s = S->slab_of[ty][s_valid[v]];
    s_n[ty][v] = s < 0 ? 0 : S->cnt[ty][s];
    if (ty == 0) S->valid[v] = s_valid[v];
  }
  __syncthreads();
  if (tid < 2) {
    const int ty = tid;
    int off = 0;
    for (int v = 0; v < nv; ++v) {
      S->sub_off[ty][v] = off;
      int n = s_n[ty][v];
      if (off + n > max_sub) { n = max_sub - off; atomicOr(&S->err, 8); }   // submap capacity: truncated, flagged
      off += n;
    }
    S->sub_off[ty][nv] = off;
    S->n_sub[ty] = off;
  }
}

// grid (valid cubes, 2 types): slab -> submap (:531-539), device to device
__global__ void __launch_bounds__(256) k_mapper_gather(const MapperState* __restrict__ S, const Pt4* __restrict__ p0, const Pt4* __restrict__ p1,
                                                       int cap0, int cap1, Pt4* __restrict__ sub0, Pt4* __restrict__ sub1) {
  pdl_launch_dependents();
  pdl_wait();   // may have been launched with a programmatic dependency on the previous kernel of the stream
  const int v = blockIdx.x, ty = blockIdx.y;
  if (v >= S->n_valid) return;
  const int s = S->slab_of[ty][S->valid[v]];
  if (s < 0) return;
  const int off = S->sub_off[ty][v], n = S->sub_off[ty][v + 1] - off;
  const Pt4* __restrict__ src = (ty ? p1 : p0) + (size_t)s * (ty ? cap1 : cap0);
  Pt4* __restrict__ dst = (ty ? sub1 : sub0) + off;
  for (int i = threadIdx.x; i < n; i += blockDim.x) dst[i] = src[i];
}

// segment descriptors of the two scan-stack filters (:543-549)
__global__ void k_seg_two(SegDesc* segs, int* n_seg, const Pt4* c_in, const int* nc, float c_leaf, Pt4* c_out, int* nc_out, const Pt4* s_in, const int* ns,
                          float s_leaf, Pt4* s_out, int* ns_out) {
  pdl_launch_dependents();
  pdl_wait();   // may have been launched with a programmatic dependency on the previous kernel of the stream
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    segs[0] = SegDesc{c_in, nc, c_leaf, c_out, nc_out};
    segs[1] = SegDesc{s_in, ns, s_leaf, s_out, ns_out};
    *n_seg = 2;
  }
}

// after the stack filters: the map-too-thin test of :554 (on the gathered submap) -> number of queries the registration sees
__global__ void k_mapper_prep(MapperState* S) {
  pdl_launch_dependents();
  pdl_wait();   // may have been launched with a programmatic dependency on the previous kernel of the stream
  if (threadIdx.x || blockIdx.x) return;
  const int total = S->stack_counts[0] + S->stack_counts[1];
  S->stack_counts[3] = total;
  const bool ok = S->n_sub[0] > 10 && S->n_sub[1] > 50;
  if (!ok) S->flags |= ALOAM_FLAG_MAP_TOO_THIN;
  S->stack_counts[2] = ok ? total : 0;   // zero residual blocks: the solve leaves the pose untouched, like the skipped optimisation
}

// transformUpdate (:148-152) ; refined pose out
__global__ void k_mapper_update(MapperState* S, double* __restrict__ out7) {
  pdl_launch_dependents();
  pdl_wait();   // may have been launched with a programmatic dependency on the previous kernel of the stream
  if (threadIdx.x || blockIdx.x) return;
  const Qd qw{S->x[0], S->x[1], S->x[2], S->x[3]};
  const Qd qo{S->q_wodom[0], S->q_wodom[1], S->q_wodom[2], S->q_wodom[3]};
  const Qd qn = qmul(qw, qinv(qo));
  double r[3]; qrot(qn, S->t_wodom, r);
  S->q_wmap_wodom[0] = qn.x; S->q_wmap_wodom[1] = qn.y; S->q_wmap_wodom[2] = qn.z; S->q_wmap_wodom[3] = qn.w;
  S->t_wmap_wodom[0] = S->x[4] - r[0]; S->t_wmap_wodom[1] = S->x[5] - r[1]; S->t_wmap_wodom[2] = S->x[6] - r[2];
  if (out7) for (int k = 0; k < 7; ++k) out7[k] = S->x[k];
  if (S->err & 6) S->flags |= ALOAM_FLAG_CUBE_OVERFLOW;
  S->frames++;
}

// parameters[7] (q_w_curr x, y, z, w ; t_w_curr) in registers
struct PoseD { double ux, uy, uz, w, tx, ty, tz; };
__device__ __forceinline__ PoseD load_pose(const double* x) { return PoseD{x[0], x[1], x[2], x[3], x[4], x[5], x[6]}; }

// pointAssociateToMap (:154-163): q_w_curr * p + t_w_curr in double, in Eigen's operation order (this file is compiled with
// -fmad=false: the bit parity with the reference depends on it), stored as float; the intensity is kept
__device__ __forceinline__ Pt4 point_associate_to_map(const Pt4& p, const PoseD& P) {
  const double vx = (double)p.x, vy = (double)p.y, vz = (double)p.z;
  double uvx = P.uy * vz - P.uz * vy, uvy = P.uz * vx - P.ux * vz, uvz = P.ux * vy - P.uy * vx;
  uvx = uvx + uvx; uvy = uvy + uvy; uvz = uvz + uvz;
  const double cx = P.uy * uvz - P.uz * uvy, cy = P.uz * uvx - P.ux * uvz, cz = P.ux * uvy - P.uy * uvx;
  Pt4 s;
  s.x = (float)(((vx + P.w * uvx) + cx) + P.tx);
  s.y = (float)(((vy + P.w * uvy) + cy) + P.ty);
  s.z = (float)(((vz + P.w * uvz) + cz) + P.tz);
  s.i = p.i;
  return s;
}

// pointAssociateToMap, then the cube of the stored point (:741-758)
// blockIdx.y = cloud (0 corner stack, 1 surf stack); the scratch of cloud 1 starts `scratch_stride` elements in
__global__ void k_cube_ids(const Pt4* __restrict__ stack0, const Pt4* __restrict__ stack1, const MapperState* __restrict__ S, Pt4* __restrict__ world,
                           int* __restrict__ cube, int scratch_stride) {
  pdl_launch_dependents();
  pdl_wait();   // may have been launched with a programmatic dependency on the previous kernel of the stream
  const int which = blockIdx.y;
  const Pt4* __restrict__ stack = which ? stack1 : stack0;
  world += (size_t)which * scratch_stride; cube += (size_t)which * scratch_stride;
  const int n = S->stack_counts[which];
  const PoseD P = load_pose(S->x);
  const int c0 = S->cen[0], c1 = S->cen[1], c2 = S->cen[2];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const Pt4 s = point_associate_to_map(stack[i], P);
    const int ci = cube_coord((double)s.x, c0), cj = cube_coord((double)s.y, c1), ck = cube_coord((double)s.z, c2);
    world[i] = s;
    cube[i] = (ci >= 0 && ci < CW && cj >= 0 && cj < CH && ck >= 0 && ck < CD) ? cube_index(ci, cj, ck) : -1;
  }
}

// stable append of the stack points to their cubes (push_back order = stack order, :759-767).  ONE CTA per cloud (blockIdx.x: the
// corner and the surf store are independent, the two appends run side by side): the stack is walked in
// chunks of 1024; inside a chunk the warps take turns, the lanes of one cube form a group (__match_any) whose leader
// advances the cube's running end in shared memory -- and takes a slab from the free list when the cube had none.
__global__ void __launch_bounds__(1024) k_cube_insert(const Pt4* __restrict__ world, const int* __restrict__ cube, int scratch_stride, MapperState* S,
                                                      Pt4* __restrict__ pts0, int cap0, Pt4* __restrict__ pts1, int cap1) {
  pdl_launch_dependents();
  pdl_wait();   // may have been launched with a programmatic dependency on the previous kernel of the stream
  const int ty = blockIdx.x;
  world += (size_t)ty * scratch_stride; cube += (size_t)ty * scratch_stride;
  Pt4* __restrict__ pts = ty ? pts1 : pts0;
  const int cap = ty ? cap1 : cap0;
  __shared__ int s_end[NCUBE];    // running end of every cube
  __shared__ int s_slab[NCUBE];   // cube -> slab (the warps' turns must not wait on global memory)
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n = S->stack_counts[ty];
  int* slab_of = S->slab_of[ty];
  int* cnt = S->cnt[ty];
  for (int c = tid; c < NCUBE; c += blockDim.x) { const int s = slab_of[c]; s_slab[c] = s; s_end[c] = s < 0 ? 0 : cnt[s]; }
  __syncthreads();
  for (int base = 0; base < n; base += 1024) {
    const int i = base + tid;
    const int mine = i < n ? cube[i] : -1;
    const Pt4 p = i < n ? world[i] : Pt4{0.f, 0.f, 0.f, 0.f};
    const int warps = min(32, (n - base + 31) / 32);
    for (int w = 0; w < warps; ++w) {
      if (warp == w) {
        const unsigned grp = __match_any_sync(0xffffffffu, mine);
        const int leader = __ffs(grp) - 1;
        int start = 0, slab = -1;
        if (mine >= 0 && lane == leader) {
          slab = s_slab[mine];
          if (slab < 0) {   // first point of an empty cube: take a slab from the pool (several group leaders of one warp may do so at once)
            int* top = ty == 0 ? &S->free_top : &S->free_top2;
            const int idx = atomicAdd(top, 1);
            if (idx < kPool) { slab = S->free_list[ty][idx]; s_slab[mine] = slab; }
            else { atomicSub(top, 1); atomicOr(&S->err, 4); }
          }
          start = s_end[mine];
          s_end[mine] = start + __popc(grp);
        }
        start = __shfl_sync(0xffffffffu, start, leader);
        slab = __shfl_sync(0xffffffffu, slab, leader);
        if (mine >= 0 && slab >= 0) {
          const int pos = start + __popc(grp & ((1u << lane) - 1u));
          if (pos < cap) pts[(size_t)slab * cap + pos] = p;
          else atomicOr(&S->err, 2);   // slab full: the overflow is dropped (flagged), the frame goes on
        }
      }
      __syncthreads();
    }
  }
  for (int c = tid; c < NCUBE; c += blockDim.x) { const int s = s_slab[c]; if (s >= 0) { slab_of[c] = s; cnt[s] = min(s_end[c], cap); } }
}

// segment descriptors of the per-cube re-filter (:770-801): every valid cube that has a slab, corner cubes then surf cubes, in place
__global__ void __launch_bounds__(256) k_seg_cubes(MapperState* S, SegDesc* segs, int* n_seg, Pt4* p0, Pt4* p1, int cap0, int cap1, float leaf0, float leaf1) {
  pdl_launch_dependents();
  pdl_wait();   // may have been launched with a programmatic dependency on the previous kernel of the stream
  const int t = threadIdx.x, nv = S->n_valid;
  if (t < 2 * nv) {
    const int ty = t >= nv, v = ty ? t - nv : t;
    const int s = S->slab_of[ty][S->valid[v]];
    Pt4* base = s < 0 ? (ty ? p1 : p0) : (ty ? p1 : p0) + (size_t)s * (ty ? cap1 : cap0);
    int* np = s < 0 ? &S->zero : &S->cnt[ty][s];
    segs[t] = SegDesc{base, np, ty ? leaf1 : leaf0, base, s < 0 ? &S->sink : np};
  }
  if (t == 0) { *n_seg = 2 * nv; S->zero = 0; }
}

// ---- map outputs (:803-848)
// segment s of a region: cube cube_of(s / 2), type s % 2 -- per cube the corner points, then the surf points (:811-812, :828-829)
__device__ __forceinline__ int region_cube(const MapperState* S, int region, int cube_pos) { return region == ALOAM_MAP_SURROUND ? S->valid[cube_pos] : cube_pos; }

// one CTA: exclusive scan of the segment sizes of `region` -> seg_off[0 .. nseg], *total = seg_off[nseg]
__global__ void __launch_bounds__(1024) k_export_offsets(const MapperState* __restrict__ S, int region, int* __restrict__ seg_off, int* __restrict__ total) {
  const int nseg = region == ALOAM_MAP_SURROUND ? 2 * S->n_valid : 2 * NCUBE;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int per = (nseg + blockDim.x - 1) / blockDim.x;
  const int s0 = min(nseg, tid * per), s1 = min(nseg, s0 + per);
  int sum = 0;
  for (int s = s0; s < s1; ++s) {
    const int ty = s & 1, slab = S->slab_of[ty][region_cube(S, region, s >> 1)];
    sum += slab < 0 ? 0 : S->cnt[ty][slab];
  }
  // block-wide exclusive scan of the per-thread sums
  int incl = sum;
  for (int d = 1; d < 32; d <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl += v; }
  __shared__ int s_warp[32];
  if (lane == 31) s_warp[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    int w = lane < (int)(blockDim.x >> 5) ? s_warp[lane] : 0;
    for (int d = 1; d < 32; d <<= 1) { const int v = __shfl_up_sync(0xffffffffu, w, d); if (lane >= d) w += v; }
    s_warp[lane] = w;
  }
  __syncthreads();
  int off = incl - sum + (warp ? s_warp[warp - 1] : 0);
  for (int s = s0; s < s1; ++s) {
    seg_off[s] = off;
    const int ty = s & 1, slab = S->slab_of[ty][region_cube(S, region, s >> 1)];
    off += slab < 0 ? 0 : S->cnt[ty][slab];
  }
  if (tid == blockDim.x - 1) { seg_off[nseg] = off; *total = off; }
}

// one CTA per segment: the points of one (cube, type) slab to out + seg_off[s]; empty segments leave at once
__global__ void __launch_bounds__(256) k_export_copy(const MapperState* __restrict__ S, int region, const int* __restrict__ seg_off, const Pt4* __restrict__ p0,
                                                     const Pt4* __restrict__ p1, int cap0, int cap1, Pt4* __restrict__ out) {
  const int s = blockIdx.x;
  const int nseg = region == ALOAM_MAP_SURROUND ? 2 * S->n_valid : 2 * NCUBE;
  if (s >= nseg) return;
  const int off = seg_off[s], n = seg_off[s + 1] - off;
  if (n == 0) return;
  const int ty = s & 1, slab = S->slab_of[ty][region_cube(S, region, s >> 1)];
  const Pt4* __restrict__ src = (ty ? p1 : p0) + (size_t)slab * (ty ? cap1 : cap0);
  for (int i = threadIdx.x; i < n; i += blockDim.x) out[off + i] = src[i];
}

// /velodyne_cloud_registered (:838-848): pointAssociateToMap of a cloud with pose x7.  n = *d_n (or n_host when d_n is null);
// the points go to out[range[0] ...] when range[1] <= capacity (range null: to out[0 .. n))
__global__ void __launch_bounds__(256) k_associate_to_map(const Pt4* __restrict__ in, const int* __restrict__ d_n, int n_host, const long long* __restrict__ range,
                                                          long long capacity, const double* __restrict__ x7, Pt4* __restrict__ out) {
  const int n = d_n ? *d_n : n_host;
  long long base = 0;
  if (range) {
    base = range[0];
    if (range[1] > capacity) return;   // this scan does not fit: the caller's buffer keeps a prefix of whole scans
  }
  const PoseD P = load_pose(x7);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) out[base + i] = point_associate_to_map(in[i], P);
}

// stage C of the registered stream: scan k's ring-major cloud to its slot buffer, and off[k + 1] = off[k] + n (off[0] = 0)
__global__ void __launch_bounds__(256) k_stage_full(const Pt4* __restrict__ full, const int* __restrict__ d_n, int k, Pt4* __restrict__ dst, long long* __restrict__ off) {
  const int n = *d_n;
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    const long long base = k ? off[k] : 0;
    if (k == 0) off[0] = 0;
    off[k + 1] = base + n;
  }
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) dst[i] = full[i];
}

int grid_for(int n) { return std::max(1, std::min((n + 255) / 256, 148 * 4)); }

int ensure_mapper(aloam_ctx* c) {
  if (c->mapper) return ALOAM_OK;
  if (c->cfg.max_map_points <= 0) return ALOAM_ERR_CAPACITY;
  Mapper* m = new (std::nothrow) Mapper();
  if (!m) return ALOAM_ERR_CUDA;
  m->cap[0] = std::min(16384, c->max_points);
  m->cap[1] = std::min(65536, c->max_points);
  m->max_sub = c->cfg.max_map_points;
  bool ok = true;
  for (int t = 0; t < 2 && ok; ++t) {
    ok = ok && cudaMalloc((void**)&m->d_pts[t], (size_t)kPool * m->cap[t] * sizeof(Pt4)) == cudaSuccess;
    ok = ok && cudaMalloc((void**)&m->d_sub[t], (size_t)m->max_sub * sizeof(Pt4)) == cudaSuccess;
    ok = ok && cudaMalloc((void**)&m->d_in[t], (size_t)c->max_points * sizeof(Pt4)) == cudaSuccess;
  }
  ok = ok && cudaMalloc((void**)&m->d_world, (size_t)2 * c->max_points * sizeof(Pt4)) == cudaSuccess;   // both stacks side by side
  ok = ok && cudaMalloc((void**)&m->d_cube, (size_t)2 * c->max_points * sizeof(int)) == cudaSuccess;
  ok = ok && cudaMalloc((void**)&m->d_state, sizeof(MapperState)) == cudaSuccess;
  ok = ok && cudaMallocHost((void**)&m->h_state, sizeof(MapperState)) == cudaSuccess;
  ok = ok && cudaMalloc((void**)&m->d_segs, ALOAM_MAX_SEGS * sizeof(SegDesc)) == cudaSuccess;
  ok = ok && cudaMalloc((void**)&m->d_nseg, 16) == cudaSuccess;
  ok = ok && cudaMalloc((void**)&m->d_off, (ALOAM_MAX_SEGS + 8) * sizeof(int)) == cudaSuccess;
  ok = ok && cudaMalloc((void**)&m->d_rank0, (ALOAM_MAX_SEGS + 8) * sizeof(int)) == cudaSuccess;
  ok = ok && cudaMalloc((void**)&m->d_bbox, ALOAM_MAX_SEGS * 6 * sizeof(int)) == cudaSuccess;
  ok = ok && cudaMalloc((void**)&m->d_total, 16) == cudaSuccess;
  ok = ok && cudaMalloc((void**)&m->d_pose_io, 16 * sizeof(double)) == cudaSuccess;
  ok = ok && cudaMalloc((void**)&m->d_seg_off, (2 * NCUBE + 2) * sizeof(int)) == cudaSuccess;
  ok = ok && cudaStreamCreateWithFlags(&m->s_aux, cudaStreamNonBlocking) == cudaSuccess;
  ok = ok && cudaEventCreateWithFlags(&m->ev_fork, cudaEventDisableTiming) == cudaSuccess && cudaEventCreateWithFlags(&m->ev_join, cudaEventDisableTiming) == cudaSuccess;
  // the re-filter sorts every point of the valid cubes (<= the submap capacity per type), the stack filter two scan clouds
  ok = ok && vox_seg_alloc(m->buf, std::max((size_t)2 * m->max_sub, (size_t)2 * c->max_points)) == ALOAM_OK;
  if (!ok) {   // publish nothing half-built
    cudaGetLastError();
    c->mapper = m; aloam_mapper_free_impl(c);
    return ALOAM_ERR_CUDA;
  }
  c->mapper = m;
  return ALOAM_OK;
}

SegFilter make_filter(Mapper* m, int idx_bits) {
  SegFilter f;
  f.seg = m->d_segs; f.n_seg = m->d_nseg; f.off = m->d_off; f.rank0 = m->d_rank0; f.bbox = m->d_bbox; f.total = m->d_total;
  f.err = &m->d_state->err; f.idx_bits = idx_bits; f.seg0 = 0; f.seg_cap = ALOAM_MAX_SEGS;
  return f;
}

}  // namespace

extern "C" void aloam_mapper_free_impl(aloam_ctx* c) {
  Mapper* m = static_cast<Mapper*>(c->mapper);
  if (!m) return;
  for (int t = 0; t < 2; ++t) { if (m->d_pts[t]) cudaFree(m->d_pts[t]); if (m->d_sub[t]) cudaFree(m->d_sub[t]); if (m->d_in[t]) cudaFree(m->d_in[t]); }
  if (m->s_aux) { cudaStreamSynchronize(m->s_aux); cudaStreamDestroy(m->s_aux); }
  if (m->ev_fork) cudaEventDestroy(m->ev_fork);
  if (m->ev_join) cudaEventDestroy(m->ev_join);
  void* ps[] = {m->d_world, m->d_cube, m->d_state, m->d_segs, m->d_nseg, m->d_off, m->d_rank0, m->d_bbox, m->d_total, m->d_pose_io, m->d_seg_off, m->d_export};
  for (void* p : ps) if (p) cudaFree(p);
  if (m->h_state) cudaFreeHost(m->h_state);
  vox_seg_free(m->buf);
  delete m;
  c->mapper = nullptr;
}

// One frame of alaserMapping's process() on the current stream, entirely on the device.  corner_last / surf_last and their
// sizes, the odometry pose (7 doubles) and the output pose slot are device pointers; n_upper_* bound the cloud sizes.
int mapper_step_device(aloam_ctx* c, const Pt4* d_corner_last, const int* d_nc, int n_upper_c, const Pt4* d_surf_last, const int* d_ns, int n_upper_s,
                       const double* d_odom7, double* d_out7) {
  int rc = ensure_mapper(c); if (rc) return rc;
  Mapper* m = static_cast<Mapper*>(c->mapper);
  MapperState* S = m->d_state;
  // the registration buffers of mapping.cu (grids, stacks, blocks) are shared with the host API
  if (!c->map_corner.grid.slots) {
    aloam_cloud_view none{nullptr, 0, 4};
    rc = aloam_map_upload_impl(c, none, none); if (rc) return rc;
  }
  // ---- stack filters (:541-550): one segmented pass for both clouds.  They read only the scan's clouds, the gather + index
  // build below only the cube store: two independent chains, the filters forked onto an auxiliary stream and joined before the
  // registration.
  {
    cudaStream_t main_stream = c->stream;
    CUDA_CHECK_RET(cudaEventRecord(m->ev_fork, main_stream));
    CUDA_CHECK_RET(cudaStreamWaitEvent(m->s_aux, m->ev_fork, 0));
    c->stream = m->s_aux;
    launch_ex(c, KID_VOXEL, k_seg_two, dim3(1), dim3(32), 0, 1, false, m->d_segs, m->d_nseg, d_corner_last, d_nc, c->cfg.line_res, c->d_stack_corner, &S->stack_counts[0], d_surf_last, d_ns,
              c->cfg.plane_res, c->d_stack_surf, &S->stack_counts[1]);
    vox_seg_filter(c, make_filter(m, 31), m->buf, 2, n_upper_c + n_upper_s, std::max(n_upper_c, n_upper_s));
    const cudaError_t e = cudaEventRecord(m->ev_join, m->s_aux);
    c->stream = main_stream;
    CUDA_CHECK_RET(e);
  }
  launch_ex(c, KID_CUBES, k_mapper_begin, dim3(1), dim3(1024), 0, 1, true, S, d_odom7, m->max_sub);
  launch_ex(c, KID_CUBES, k_mapper_gather, dim3(dim3(kMaxValid, 2)), dim3(256), 0, 1, true, (const MapperState*)S, (const Pt4*)m->d_pts[0], (const Pt4*)m->d_pts[1], m->cap[0], m->cap[1],
         m->d_sub[0], m->d_sub[1]);
  if (c->shard_count > 1) {
    // A rank of a sharded job keeps the WHOLE cube store (the insertions below are replicated: the refined pose is bit-identical
    // on every rank) but indexes and searches only its x-slabs (+ halo) of the submap; the ranks meet in the all-reduce of the
    // normal equations inside the solve.  The too-thin test of k_mapper_prep is on the whole submap, the same on every rank.
    rc = map_shard_index_device(c, m->d_sub[0], &S->n_sub[0], m->d_sub[1], &S->n_sub[1], m->max_sub, &S->err); if (rc) return rc;
  } else {
    launch_ex(c, KID_MAP_GRID, k_grid_setup, dim3(1), dim3(32), 0, 1, true, c->map_corner.grid, (const int*)&S->n_sub[0], c->map_surf.grid, (const int*)&S->n_sub[1]);
    map_index_build(c, m->d_sub[0], m->d_sub[1], m->max_sub);
  }
  c->have_map = true;
  CUDA_CHECK_RET(cudaStreamWaitEvent(c->stream, m->ev_join, 0));   // join: the filtered stacks are ready
  launch_ex(c, KID_CUBES, k_mapper_prep, dim3(1), dim3(32), 0, 1, true, S);
  // ---- optimisation (:554-733)
  const int nq_upper = std::min(n_upper_c + n_upper_s, 2 * c->max_points);
  map_register_device(c, c->d_stack_corner, c->d_stack_surf, S->stack_counts, nq_upper, S->x, false);
  launch_ex(c, KID_CUBES, k_mapper_update, dim3(1), dim3(32), 0, 1, true, S, d_out7);
  // ---- insertion (:736-767)
  const int up = std::max(n_upper_c, n_upper_s);
  launch_ex(c, KID_CUBES, k_cube_ids, dim3(std::max(1, std::min((up + 255) / 256, 148 * 2)), 2), dim3(256), 0, 1, true, (const Pt4*)c->d_stack_corner, (const Pt4*)c->d_stack_surf,
            (const MapperState*)S, m->d_world, m->d_cube, c->max_points);
  launch_ex(c, KID_CUBES, k_cube_insert, dim3(2), dim3(1024), 0, 1, true, (const Pt4*)m->d_world, (const int*)m->d_cube, c->max_points, S, m->d_pts[0], m->cap[0], m->d_pts[1], m->cap[1]);
  // ---- per-cube re-filter of the valid cubes (:770-801): one segmented pass over <= 150 cubes, in place
  launch_ex(c, KID_CUBES, k_seg_cubes, dim3(1), dim3(256), 0, 1, true, S, m->d_segs, m->d_nseg, m->d_pts[0], m->d_pts[1], m->cap[0], m->cap[1], c->cfg.line_res, c->cfg.plane_res);
  // index bits of a 50 m cube at the finer leaf: (50 / leaf + 3)^3 voxels at most (PCL itself gives up beyond 2^31)
  int cube_bits = 1;
  { const double side = std::floor(50.0 / std::min(c->cfg.line_res, c->cfg.plane_res)) + 3.0; const double cells = side * side * side;
    while (cube_bits < 31 && (double)(1ull << cube_bits) < cells) ++cube_bits; }
  vox_seg_filter(c, make_filter(m, cube_bits), m->buf, 2 * 75, (int)std::min(m->buf.cap, (size_t)2 * m->max_sub + (size_t)2 * c->max_points), m->cap[1]);
  CUDA_CHECK_RET(cudaGetLastError());
  m->stepped = true;
  return ALOAM_OK;
}

void map_out_stage_full(aloam_ctx* c, const Pt4* full, const int* d_n, int n_upper, int k, Pt4* dst, long long* off) {
  LAUNCH(c, KID_MAP_OUTPUT, k_stage_full, grid_for(n_upper), 256, 0, full, d_n, k, dst, off);
}
void map_out_register(aloam_ctx* c, const Pt4* src, const int* d_n, int n_upper, const long long* off_k, long long capacity, const double* x7, Pt4* out) {
  LAUNCH(c, KID_MAP_OUTPUT, k_associate_to_map, grid_for(n_upper), 256, 0, src, d_n, 0, off_k, capacity, x7, out);
}

extern "C" {

int aloam_mapper_reset(aloam_ctx* c) {
  if (!c) return ALOAM_ERR_INVALID_ARG;
  CUDA_CHECK_RET(cudaSetDevice(c->cfg.device));
  int rc = ensure_mapper(c); if (rc) return rc;
  Mapper* m = static_cast<Mapper*>(c->mapper);
  MapperState* h = m->h_state;
  std::memset(h, 0, sizeof(*h));
  h->q_wmap_wodom[3] = 1.0;
  h->cen[0] = 10; h->cen[1] = 10; h->cen[2] = 5;
  for (int t = 0; t < 2; ++t) {
    for (int i = 0; i < NCUBE; ++i) h->slab_of[t][i] = -1;
    for (int i = 0; i < kPool; ++i) h->free_list[t][i] = i;
  }
  CUDA_CHECK_RET(cudaMemcpyAsync(m->d_state, h, sizeof(*h), cudaMemcpyHostToDevice, c->stream));
  CUDA_CHECK_RET(cudaStreamSynchronize(c->stream));
  m->stepped = false;
  return ALOAM_OK;
}

int aloam_mapper_step(aloam_ctx* c, aloam_cloud_view corner_last, aloam_cloud_view surf_last, const double q_wodom_curr[4],
                      const double t_wodom_curr[3], double q_w_curr[4], double t_w_curr[3], aloam_stats* stats) {
  if (!c || !q_wodom_curr || !t_wodom_curr || !q_w_curr || !t_w_curr) return ALOAM_ERR_INVALID_ARG;
  int rc = check_view(corner_last); if (rc) return rc;
  rc = check_view(surf_last); if (rc) return rc;
  if (corner_last.n > c->max_points || surf_last.n > c->max_points) return ALOAM_ERR_CAPACITY;   // before any state is touched
  CUDA_CHECK_RET(cudaSetDevice(c->cfg.device));
  const bool fresh = c->mapper == nullptr;
  rc = ensure_mapper(c); if (rc) return rc;
  if (fresh) { rc = aloam_mapper_reset(c); if (rc) return rc; }
  Mapper* m = static_cast<Mapper*>(c->mapper);
  CUDA_CHECK_RET(cudaEventRecord(c->ev0, c->stream));
  // the inputs are uploaded to mapper-owned device buffers first: the views may alias any ctx-owned pinned buffer
  rc = upload_cloud(c, corner_last, m->d_in[0], c->max_points); if (rc) return rc;
  rc = upload_cloud(c, surf_last, m->d_in[1], c->max_points); if (rc) return rc;
  c->h_ints[112] = corner_last.n; c->h_ints[113] = surf_last.n;
  CUDA_CHECK_RET(cudaMemcpyAsync(m->d_state->in_counts, c->h_ints + 112, 8, cudaMemcpyHostToDevice, c->stream));
  for (int k = 0; k < 4; ++k) c->h_dbl[64 + k] = q_wodom_curr[k];
  for (int k = 0; k < 3; ++k) c->h_dbl[68 + k] = t_wodom_curr[k];
  CUDA_CHECK_RET(cudaMemcpyAsync(m->d_pose_io, c->h_dbl + 64, 56, cudaMemcpyHostToDevice, c->stream));
  rc = mapper_step_device(c, m->d_in[0], &m->d_state->in_counts[0], corner_last.n, m->d_in[1], &m->d_state->in_counts[1], surf_last.n, m->d_pose_io, m->d_pose_io + 7);
  if (rc) return rc;
  CUDA_CHECK_RET(cudaMemcpyAsync(c->h_dbl + 72, m->d_pose_io + 7, 56, cudaMemcpyDeviceToHost, c->stream));
  CUDA_CHECK_RET(cudaMemcpyAsync(c->h_summary, c->d_map_summary, sizeof(LmSummary) * 4, cudaMemcpyDeviceToHost, c->stream));
  CUDA_CHECK_RET(cudaMemcpyAsync(&m->h_state->flags, &m->d_state->flags, 2 * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  CUDA_CHECK_RET(cudaEventRecord(c->ev1, c->stream));
  CUDA_CHECK_RET(cudaStreamSynchronize(c->stream));
  CUDA_CHECK_RET(cudaGetLastError());
  prof_collect(c);
  for (int k = 0; k < 4; ++k) q_w_curr[k] = c->h_dbl[72 + k];
  for (int k = 0; k < 3; ++k) t_w_curr[k] = c->h_dbl[76 + k];
  float ms = 0; cudaEventElapsedTime(&ms, c->ev0, c->ev1);
  if (m->h_state->flags & ALOAM_FLAG_MAP_TOO_THIN) { if (stats) { std::memset(stats, 0, sizeof(*stats)); stats->flags = m->h_state->flags; stats->ms_total = ms; } }
  else fill_stats(c, stats, c->cfg.outer_iters, m->h_state->flags, ms);
  if (m->h_state->err & 1) return ALOAM_ERR_CAPACITY;   // a voxel index range beyond the key width: results would be wrong
  return ALOAM_OK;
}

int aloam_mapper_debug_state(aloam_ctx* c, int centre[3], int* n_valid, int valid[125], double q_wmap_wodom[4], double t_wmap_wodom[3],
                             long long totals[2]) {
  if (!c || !c->mapper) return ALOAM_ERR_STATE;
  Mapper* m = static_cast<Mapper*>(c->mapper);
  CUDA_CHECK_RET(cudaSetDevice(c->cfg.device));
  CUDA_CHECK_RET(cudaMemcpy(m->h_state, m->d_state, sizeof(MapperState), cudaMemcpyDeviceToHost));
  const MapperState* h = m->h_state;
  if (centre) for (int a = 0; a < 3; ++a) centre[a] = h->cen[a];
  if (n_valid) *n_valid = h->n_valid;
  if (valid) for (int i = 0; i < h->n_valid && i < 125; ++i) valid[i] = h->valid[i];
  if (q_wmap_wodom) for (int k = 0; k < 4; ++k) q_wmap_wodom[k] = h->q_wmap_wodom[k];
  if (t_wmap_wodom) for (int k = 0; k < 3; ++k) t_wmap_wodom[k] = h->t_wmap_wodom[k];
  if (totals)
    for (int t = 0; t < 2; ++t) {
      totals[t] = 0;
      for (int i = 0; i < NCUBE; ++i) { const int s = h->slab_of[t][i]; if (s >= 0) totals[t] += h->cnt[t][s]; }
    }
  return ALOAM_OK;
}

int aloam_mapper_debug_cube(aloam_ctx* c, int which, int cube, aloam_cloud_view* out) {
  if (!c || !c->mapper || !out || which < 0 || which > 1 || cube < 0 || cube >= NCUBE) return ALOAM_ERR_INVALID_ARG;
  Mapper* m = static_cast<Mapper*>(c->mapper);
  CUDA_CHECK_RET(cudaSetDevice(c->cfg.device));
  CUDA_CHECK_RET(cudaMemcpy(m->h_state, m->d_state, sizeof(MapperState), cudaMemcpyDeviceToHost));
  const int s = m->h_state->slab_of[which][cube];
  const int n = s < 0 ? 0 : m->h_state->cnt[which][s];
  out->data = reinterpret_cast<const float*>(c->h_out[4]); out->n = n; out->stride_floats = 4;
  if (n > 0) CUDA_CHECK_RET(cudaMemcpy(c->h_out[4], m->d_pts[which] + (size_t)s * m->cap[which], (size_t)n * sizeof(Pt4), cudaMemcpyDeviceToHost));
  return ALOAM_OK;
}

int aloam_mapper_export(aloam_ctx* c, int region, float* out, long long capacity_points, long long* n_points) {
  if (!c || !n_points || (region != ALOAM_MAP_SURROUND && region != ALOAM_MAP_ALL) || capacity_points < 0 || (!out && capacity_points != 0))
    return ALOAM_ERR_INVALID_ARG;
  if (!c->mapper) return ALOAM_ERR_STATE;
  Mapper* m = static_cast<Mapper*>(c->mapper);
  CUDA_CHECK_RET(cudaSetDevice(c->cfg.device));
  // sizes and offsets on the device (one scan over <= 2 x 4851 counts), one synchronisation to learn the total
  LAUNCH(c, KID_MAP_OUTPUT, k_export_offsets, 1, 1024, 0, (const MapperState*)m->d_state, region, m->d_seg_off, m->d_seg_off + 2 * NCUBE + 1);
  CUDA_CHECK_RET(cudaMemcpyAsync(c->h_ints + 120, m->d_seg_off + 2 * NCUBE + 1, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  CUDA_CHECK_RET(cudaStreamSynchronize(c->stream));
  CUDA_CHECK_RET(cudaGetLastError());
  const long long n = c->h_ints[120];
  *n_points = n;
  if (!out) return ALOAM_OK;                                  // size query
  if (n > capacity_points) return ALOAM_ERR_CAPACITY;        // nothing written
  if (n == 0) return ALOAM_OK;
  cudaPointerAttributes pa;
  if (cudaPointerGetAttributes(&pa, out) != cudaSuccess) { cudaGetLastError(); pa.type = cudaMemoryTypeUnregistered; }
  const bool on_device = pa.type == cudaMemoryTypeDevice || pa.type == cudaMemoryTypeManaged;
  Pt4* dst = reinterpret_cast<Pt4*>(out);
  if (!on_device) {   // host memory: through the mapper's staging buffer, then one copy
    if (m->export_cap < (size_t)n) {
      if (m->d_export) cudaFree(m->d_export);
      m->d_export = nullptr; m->export_cap = 0;
      CUDA_CHECK_RET(cudaMalloc((void**)&m->d_export, (size_t)n * sizeof(Pt4)));
      m->export_cap = (size_t)n;
    }
    dst = m->d_export;
  }
  LAUNCH(c, KID_MAP_OUTPUT, k_export_copy, region == ALOAM_MAP_SURROUND ? 2 * kMaxValid : 2 * NCUBE, 256, 0, (const MapperState*)m->d_state, region,
         (const int*)m->d_seg_off, (const Pt4*)m->d_pts[0], (const Pt4*)m->d_pts[1], m->cap[0], m->cap[1], dst);
  if (!on_device) CUDA_CHECK_RET(cudaMemcpyAsync(out, dst, (size_t)n * sizeof(Pt4), cudaMemcpyDeviceToHost, c->stream));
  CUDA_CHECK_RET(cudaStreamSynchronize(c->stream));
  CUDA_CHECK_RET(cudaGetLastError());
  return ALOAM_OK;
}

int aloam_mapper_associate_to_map(aloam_ctx* c, aloam_cloud_view in, float* out) {
  if (!c || (!out && in.n > 0)) return ALOAM_ERR_INVALID_ARG;
  int rc = check_view(in); if (rc) return rc;
  if (in.n > c->max_points) return ALOAM_ERR_CAPACITY;
  if (!c->mapper || !static_cast<Mapper*>(c->mapper)->stepped) return ALOAM_ERR_STATE;
  if (in.n == 0) return ALOAM_OK;
  Mapper* m = static_cast<Mapper*>(c->mapper);
  CUDA_CHECK_RET(cudaSetDevice(c->cfg.device));
  rc = upload_cloud(c, in, m->d_in[0], c->max_points); if (rc) return rc;
  LAUNCH(c, KID_MAP_OUTPUT, k_associate_to_map, grid_for(in.n), 256, 0, (const Pt4*)m->d_in[0], (const int*)nullptr, in.n, (const long long*)nullptr, 0LL,
         (const double*)m->d_state->x, m->d_world);
  CUDA_CHECK_RET(cudaMemcpyAsync(out, m->d_world, (size_t)in.n * sizeof(Pt4), cudaMemcpyDefault, c->stream));
  CUDA_CHECK_RET(cudaStreamSynchronize(c->stream));
  CUDA_CHECK_RET(cudaGetLastError());
  return ALOAM_OK;
}

}  // extern "C"
