// badba.cu -- C ABI (include/badba.h) and host orchestration of libbadba_b200.
//
// Host-side structure mirrors the reference's DirectBA (direct_ba.{h,cc}, direct_ba_alternating.cc) but the
// schedule is B200-first: per outer BA iteration the device runs
//     1 launch   activation + normals      (reference: 1 + K_active + 1 + K + 1 launches)
//     1 launch   position + descriptors    (reference: 1 + K + 1 launches)
//     <=30 x 2   pose accumulate + solve for ALL keyframes at once (reference: K x n_GN x {2 clears, kernel,
//                2 D2H copies, stream sync}, kernel_opt_pose.cc:67-96)
// and the host synchronises ONCE per outer iteration to read back the poses.
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <string>
#include <thread>
#include <vector>

#include "../../include/badba.h"
#include "host_math.hpp"
#include "kernels.cuh"
#include "odometry.cuh"
#include "preprocess_tile.cuh"

namespace {

using bba::KfDevice;
using bba::Pose;

struct Frustum {   // libvis/src/libvis/camera_frustum.h:43-250
  float p[8][3];
  float bmin[3], bmax[3];
  float axes[6][3];
  float plane_n[6][3];
  float plane_d[6];
};

inline void Sub(const float a[3], const float b[3], float o[3]) { o[0] = a[0] - b[0]; o[1] = a[1] - b[1]; o[2] = a[2] - b[2]; }
inline void CrossP(const float a[3], const float b[3], float o[3]) {
  o[0] = a[1] * b[2] - a[2] * b[1];
  o[1] = a[2] * b[0] - a[0] * b[2];
  o[2] = a[0] * b[1] - a[1] * b[0];
}
inline float DotP(const float a[3], const float b[3]) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }

void MakeFrustum(Frustum* f, const float K[4], int width, int height, float min_depth, float max_depth, const Pose& global_T_cam) {
  float M[12];
  bba::ToMatrix3x4(global_T_cam, M);
  for (int i = 0; i < 3; ++i) {
    f->bmin[i] = std::numeric_limits<float>::infinity();
    f->bmax[i] = -std::numeric_limits<float>::infinity();
  }
  // corner order of camera_frustum.h:155-177: top-left, top-right, bottom-left, bottom-right; min then max depth
  const float cx[4] = {0.f, static_cast<float>(width), 0.f, static_cast<float>(width)};
  const float cy[4] = {0.f, 0.f, static_cast<float>(height), static_cast<float>(height)};
  for (int c = 0; c < 4; ++c) {
    const float dx = (cx[c] - K[2]) / K[0], dy = (cy[c] - K[3]) / K[1];   // UnprojectFromPixelCornerConv
    for (int d = 0; d < 2; ++d) {
      const float depth = d ? max_depth : min_depth;
      const float v[3] = {depth * dx, depth * dy, depth};
      float* o = f->p[2 * c + d];
      for (int r = 0; r < 3; ++r) {
        o[r] = M[r * 4] * v[0] + M[r * 4 + 1] * v[1] + M[r * 4 + 2] * v[2] + M[r * 4 + 3];
        f->bmin[r] = std::fmin(f->bmin[r], o[r]);
        f->bmax[r] = std::fmax(f->bmax[r], o[r]);
      }
    }
  }
  // camera_frustum.h:180-218
  Sub(f->p[7], f->p[6], f->axes[0]);
  Sub(f->p[3], f->p[2], f->axes[1]);
  Sub(f->p[5], f->p[4], f->axes[2]);
  Sub(f->p[1], f->p[0], f->axes[3]);
  Sub(f->p[2], f->p[6], f->axes[4]);
  Sub(f->p[0], f->p[2], f->axes[5]);
  float fwd[3];
  CrossP(f->axes[5], f->axes[4], fwd);
  for (int i = 0; i < 3; ++i) {
    f->plane_n[0][i] = fwd[i];
    f->plane_n[1][i] = -fwd[i];
  }
  f->plane_d[0] = -DotP(fwd, f->p[1]);
  f->plane_d[1] = DotP(fwd, f->p[0]);
  CrossP(f->axes[0], f->axes[4], f->plane_n[2]); f->plane_d[2] = -DotP(f->plane_n[2], f->p[6]);
  CrossP(f->axes[1], f->axes[5], f->plane_n[3]); f->plane_d[3] = -DotP(f->plane_n[3], f->p[2]);
  CrossP(f->axes[4], f->axes[2], f->plane_n[4]); f->plane_d[4] = -DotP(f->plane_n[4], f->p[4]);
  CrossP(f->axes[5], f->axes[0], f->plane_n[5]); f->plane_d[5] = -DotP(f->plane_n[5], f->p[6]);
}

bool AllOutside(const Frustum& planes_of, const Frustum& points_of) {
  for (int pl = 0; pl < 6; ++pl) {
    int v = 0;
    for (; v < 8; ++v)
      if (DotP(planes_of.plane_n[pl], points_of.p[v]) + planes_of.plane_d[pl] < 0) break;
    if (v == 8) return true;
  }
  return false;
}

bool FrustaIntersect(const Frustum& a, const Frustum& b) {   // camera_frustum.h:73-143
  for (int i = 0; i < 3; ++i)
    if (std::fmax(a.bmin[i], b.bmin[i]) > std::fmin(a.bmax[i], b.bmax[i])) return false;
  if (AllOutside(a, b) || AllOutside(b, a)) return false;
  // Separating-axis part.  The reference crosses two edge directions of the SAME frustum (camera_frustum.h:122
  // uses axes_[this_edge] and axes_[other_edge], both members of `this`); kept as is for parity.
  for (int e1 = 0; e1 < 6; ++e1)
    for (int e2 = 0; e2 < 6; ++e2) {
      float dir[3];
      CrossP(a.axes[e1], a.axes[e2], dir);
      if (DotP(dir, dir) < 1e-5f) continue;
      float amin = INFINITY, amax = -INFINITY, bmin = INFINITY, bmax = -INFINITY;
      for (int p = 0; p < 8; ++p) {
        const float va = DotP(dir, a.p[p]), vb = DotP(dir, b.p[p]);
        amin = std::fmin(amin, va); amax = std::fmax(amax, va);
        bmin = std::fmin(bmin, vb); bmax = std::fmax(bmax, vb);
      }
      if (amax <= bmin || amin >= bmax) return false;
    }
  return true;
}

struct Keyframe {
  const uint16_t* depth = nullptr;
  const uint16_t* normals = nullptr;
  const uint16_t* radius = nullptr;
  size_t depth_pitch = 0, normals_pitch = 0, radius_pitch = 0;
  cudaArray_t luma = nullptr;   // library-owned u8 CUDA array (the .w channel of the caller's uchar4 colour buffer)
  cudaTextureObject_t tex = 0;
  bool tex_alias = false;       // development switch BADBA_ALIAS_LUMA (tools/ab_locality.py): tex belongs to keyframe 0
  void* owned[3] = {nullptr, nullptr, nullptr};   // depth / normals / radius copies made by bba_add_keyframe_host
  const uint8_t* rgba = nullptr;   // uchar4 colour image (caller-owned, or owned_rgba): surfel colours at creation
  size_t rgba_pitch = 0;
  void* owned_rgba = nullptr;
  int last_active_in_ba_iteration = -1;   // keyframe.cc:47-48
  int last_covis_in_ba_iteration = -1;
  Pose pose;                 // global_T_frame
  int activation = BBA_KF_ACTIVE;
  float min_depth = 0.f, max_depth = 0.f;
  Frustum frustum;
  std::vector<int> covis;
};

}  // namespace

struct bba_context {
  bba_config cfg;
  float depth_K[4], color_K[4];
  float depth_a = 0.f;
  int cf_w = 0, cf_h = 0;
  int sm_count = 148;
  std::string error;

  float* surfels = nullptr;
  size_t surfel_pitch_bytes = 0;
  uint32_t surfels_size = 0;
  uint8_t* active = nullptr;
  float* owned_surfels = nullptr;
  size_t owned_surfel_pitch = 0;
  uint8_t* owned_active = nullptr;

  float* d_cfactor = nullptr;
  uint8_t* luma_staging = nullptr;    // u8 plane staging for the luma arrays
  size_t luma_staging_pitch = 0;
  cudaEvent_t luma_staging_free = nullptr;   // recorded after the staging plane was consumed; the next user (any stream) waits on it
  uint8_t* color_staging = nullptr;   // uchar4 staging image for bba_update_keyframe_host
  size_t color_staging_pitch = 0;
  std::vector<Keyframe> keyframes;

  // device state sized for cfg.max_keyframes
  KfDevice* d_kfs = nullptr;
  KfDevice* d_work_records = nullptr;   // [max_kf] the pose kernel's work list as contiguous records
  float* d_frames = nullptr;            // [9][frames_pitch] per-surfel normal + tangent points, rebuilt at the start of a pose step
  uint32_t frames_pitch = 0;
  float* d_pose_est = nullptr;
  double* d_acc = nullptr;
  unsigned long long* d_stage_counts = nullptr;
  int* d_work[2] = {nullptr, nullptr};
  int* d_count = nullptr;   // 2 ints
  int* d_iterations = nullptr;
  int* d_converged = nullptr;
  double* d_first_stats = nullptr;
  int* d_geo_list = nullptr;
  unsigned long long* d_totals = nullptr;   // [8]
  unsigned int* d_queue = nullptr;          // work-item counter of the pose kernel
  unsigned int* d_geo_queue = nullptr;      // work-item counter of the geometry kernels
  unsigned int* d_tile_epoch = nullptr;     // per-tile group epochs of the geometry kernels
  uint32_t tile_epoch_capacity = 0;
  volatile int* h_flag = nullptr;           // mapped pinned: {iterations completed, work items left}
  int* d_flag = nullptr;                    // device alias of h_flag

  // pinned staging
  KfDevice* h_kfs = nullptr;
  float* h_pose_est = nullptr;
  int* h_work = nullptr;    // max_kf + 2
  int* h_geo_list = nullptr;
  int* h_iterations = nullptr;
  int* h_converged = nullptr;
  double* h_first_stats = nullptr;
  double* h_acc = nullptr;        // one record (32) + 2 stage counts, for bba_accumulate_pose_coeffs
  cudaEvent_t staging_event = nullptr;
  bool staging_pending = false;
  // Multi-GPU with mapped peers: set by every REPLICATED whole-buffer pass (surfel creation / merge / compaction / end tasks),
  // cleared by the next collective.  The geometry kernels store into the other ranks' replicas; a rank must not start them
  // while a slower rank is still reading or rewriting its whole replica in such a pass (PeerFence).
  bool replicated_pass_pending = false;
  cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};

  bba_collective_fn collective = nullptr;
  void* collective_user = nullptr;
  float* d_exchange = nullptr;        // [world][kShardRows][shard_len] floats
  size_t exchange_floats = 0;
  float* d_pose_pack = nullptr;       // [max_kf][kPoseSlot] floats
  float* h_pose_pack = nullptr;       // pinned copy
  int* d_local_ids = nullptr;         // [max_kf]

  // intrinsics step (lazily allocated): [head 64 | B 5P | D P | b2 P | obs P | x1 8] floats + 34 fp64 sums
  float* d_intr = nullptr;
  double* d_intr_sums = nullptr;
  int* d_all_list = nullptr;          // 0 .. max_kf-1
  double* h_intr_sums = nullptr;      // pinned
  float* h_intr_x1 = nullptr;         // pinned, 8 floats

  // NVLink peer replicas (bba_peer_import)
  bba::PeerSet peers{};                       // count == 0: not mapped
  void* peer_bases[2 * bba::kMaxPeers] = {};  // what cudaIpcOpenMemHandle returned (closed on unmap)
  int peer_base_count = 0;
  float* d_barrier = nullptr;

  // in-loop surfel lifecycle (creation / merge), lazily allocated
  unsigned int* d_sup = nullptr;         // [3][cells]
  unsigned int* d_cell_bits = nullptr;   // [cells]
  unsigned int* d_flags = nullptr;       // [w * h]
  unsigned int* d_scan_out = nullptr;    // [w * h]
  unsigned int* d_scan_sums = nullptr;
  bba::CovisEntry* d_covis = nullptr;    // [max_keyframes]
  bba::CovisEntry* h_covis = nullptr;    // pinned

  // end-of-BA surfel maintenance (PerformBASchemeEndTasks)
  int last_ba_iteration_count = -1;          // direct_ba.cc:126
  bba::KfRadius* d_kf_radius = nullptr;      // [max_keyframes], lazily allocated
  bba::KfRadius* h_kf_radius = nullptr;      // pinned
  unsigned int* d_deleted_count = nullptr;
  unsigned int* h_deleted_count = nullptr;   // pinned
  float* d_count_xchg = nullptr;             // [2] deleted count of this rank's shard for the sum all-reduce (multi-GPU)
  float* h_count_xchg = nullptr;             // pinned
  unsigned int* d_compact_sums = nullptr;
  uint32_t compact_sums_capacity = 0;

  // frame-to-model tracking of a frame that is not a keyframe (bba_estimate_frame_pose_for_frame): luma array + texture
  cudaArray_t scratch_luma = nullptr;
  cudaTextureObject_t scratch_tex = 0;

  // image-pair odometry (bba_track_frame_pairwise), lazily allocated: intensity / gradient-magnitude images of both frames
  // (colour-sized), the depth / normal / colour pyramids of both frames, accumulators + barrier + result of the persistent kernel
  struct Odometry {
    int num_scales = 0;          // levels allocated
    int last_num_scales = 0;     // levels filled by the last call (parity hooks)
    int last_first_scale = 0;
    uint8_t* gradmag[2] = {nullptr, nullptr};
    size_t gradmag_pitch[2] = {0, 0};
    cudaTextureObject_t gradmag_tex[2] = {0, 0};
    bba::odom::Image image[2][bba::odom::kMaxScales] = {};   // [0 base | 1 tracked][scale]; owned planes only (level-0 normals are the caller's)
    bool owns_normals[2][bba::odom::kMaxScales] = {};
    int w[bba::odom::kMaxScales] = {}, h[bba::odom::kMaxScales] = {};
    bba::odom::Level level[bba::odom::kMaxScales] = {};      // as passed to the last launch
    double* d_acc = nullptr;             // [3][32]
    unsigned int* d_barrier = nullptr;   // [2]
    bba::odom::TrackResult* d_result = nullptr;
    bba::odom::TrackResult* h_result = nullptr;   // pinned
  } odo;

  // keyframe preprocessing (bba_preprocess_frame), lazily allocated
  float* d_min_max = nullptr;
  float* h_min_max = nullptr;                // pinned

  // PCG solver (lazily allocated): r, M, delta, g, p with pcg_capacity floats each
  float* d_pcg[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
  size_t pcg_capacity = 0;
  double* d_pcg_scalars = nullptr;    // [0] / [2] alpha_n, beta_n (roles swap), [1] alpha_d
  double* h_pcg_scalars = nullptr;    // pinned copy
  float* h_pcg_delta = nullptr;       // pinned: pose part (6 * max_keyframes) + 16

  uint64_t launches = 0;
  int ba_iteration_count = 0;
  // predicted cost of one pose step per keyframe (Gauss-Newton iterations x per-evaluation cost of the last step it took
  // part in); 0 = unknown.  Identical on every rank; drives the keyframe -> rank assignment of the pose step.
  std::vector<float> kf_cost;

  // profiling (bba_set_profiling)
  int profiling = 0;   // 0 off, 1 event timing, 2 event timing + byte-model counters in every iteration
  bba_profile profile;
  cudaEvent_t prof_ev[64];
  unsigned long long* h_totals = nullptr;
};

namespace {

bba_status Fail(bba_handle h, bba_status s, const std::string& msg) {
  if (h) h->error = msg;
  return s;
}

#define BBA_CUDA(h, expr)                                                                                  \
  do {                                                                                                      \
    cudaError_t e__ = (expr);                                                                               \
    if (e__ != cudaSuccess)                                                                                 \
      return Fail(h, BBA_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e__));                    \
  } while (0)

void UnmapPeers(bba_handle h) {
  for (int i = 0; i < h->peer_base_count; ++i) cudaIpcCloseMemHandle(h->peer_bases[i]);
  h->peer_base_count = 0;
  h->peers = bba::PeerSet{};
}

// BADBA_TRACE=1: stage markers on stderr (debugging aid for host-side faults)
#define BBA_TRACE(msg)                                                                   \
  do {                                                                                   \
    static const bool on__ = std::getenv("BADBA_TRACE") != nullptr;                      \
    if (on__) { std::fprintf(stderr, "[badba] %s:%d %s\n", __func__, __LINE__, msg); std::fflush(stderr); } \
  } while (0)

Pose PoseFromArray(const float p[7]) {
  Pose r;
  r.q[0] = p[0]; r.q[1] = p[1]; r.q[2] = p[2]; r.q[3] = p[3];
  r.t[0] = p[4]; r.t[1] = p[5]; r.t[2] = p[6];
  return r;
}
void PoseToArray(const Pose& r, float p[7]) {
  p[0] = r.q[0]; p[1] = r.q[1]; p[2] = r.q[2]; p[3] = r.q[3];
  p[4] = r.t[0]; p[5] = r.t[1]; p[6] = r.t[2];
}

bba::CameraParams MakeCamera(bba_handle h) {
  bba::CameraParams c;
  c.w = h->cfg.depth_width; c.h = h->cfg.depth_height; c.cw = h->cfg.color_width; c.ch = h->cfg.color_height;
  // surfel_projection.h:42-67
  c.fx = h->depth_K[0]; c.fy = h->depth_K[1]; c.cx = h->depth_K[2]; c.cy = h->depth_K[3];
  c.fx_inv = 1.0f / c.fx;
  c.fy_inv = 1.0f / c.fy;
  c.cx_inv = -(c.cx - 0.5f) * c.fx_inv;
  c.cy_inv = -(c.cy - 0.5f) * c.fy_inv;
  c.cfx = h->color_K[0]; c.cfy = h->color_K[1]; c.ccx = h->color_K[2]; c.ccy = h->color_K[3];
  // surfel_projection.h:105-124
  c.d2c_fx = c.cfx / c.fx;
  c.d2c_cx = -1 * c.cfx * c.cx / c.fx + c.ccx;
  c.d2c_fy = c.cfy / c.fy;
  c.d2c_cy = -1 * c.cfy * c.cy / c.fy + c.ccy;
  c.a = h->depth_a;
  c.raw_to_float = h->cfg.raw_to_float_depth;
  c.baseline_fx = h->cfg.baseline_fx;
  c.cell = h->cfg.sparse_surfel_cell_size;
  c.cf_w = h->cf_w;
  c.cell_magic = c.cell > 1 ? static_cast<unsigned int>((0x100000000ull + c.cell - 1) / c.cell) : 0u;
  c.cfactor = h->d_cfactor;
  c.use_depth = h->cfg.use_depth_residuals;
  c.use_desc = h->cfg.use_descriptor_residuals;
  return c;
}

bba_status WaitStaging(bba_handle h) {
  if (h->staging_pending) {
    BBA_CUDA(h, cudaEventSynchronize(h->staging_event));
    h->staging_pending = false;
  }
  return BBA_OK;
}
bba_status MarkStaging(bba_handle h, cudaStream_t s) {
  BBA_CUDA(h, cudaEventRecord(h->staging_event, s));
  h->staging_pending = true;
  return BBA_OK;
}

void FillKfDevice(const Keyframe& kf, const Pose& global_T_frame, KfDevice* d) {
  bba::ToMatrix3x4(bba::Inverse(global_T_frame), d->T);
  d->depth = kf.depth;
  d->normals = kf.normals;
  d->tex = kf.tex;
  d->depth_pitch = static_cast<uint32_t>(kf.depth_pitch);
  d->normals_pitch = static_cast<uint32_t>(kf.normals_pitch);
  d->activation = kf.activation;
  d->pad = 0;
}

// Uploads every keyframe's parameters (pose, pointers, activation).  K x 96 bytes.
bba_status UploadKeyframes(bba_handle h, cudaStream_t s) {
  const int K = static_cast<int>(h->keyframes.size());
  if (K == 0) return BBA_OK;
  if (bba_status st = WaitStaging(h)) return st;
  for (int k = 0; k < K; ++k) FillKfDevice(h->keyframes[k], h->keyframes[k].pose, h->h_kfs + k);
  BBA_CUDA(h, cudaMemcpyAsync(h->d_kfs, h->h_kfs, sizeof(KfDevice) * K, cudaMemcpyHostToDevice, s));
  return MarkStaging(h, s);
}

bba_status CheckSurfels(bba_handle h) {
  if (!h->surfels || !h->active) return Fail(h, BBA_ERR_STATE, "surfel buffer / active flags not set");
  return BBA_OK;
}

// Runs the Gauss-Newton loop of EstimateFramePose for the keyframes in `ids`, all at once, starting from
// `init` poses.  On return (stream synchronised) h_pose_est / h_iterations / h_converged / h_first_stats hold the results.
bba_status CheckCollective(bba_handle h);

// Keyframe -> rank assignment of a pose step.  Without statistics: round-robin over the work list
// (bba_shard_keyframe_owner).  With the statistics of the previous pose step (replicated, hence identical on all ranks):
// longest-processing-time-first onto the least loaded rank, so that the ranks finish their Gauss-Newton loops together.
void BalanceWork(const float* cost, int n, int world, int* owner) {
  double known_sum = 0;
  int known = 0;
  for (int i = 0; i < n; ++i)
    if (cost && cost[i] > 0) { known_sum += cost[i]; ++known; }
  if (known == 0 || world <= 1) {
    for (int i = 0; i < n; ++i) owner[i] = world > 1 ? i % world : 0;
    return;
  }
  const double fallback = known_sum / known;
  std::vector<std::pair<double, int>> order(n);
  for (int i = 0; i < n; ++i) order[i] = {-(cost[i] > 0 ? static_cast<double>(cost[i]) : fallback), i};
  std::sort(order.begin(), order.end());   // descending cost, ties by list position
  std::vector<double> load(world, 0.0);
  for (const auto& e : order) {
    int best = 0;
    for (int r = 1; r < world; ++r)
      if (load[r] < load[best]) best = r;
    owner[e.second] = best;
    load[best] -= e.first;
  }
}

void AssignKeyframes(bba_handle h, const std::vector<int>& ids, std::vector<int>* owner) {
  std::vector<float> cost(ids.size(), 0.f);
  for (size_t i = 0; i < ids.size(); ++i)
    if (ids[i] < static_cast<int>(h->kf_cost.size())) cost[i] = h->kf_cost[ids[i]];
  BalanceWork(cost.data(), static_cast<int>(ids.size()), h->cfg.world_size, owner->data());
}

bba_status RunPoseStep(bba_handle h, const std::vector<int>& ids, const std::vector<Pose>& init, int max_iterations, cudaStream_t s) {
  const int K = static_cast<int>(h->keyframes.size());
  const int n = static_cast<int>(ids.size());
  if (n == 0) return BBA_OK;
  if (bba_status st = WaitStaging(h)) return st;
  for (int k = 0; k < K; ++k) {
    FillKfDevice(h->keyframes[k], h->keyframes[k].pose, h->h_kfs + k);
    PoseToArray(h->keyframes[k].pose, h->h_pose_est + 7 * k);
  }
  // Multi-GPU: the work list is dealt to the ranks (AssignKeyframes); every rank runs the Gauss-Newton loops of its own
  // keyframes and the results are published with one sum all-reduce over disjoint slots (below).
  const int world = h->cfg.world_size, rank = h->cfg.rank;
  if (bba_status st = CheckCollective(h)) return st;
  std::vector<int> owner(n, 0);
  if (world > 1) AssignKeyframes(h, ids, &owner);
  std::vector<int> local;
  local.reserve(n);
  for (int i = 0; i < n; ++i) {
    FillKfDevice(h->keyframes[ids[i]], init[i], h->h_kfs + ids[i]);
    PoseToArray(init[i], h->h_pose_est + 7 * ids[i]);
    if (owner[i] == rank) {
      h->h_work[local.size()] = ids[i];
      local.push_back(ids[i]);
    }
  }
  const int n_local = static_cast<int>(local.size());
  h->h_work[h->cfg.max_keyframes] = n_local;
  h->h_work[h->cfg.max_keyframes + 1] = 0;
  BBA_CUDA(h, cudaMemcpyAsync(h->d_kfs, h->h_kfs, sizeof(KfDevice) * K, cudaMemcpyHostToDevice, s));
  BBA_CUDA(h, cudaMemcpyAsync(h->d_pose_est, h->h_pose_est, sizeof(float) * 7 * K, cudaMemcpyHostToDevice, s));
  if (n_local) BBA_CUDA(h, cudaMemcpyAsync(h->d_work[0], h->h_work, sizeof(int) * n_local, cudaMemcpyHostToDevice, s));
  if (world > 1 && n_local) BBA_CUDA(h, cudaMemcpyAsync(h->d_local_ids, h->h_work, sizeof(int) * n_local, cudaMemcpyHostToDevice, s));
  BBA_CUDA(h, cudaMemcpyAsync(h->d_count, h->h_work + h->cfg.max_keyframes, sizeof(int) * 2, cudaMemcpyHostToDevice, s));
  BBA_CUDA(h, cudaMemsetAsync(h->d_acc, 0, sizeof(double) * bba::kPoseAccSize * K, s));
  BBA_CUDA(h, cudaMemsetAsync(h->d_stage_counts, 0, sizeof(unsigned long long) * 2 * K, s));
  BBA_CUDA(h, cudaMemsetAsync(h->d_iterations, 0, sizeof(int) * K, s));
  BBA_CUDA(h, cudaMemsetAsync(h->d_converged, 0, sizeof(int) * K, s));
  BBA_CUDA(h, cudaMemsetAsync(h->d_queue, 0, sizeof(unsigned int), s));
  if (bba_status st = MarkStaging(h, s)) return st;

  bba::PoseAccumulateArgs acc;
  acc.cam = MakeCamera(h);
  acc.surfels = h->surfels;
  acc.pitch = static_cast<uint32_t>(h->surfel_pitch_bytes / sizeof(float));
  acc.n = h->surfels_size;
  acc.kfs = h->d_kfs;
  acc.work_records = h->d_work_records;
  acc.acc = h->d_acc;
  acc.stage_counts = h->d_stage_counts;
  acc.queue = h->d_queue;
  acc.frames = nullptr;
  acc.frames_pitch = 0;
  // The surfels do not move during a pose step: what the descriptor residual needs of a surfel alone (unpacked normal, the two
  // tangent points) is computed once here instead of once per (surfel, keyframe, Gauss-Newton iteration) pair.  Not worth a
  // launch + 9 rows of traffic for a handful of keyframes (frame tracking): the kernel then derives them per pair.
  if (h->cfg.use_descriptor_residuals && n_local >= 4 && h->surfels_size > 0) {
    const uint32_t pitch = static_cast<uint32_t>(h->surfel_pitch_bytes / sizeof(float));
    if (!h->d_frames || h->frames_pitch < pitch) {
      cudaFree(h->d_frames);
      h->d_frames = nullptr;
      h->frames_pitch = pitch;
      BBA_CUDA(h, cudaMalloc(&h->d_frames, sizeof(float) * 9 * static_cast<size_t>(pitch)));
    }
    bba::LaunchSurfelFrames(h->surfels, pitch, h->surfels_size, h->d_frames, h->frames_pitch, s);
    ++h->launches;
    acc.frames = h->d_frames;
    acc.frames_pitch = h->frames_pitch;
  }
  bba::PoseSolveArgs sol;
  sol.kfs = h->d_kfs;
  sol.pose_est = h->d_pose_est;
  sol.acc = h->d_acc;
  sol.stage_counts = h->d_stage_counts;
  sol.iterations = h->d_iterations;
  sol.converged = h->d_converged;
  sol.first_stats = h->d_first_stats;
  sol.max_iterations = max_iterations;
  sol.totals = h->d_totals;
  sol.host_flag = h->d_flag;
  sol.queue = h->d_queue;
  h->h_flag[0] = 0;
  h->h_flag[1] = n_local;
  if (h->profiling) BBA_CUDA(h, cudaMemsetAsync(h->d_totals, 0, sizeof(unsigned long long) * 8, s));
  int enqueued = 0;
  for (int it = 0; it < max_iterations; ++it) {
    const int cur = it & 1;
    acc.work_list = h->d_work[cur];
    acc.work_count = h->d_count + cur;
    if (h->surfels_size > 0) {
      if (h->profiling && it < 32) BBA_CUDA(h, cudaEventRecord(h->prof_ev[2 * it], s));
      bba::LaunchPoseAccumulate(acc, h->sm_count, /*with_stats=*/it == 0 || h->profiling >= 2, n_local, s);
      if (h->profiling && it < 32) BBA_CUDA(h, cudaEventRecord(h->prof_ev[2 * it + 1], s));
      h->launches += 2;   // record packing + the kernel
    }
    sol.work_in = h->d_work[cur];
    sol.count_in = h->d_count + cur;
    sol.work_out = h->d_work[cur ^ 1];
    sol.count_out = h->d_count + (cur ^ 1);
    sol.iteration = it;
    bba::LaunchPoseSolve(sol, s);
    ++h->launches;
    ++enqueued;
    // Keep kDepth iterations queued ahead of the one executing: wait (host poll on zero-copy memory, the stream is never
    // blocked) until iteration it-kDepth has finished, and stop as soon as an iteration left no unconverged keyframe.  (An
    // iteration whose list turned out empty costs three immediately-returning launches, ~10 us; the depth rides out a host
    // thread that is descheduled for a moment -- on a box whose cores were oversubscribed, 2 CPUs for 4 ranks, a depth of one
    // left the GPU idle between iterations.)
    constexpr int kDepth = 3;
    if (it >= kDepth) {
      unsigned int polls = 0;
      while (h->h_flag[0] < it - kDepth + 1) {
        // cudaSuccess: everything drained; any other result than "not ready" is a (sticky) device fault that would
        // otherwise leave this loop spinning for ever -- the BBA_CUDA check below reports it
        if (cudaStreamQuery(s) != cudaErrorNotReady) break;
        if (++polls > 256 && (polls & 15) == 0) std::this_thread::yield();   // let the other ranks' host threads run
      }
    }
    if (it >= 1 && h->h_flag[0] >= 1 && h->h_flag[1] == 0) break;   // (h_flag[1] belongs to the last finished iteration)
  }
  BBA_CUDA(h, cudaGetLastError());
  if (world > 1) {
    // ONE all-reduce per pose step: every rank contributes the slots of its keyframes, all others are zero.
    BBA_CUDA(h, cudaMemsetAsync(h->d_pose_pack, 0, sizeof(float) * bba::kPoseSlot * K, s));
    bba::LaunchPackPoseResults(h->d_local_ids, n_local, h->d_pose_est, h->d_iterations, h->d_converged, h->d_first_stats,
                               h->d_pose_pack, s);
    ++h->launches;
    h->collective(h->collective_user, BBA_COLLECTIVE_ALLREDUCE_SUM, h->d_pose_pack, static_cast<size_t>(bba::kPoseSlot) * K, s);
    h->replicated_pass_pending = false;   // (every rank's earlier work on this stream precedes its contribution)
    BBA_CUDA(h, cudaMemcpyAsync(h->h_pose_pack, h->d_pose_pack, sizeof(float) * bba::kPoseSlot * K, cudaMemcpyDeviceToHost, s));
  } else {
    BBA_CUDA(h, cudaMemcpyAsync(h->h_pose_est, h->d_pose_est, sizeof(float) * 7 * K, cudaMemcpyDeviceToHost, s));
    BBA_CUDA(h, cudaMemcpyAsync(h->h_iterations, h->d_iterations, sizeof(int) * K, cudaMemcpyDeviceToHost, s));
    BBA_CUDA(h, cudaMemcpyAsync(h->h_converged, h->d_converged, sizeof(int) * K, cudaMemcpyDeviceToHost, s));
    BBA_CUDA(h, cudaMemcpyAsync(h->h_first_stats, h->d_first_stats, sizeof(double) * 8 * K, cudaMemcpyDeviceToHost, s));
  }
  if (h->profiling) BBA_CUDA(h, cudaMemcpyAsync(h->h_totals, h->d_totals, sizeof(unsigned long long) * 8, cudaMemcpyDeviceToHost, s));
  BBA_CUDA(h, cudaStreamSynchronize(s));
  h->staging_pending = false;
  if (world > 1) {
    for (int i = 0; i < n; ++i) {
      const int kf = ids[i];
      const float* slot = h->h_pose_pack + static_cast<size_t>(kf) * bba::kPoseSlot;
      std::memcpy(h->h_pose_est + 7 * kf, slot, sizeof(float) * 7);
      h->h_iterations[kf] = static_cast<int>(slot[7] + 0.5f);
      h->h_converged[kf] = static_cast<int>(slot[8] + 0.5f);
      for (int j = 0; j < 8; ++j) h->h_first_stats[8 * kf + j] = slot[9 + j];
    }
  }
  // cost model for the next assignment: a culled pair costs ~6 % of a pair that projects into the image
  if (h->kf_cost.size() < static_cast<size_t>(K)) h->kf_cost.resize(h->cfg.max_keyframes, 0.f);
  for (int kf : ids)
    h->kf_cost[kf] = static_cast<float>(std::max(1, h->h_iterations[kf]) *
                                        (0.06 * h->surfels_size + h->h_first_stats[8 * kf + 5]));
  if (h->profiling && h->surfels_size > 0) {
    int real_iterations = 0;   // iterations that had a non-empty work list
    for (int kf : local) real_iterations = std::max(real_iterations, h->h_iterations[kf]);
    for (int it = 0; it < std::min(real_iterations, std::min(enqueued, 32)); ++it) {
      float ms = 0.f;
      cudaEventElapsedTime(&ms, h->prof_ev[2 * it], h->prof_ev[2 * it + 1]);
      h->profile.pose_ms += ms;
      ++h->profile.pose_launches;
    }
    h->profile.kf_evals += h->h_totals[0];
    h->profile.n_pair += h->h_totals[0] * static_cast<uint64_t>(h->surfels_size);
    h->profile.n_inimg += h->h_totals[1];
    h->profile.n_depthok += h->h_totals[2];
    h->profile.n_assoc += h->h_totals[3];
    h->profile.n_photo += h->h_totals[4];
  }
  return BBA_OK;
}

// ---- multi-GPU sharding (one process per GPU) --------------------------------------------------------------------
// 256-surfel granules dealt round-robin (kernels.cuh SurfelShardToGlobal).  local_cap: size of this rank's local index space
// (a multiple of 256; the last granule may reach past n); shard_len: the same for rank 0 = slice length of the exchange.
void ShardSurfels(uint32_t n, int rank, int world, uint32_t* local_cap, uint32_t* shard_len) {
  const uint32_t granules = (n + 255u) / 256u;
  const uint32_t w = static_cast<uint32_t>(std::max(world, 1)), r = static_cast<uint32_t>(rank);
  const uint32_t mine = granules > r ? (granules - r + w - 1) / w : 0;
  if (local_cap) *local_cap = (world <= 1) ? n : mine * 256u;
  if (shard_len) *shard_len = ((granules + w - 1) / w) * 256u;
}

bba_status CheckCollective(bba_handle h) {
  if (h->cfg.world_size > 1 && !h->collective)
    return Fail(h, BBA_ERR_STATE, "world_size > 1 but no collective registered (bba_set_collective)");
  return BBA_OK;
}

// After the geometry step every rank has updated only its own surfel shard: one all-gather makes the replicas equal.
bba_status ExchangeGeometry(bba_handle h, cudaStream_t s) {
  if (h->cfg.world_size <= 1 || h->surfels_size == 0) return BBA_OK;
  const int world = h->cfg.world_size, rank = h->cfg.rank;
  if (h->peers.count == world - 1) {
    // the geometry kernels already stored the updated rows into every replica over NVLink: only a barrier is left (every
    // rank's kernels have completed, in stream order, before its contribution to the all-reduce)
    if (!h->d_barrier) BBA_CUDA(h, cudaMalloc(&h->d_barrier, sizeof(float)));
    BBA_CUDA(h, cudaMemsetAsync(h->d_barrier, 0, sizeof(float), s));
    h->collective(h->collective_user, BBA_COLLECTIVE_ALLREDUCE_SUM, h->d_barrier, 1, s);
    return BBA_OK;
  }
  uint32_t shard_len;
  ShardSurfels(h->surfels_size, rank, world, nullptr, &shard_len);
  const size_t need = static_cast<size_t>(world) * bba::kShardRows * shard_len;
  if (need > h->exchange_floats) {
    cudaFree(h->d_exchange);
    h->d_exchange = nullptr;
    uint32_t max_len;
    ShardSurfels(std::max(h->cfg.max_surfel_count, h->surfels_size), 0, world, nullptr, &max_len);
    h->exchange_floats = static_cast<size_t>(world) * bba::kShardRows * max_len;
    BBA_CUDA(h, cudaMalloc(&h->d_exchange, sizeof(float) * h->exchange_floats));
  }
  const uint32_t pitch = static_cast<uint32_t>(h->surfel_pitch_bytes / sizeof(float));
  const size_t slice_floats = static_cast<size_t>(bba::kShardRows) * shard_len;
  bba::LaunchPackShard(h->surfels, pitch, h->active, h->surfels_size, rank, world, shard_len, h->d_exchange + slice_floats * rank, s);
  h->collective(h->collective_user, BBA_COLLECTIVE_ALLGATHER, h->d_exchange, slice_floats * sizeof(float), s);
  bba::LaunchUnpackShards(h->surfels, pitch, h->active, h->surfels_size, shard_len, world, rank, h->d_exchange, s);
  h->launches += 2;
  BBA_CUDA(h, cudaGetLastError());
  return BBA_OK;
}

// direct_ba.cc:549-564
void DetermineCovisibleActiveKeyframes(bba_handle h) {
  for (Keyframe& kf : h->keyframes) {
    if (kf.activation != BBA_KF_ACTIVE) continue;
    for (int o : kf.covis) {
      Keyframe& other = h->keyframes[o];
      if (other.activation == BBA_KF_INACTIVE) other.activation = BBA_KF_COVISIBLE_ACTIVE;
    }
  }
}

// A barrier across the ranks (1-element all-reduce) in front of kernels that write into the peers' replicas, needed only when a
// replicated pass ran since the last collective.
bba_status PeerFence(bba_handle h, cudaStream_t s) {
  if (h->cfg.world_size <= 1 || !h->replicated_pass_pending) return BBA_OK;
  h->replicated_pass_pending = false;
  if (h->peers.count != h->cfg.world_size - 1) return BBA_OK;   // exchange through the host's collective: no remote stores
  if (bba_status st = CheckCollective(h)) return st;
  if (!h->d_barrier) BBA_CUDA(h, cudaMalloc(&h->d_barrier, sizeof(float)));
  BBA_CUDA(h, cudaMemsetAsync(h->d_barrier, 0, sizeof(float), s));
  h->collective(h->collective_user, BBA_COLLECTIVE_ALLREDUCE_SUM, h->d_barrier, 1, s);
  return BBA_OK;
}

// Number of this rank's LOCAL surfel indices whose global index is below `global_end` (local -> global is monotonic).
uint32_t LocalCountBelow(uint32_t global_end, int rank, int world) {
  if (world <= 1) return global_end;
  const uint32_t full = global_end >> 8, rest = global_end & 255u;   // granules completely below, surfels of the next one
  const uint32_t w = static_cast<uint32_t>(world), r = static_cast<uint32_t>(rank);
  uint32_t mine = full > r ? (full - r + w - 1) / w : 0;
  uint32_t n = mine * 256u;
  if (full % w == r) n += rest;
  return n;
}

bba_status BuildGeometryArgs(bba_handle h, bba::GeometryArgs* g, cudaStream_t s) {
  if (bba_status st = PeerFence(h, s)) return st;
  const int K = static_cast<int>(h->keyframes.size());
  int cnt = 0;
  for (int k = 0; k < K; ++k)
    if (h->keyframes[k].activation != BBA_KF_INACTIVE) h->h_geo_list[cnt++] = k;
  if (cnt) BBA_CUDA(h, cudaMemcpyAsync(h->d_geo_list, h->h_geo_list, sizeof(int) * cnt, cudaMemcpyHostToDevice, s));
  g->cam = MakeCamera(h);
  g->surfels = h->surfels;
  g->pitch = static_cast<uint32_t>(h->surfel_pitch_bytes / sizeof(float));
  g->n = h->surfels_size;
  g->begin = 0;
  g->shard_rank = static_cast<uint32_t>(h->cfg.rank);
  g->shard_world = static_cast<uint32_t>(h->cfg.world_size);
  ShardSurfels(h->surfels_size, h->cfg.rank, h->cfg.world_size, &g->end, nullptr);
  g->active = h->active;
  g->kfs = h->d_kfs;
  g->kf_list = h->d_geo_list;
  g->kf_count = cnt;
  g->queue = h->d_geo_queue;
  g->tile_shift = 8;
  g->peers = (h->cfg.world_size > 1 && h->peers.count == h->cfg.world_size - 1) ? h->peers : bba::PeerSet{};
  if (!h->d_tile_epoch || h->tile_epoch_capacity < (h->surfels_size + 31u) / 32u) {
    cudaFree(h->d_tile_epoch);
    h->tile_epoch_capacity = std::max<uint32_t>((h->cfg.max_surfel_count + 31u) / 32u, (h->surfels_size + 31u) / 32u) + 1;
    BBA_CUDA(h, cudaMalloc(&h->d_tile_epoch, sizeof(unsigned int) * h->tile_epoch_capacity));
  }
  g->tile_epoch = h->d_tile_epoch;
  return BBA_OK;
}

// OptimizeIntrinsicsCUDA (kernel_opt_intrinsics.cc:39-281): accumulate over EVERY keyframe, Schur-complement the
// per-cell cfactors away, solve the 5x5 / 4x4 systems in fp64 on the host, update intrinsics, a and the cfactors.
bba_status OptimizeIntrinsics(bba_handle h, bool opt_depth, bool opt_color, cudaStream_t s) {
  const int K = static_cast<int>(h->keyframes.size());
  if (h->surfels_size == 0 || K == 0) return BBA_OK;   // :56-58
  const uint32_t P = static_cast<uint32_t>(h->cf_w) * h->cf_h;
  const size_t intr_floats = 64 + static_cast<size_t>(8) * P + 8;
  if (!h->d_intr) {
    BBA_CUDA(h, cudaMalloc(&h->d_intr, sizeof(float) * intr_floats));
    BBA_CUDA(h, cudaMalloc(&h->d_intr_sums, sizeof(double) * bba::kIntrinsicsSums));
    BBA_CUDA(h, cudaMalloc(&h->d_all_list, sizeof(int) * h->cfg.max_keyframes));
    BBA_CUDA(h, cudaMallocHost(&h->h_intr_sums, sizeof(double) * bba::kIntrinsicsSums));
    BBA_CUDA(h, cudaMallocHost(&h->h_intr_x1, sizeof(float) * 8));
    std::vector<int> iota(h->cfg.max_keyframes);
    for (int i = 0; i < h->cfg.max_keyframes; ++i) iota[i] = i;
    BBA_CUDA(h, cudaMemcpy(h->d_all_list, iota.data(), sizeof(int) * iota.size(), cudaMemcpyHostToDevice));
  }
  if (bba_status st = UploadKeyframes(h, s)) return st;
  BBA_CUDA(h, cudaMemsetAsync(h->d_intr, 0, sizeof(float) * intr_floats, s));                      // :69-80
  BBA_CUDA(h, cudaMemsetAsync(h->d_intr_sums, 0, sizeof(double) * bba::kIntrinsicsSums, s));
  float* cell_B = h->d_intr + 64;
  float* cell_D = cell_B + static_cast<size_t>(5) * P;
  float* cell_b2 = cell_D + P;
  float* cell_obs = cell_b2 + P;
  float* d_x1 = cell_obs + P;

  bba::IntrinsicsArgs a;
  a.cam = MakeCamera(h);
  a.surfels = h->surfels;
  a.pitch = static_cast<uint32_t>(h->surfel_pitch_bytes / sizeof(float));
  a.n = h->surfels_size;
  a.begin = 0;
  a.shard_rank = static_cast<uint32_t>(h->cfg.rank);
  a.shard_world = static_cast<uint32_t>(h->cfg.world_size);
  ShardSurfels(h->surfels_size, h->cfg.rank, h->cfg.world_size, &a.end, nullptr);
  a.kfs = h->d_kfs;
  a.kf_list = h->d_all_list;
  a.kf_count = K;
  a.queue = h->d_geo_queue;
  a.sums = h->d_intr_sums;
  a.cell_B = cell_B;
  a.cell_D = cell_D;
  a.cell_b2 = cell_b2;
  a.cell_obs = cell_obs;
  a.cell_count = P;
  bba::LaunchIntrinsicsAccumulate(a, h->sm_count, opt_color, opt_depth, s);   // :84-108, one launch for all keyframes
  ++h->launches;
  if (h->cfg.world_size > 1) {
    // every rank accumulated its surfel shard: one sum all-reduce over [34 global sums | B | D | b2 | obs]
    bba::LaunchIntrinsicsConvertSums(h->d_intr_sums, h->d_intr, true, s);
    h->collective(h->collective_user, BBA_COLLECTIVE_ALLREDUCE_SUM, h->d_intr, 64 + static_cast<size_t>(8) * P, s);
    bba::LaunchIntrinsicsConvertSums(h->d_intr_sums, h->d_intr, false, s);
    h->launches += 2;
  }
  if (opt_depth) {
    bba::LaunchIntrinsicsSchur(P, cell_B, cell_D, cell_b2, h->d_intr_sums, s);   // :120-127
    ++h->launches;
  }
  BBA_CUDA(h, cudaGetLastError());
  BBA_CUDA(h, cudaMemcpyAsync(h->h_intr_sums, h->d_intr_sums, sizeof(double) * bba::kIntrinsicsSums, cudaMemcpyDeviceToHost, s));
  BBA_CUDA(h, cudaStreamSynchronize(s));   // :136

  if (opt_depth) {
    // the reference keeps A and b1 in fp32 buffers and solves in fp64 (:130-171)
    double A[15], b1[5], x1[5];
    for (int i = 0; i < 15; ++i) A[i] = static_cast<double>(static_cast<float>(h->h_intr_sums[i]));
    for (int i = 0; i < 5; ++i) b1[i] = static_cast<double>(static_cast<float>(h->h_intr_sums[15 + i]));
    constexpr float kAPriorWeight = 10;   // :153-155
    A[14] = static_cast<double>(static_cast<float>(A[14]) + kAPriorWeight * kAPriorWeight);
    b1[4] = static_cast<double>(static_cast<float>(b1[4]) + kAPriorWeight * kAPriorWeight * h->depth_a);
    bba::SolveLDLT<5>(A, b1, x1);
    float x1f[5];
    for (int i = 0; i < 5; ++i) x1f[i] = static_cast<float>(x1[i]);
    const bba::CameraParams& c = a.cam;   // :183-194
    const float new_fx = 1.0f / (c.fx_inv - x1f[0]);
    const float new_fy = 1.0f / (c.fy_inv - x1f[1]);
    const float new_cx = -(new_fx * (c.cx_inv - x1f[2])) + 0.5f;
    const float new_cy = -(new_fy * (c.cy_inv - x1f[3])) + 0.5f;
    for (int i = 0; i < 5; ++i) h->h_intr_x1[i] = x1f[i];
    BBA_CUDA(h, cudaMemcpyAsync(d_x1, h->h_intr_x1, sizeof(float) * 5, cudaMemcpyHostToDevice, s));   // :196
    bba::LaunchIntrinsicsCellUpdate(P, cell_obs, cell_B, cell_D, d_x1, h->d_cfactor, s);             // :205-212
    ++h->launches;
    BBA_CUDA(h, cudaGetLastError());
    BBA_CUDA(h, cudaStreamSynchronize(s));   // h_intr_x1 is reused by the next call
    h->depth_K[0] = new_fx; h->depth_K[1] = new_fy; h->depth_K[2] = new_cx; h->depth_K[3] = new_cy;
    h->depth_a -= x1f[4];
  }
  if (opt_color) {   // :256-280
    double H[10], b[4], x[4];
    for (int i = 0; i < 10; ++i) H[i] = static_cast<double>(static_cast<float>(h->h_intr_sums[20 + i]));
    for (int i = 0; i < 4; ++i) b[i] = static_cast<double>(static_cast<float>(h->h_intr_sums[30 + i]));
    bba::SolveLDLT<4>(H, b, x);
    for (int i = 0; i < 4; ++i) h->color_K[i] -= static_cast<float>(x[i]);
  }
  return BBA_OK;
}

int GetMinObservationCount(bba_handle h);

// ---- in-loop surfel lifecycle ---------------------------------------------------------------------------------------------
uint32_t SurfelCapacity(bba_handle h) {
  return std::min<uint32_t>(h->cfg.max_surfel_count, static_cast<uint32_t>(h->surfel_pitch_bytes / sizeof(float)));
}

bba_status MakeLifecycleArgs(bba_handle h, int k, bba::LifecycleArgs* a, cudaStream_t s) {
  const uint32_t cells = static_cast<uint32_t>(h->cf_w) * h->cf_h;
  const uint32_t pixels = static_cast<uint32_t>(h->cfg.depth_width) * h->cfg.depth_height;
  if (!h->d_sup) {
    BBA_CUDA(h, cudaMalloc(&h->d_sup, sizeof(unsigned int) * 3 * cells));
    BBA_CUDA(h, cudaMalloc(&h->d_cell_bits, sizeof(unsigned int) * cells));
    BBA_CUDA(h, cudaMalloc(&h->d_flags, sizeof(unsigned int) * pixels));
    BBA_CUDA(h, cudaMalloc(&h->d_scan_out, sizeof(unsigned int) * pixels));
    BBA_CUDA(h, cudaMalloc(&h->d_scan_sums, sizeof(unsigned int) * bba::ScanScratchWords(pixels)));
    BBA_CUDA(h, cudaMalloc(&h->d_covis, sizeof(bba::CovisEntry) * h->cfg.max_keyframes));
    BBA_CUDA(h, cudaMallocHost(&h->h_covis, sizeof(bba::CovisEntry) * h->cfg.max_keyframes));
  }
  if (!h->d_deleted_count) {
    BBA_CUDA(h, cudaMalloc(&h->d_deleted_count, sizeof(unsigned int)));
    BBA_CUDA(h, cudaMallocHost(&h->h_deleted_count, sizeof(unsigned int)));
  }
  const Keyframe& kf = h->keyframes[k];
  a->cam = MakeCamera(h);
  bba::ToMatrix3x4(bba::Inverse(kf.pose), a->T);
  bba::ToMatrix3x4(kf.pose, a->G);
  a->depth = kf.depth;
  a->normals = kf.normals;
  a->radius = kf.radius;
  a->depth_pitch = static_cast<uint32_t>(kf.depth_pitch);
  a->normals_pitch = static_cast<uint32_t>(kf.normals_pitch);
  a->radius_pitch = static_cast<uint32_t>(kf.radius_pitch);
  a->tex = kf.tex;
  a->rgba = kf.rgba;
  a->rgba_pitch = static_cast<uint32_t>(kf.rgba_pitch);
  a->surfels = h->surfels;
  a->pitch = static_cast<uint32_t>(h->surfel_pitch_bytes / sizeof(float));
  a->n = h->surfels_size;
  a->sup = h->d_sup;
  a->cell_bits = h->d_cell_bits;
  a->cells = cells;
  a->flags = h->d_flags;
  a->covis = h->d_covis;
  a->covis_count = 0;
  a->min_observation_count = GetMinObservationCount(h);
  const float c = static_cast<float>(h->cfg.sparse_surfel_cell_size);
  a->cell_merge_dist_squared = c * c * h->cfg.surfel_merge_dist_factor * h->cfg.surfel_merge_dist_factor;   // kernel_supporting_surfels.cc:76-78
  a->counter = h->d_deleted_count;
  (void)s;
  return BBA_OK;
}

// DirectBA::CreateSurfelsForKeyframe (direct_ba.cc:340-405)
bba_status CreateSurfelsForKeyframe(bba_handle h, int k, bool filter, cudaStream_t s, uint32_t* new_count) {
  *new_count = 0;
  const Keyframe& kf = h->keyframes[k];
  if (!kf.radius || !kf.rgba) return Fail(h, BBA_ERR_STATE, "surfel creation needs the keyframe's radius and colour buffers");
  BBA_TRACE("create: enter");
  h->replicated_pass_pending = true;
  if (bba_status st = WaitStaging(h)) return st;
  bba::LifecycleArgs a;
  if (bba_status st = MakeLifecycleArgs(h, k, &a, s)) return st;
  BBA_TRACE("create: args made");
  if (filter) {   // covis_T_frame for every co-visible keyframe (direct_ba.cc:365-370)
    int cnt = 0;
    for (int c : kf.covis) {
      const Keyframe& other = h->keyframes[c];
      bba::CovisEntry& e = h->h_covis[cnt++];
      bba::ToMatrix3x4(bba::Compose(bba::Inverse(other.pose), kf.pose), e.R);
      e.depth = other.depth;
      e.normals = other.normals;
      e.depth_pitch = static_cast<uint32_t>(other.depth_pitch);
      e.normals_pitch = static_cast<uint32_t>(other.normals_pitch);
      e.pad[0] = e.pad[1] = 0;
    }
    a.covis_count = cnt;
    if (cnt) BBA_CUDA(h, cudaMemcpyAsync(h->d_covis, h->h_covis, sizeof(bba::CovisEntry) * cnt, cudaMemcpyHostToDevice, s));
  }
  BBA_TRACE("create: covis uploaded");
  const uint32_t pixels = static_cast<uint32_t>(h->cfg.depth_width) * h->cfg.depth_height;
  bba::LaunchSupportSurfels(a, h->sm_count, s);     // DetermineSupportingSurfelsCUDA: is the cell supported at all
  bba::LaunchSeedNewSurfels(a, filter, s);
  bba::LaunchExclusiveScan(h->d_flags, pixels, h->d_scan_out, h->d_scan_sums, s);
  h->launches += 6 + (filter ? 1 : 0);
  BBA_CUDA(h, cudaGetLastError());
  const uint32_t n_blocks = (pixels + 4095) / 4096;
  BBA_CUDA(h, cudaMemcpyAsync(h->h_deleted_count, h->d_scan_sums + n_blocks, sizeof(unsigned int), cudaMemcpyDeviceToHost, s));
  BBA_CUDA(h, cudaStreamSynchronize(s));   // kernel_create_surfels.cu:466-474
  h->staging_pending = false;
  const uint32_t created = *h->h_deleted_count;
  BBA_TRACE("create: counted");
  if (created == 0) return BBA_OK;
  if (h->surfels_size + static_cast<uint64_t>(created) > SurfelCapacity(h)) {
    // the reference logs "Maximum surfel count exceeded" and creates nothing (kernel_create_surfels.cc:163-166)
    h->error = "maximum surfel count exceeded: no surfels created for this keyframe";
    return BBA_OK;
  }
  bba::LaunchCreateSurfels(a, h->d_scan_out, s);
  ++h->launches;
  BBA_CUDA(h, cudaGetLastError());
  BBA_TRACE("create: appended");
  h->surfels_size += created;
  *new_count = created;
  return MarkStaging(h, s);
}

// DetermineSupportingSurfelsAndMergeSurfelsCUDA (kernel_supporting_surfels.cc:40-118); deleted surfels are only marked
bba_status MergeSurfelsForKeyframe(bba_handle h, int k, cudaStream_t s, uint32_t* deleted) {
  *deleted = 0;
  if (h->surfels_size == 0) return BBA_OK;
  h->replicated_pass_pending = true;
  bba::LifecycleArgs a;
  if (bba_status st = MakeLifecycleArgs(h, k, &a, s)) return st;
  BBA_CUDA(h, cudaMemsetAsync(h->d_deleted_count, 0, sizeof(unsigned int), s));
  bba::LaunchMergeSurfels(a, h->sm_count, s);
  h->launches += 5;
  BBA_CUDA(h, cudaGetLastError());
  BBA_CUDA(h, cudaMemcpyAsync(h->h_deleted_count, h->d_deleted_count, sizeof(unsigned int), cudaMemcpyDeviceToHost, s));
  BBA_CUDA(h, cudaStreamSynchronize(s));   // kernel_supporting_surfels.cc:93-96
  *deleted = *h->h_deleted_count;
  return BBA_OK;
}

bba_status CompactSurfels(bba_handle h, uint32_t free_count, bool with_active, cudaStream_t s) {
  const uint32_t N = h->surfels_size;
  if (free_count == 0 || N == 0) return BBA_OK;
  h->replicated_pass_pending = true;
  const uint32_t words = bba::CompactScratchWords(N);
  if (words > h->compact_sums_capacity) {
    cudaFree(h->d_compact_sums);
    h->compact_sums_capacity = std::max(words, bba::CompactScratchWords(std::max(h->cfg.max_surfel_count, N)));
    BBA_CUDA(h, cudaMalloc(&h->d_compact_sums, sizeof(unsigned int) * h->compact_sums_capacity));
  }
  bba::LaunchCompactSurfels(h->surfels, static_cast<uint32_t>(h->surfel_pitch_bytes / sizeof(float)), N, free_count, h->d_compact_sums,
                            with_active ? h->active : nullptr, s);
  h->launches += 4;
  BBA_CUDA(h, cudaGetLastError());
  h->surfels_size = N - free_count;
  return BBA_OK;
}

// direct_ba.h:220-226
int GetMinObservationCount(bba_handle h) {
  const size_t K = h->keyframes.size();
  return (K < 10) ? ((K < 5) ? h->cfg.min_observation_count_while_bootstrapping_1 : h->cfg.min_observation_count_while_bootstrapping_2)
                  : h->cfg.min_observation_count;
}

// DirectBA::PerformBASchemeEndTasks (direct_ba.cc:566-653) without the final merge (do_surfel_updates is not supported yet):
// DeleteSurfelsAndUpdateRadiiCUDA over every keyframe, then CompactSurfelsCUDA.  Replicated on every rank of a multi-GPU
// job (once per BA call, deterministic, identical inputs -> identical surfel buffers without an exchange).
bba_status PerformEndTasks(bba_handle h, cudaStream_t s, uint32_t* deleted_out, bool do_surfel_updates = false) {
  if (deleted_out) *deleted_out = 0;
  const int K = static_cast<int>(h->keyframes.size());
  const uint32_t N = h->surfels_size;
  if (N == 0) return BBA_OK;   // kernel_delete_surfels.cc:52-54
  h->replicated_pass_pending = true;
  if (!h->d_kf_radius) {
    BBA_CUDA(h, cudaMalloc(&h->d_kf_radius, sizeof(bba::KfRadius) * h->cfg.max_keyframes));
    BBA_CUDA(h, cudaMallocHost(&h->h_kf_radius, sizeof(bba::KfRadius) * h->cfg.max_keyframes));
  }
  if (!h->d_deleted_count) {
    BBA_CUDA(h, cudaMalloc(&h->d_deleted_count, sizeof(unsigned int)));
    BBA_CUDA(h, cudaMallocHost(&h->h_deleted_count, sizeof(unsigned int)));
  }
  BBA_TRACE("end tasks");
  // merge similar surfels using all keyframes which were active in this BA iteration block (direct_ba.cc:577-601)
  uint32_t merged = 0;
  if (do_surfel_updates) {
    for (int k = 0; k < K; ++k) {
      if (h->keyframes[k].last_active_in_ba_iteration != h->ba_iteration_count) continue;
      uint32_t d = 0;
      if (bba_status st = MergeSurfelsForKeyframe(h, k, s, &d)) return st;
      merged += d;
    }
  }
  if (bba_status st = UploadKeyframes(h, s)) return st;   // (waits for the previous use of the staging buffers)
  for (int k = 0; k < K; ++k) {
    if (!h->keyframes[k].radius) return Fail(h, BBA_ERR_STATE, "end tasks need the keyframes' radius buffers");
    h->h_kf_radius[k].ptr = h->keyframes[k].radius;
    h->h_kf_radius[k].pitch = static_cast<uint32_t>(h->keyframes[k].radius_pitch);
    h->h_kf_radius[k].pad = 0;
  }
  if (K) BBA_CUDA(h, cudaMemcpyAsync(h->d_kf_radius, h->h_kf_radius, sizeof(bba::KfRadius) * K, cudaMemcpyHostToDevice, s));
  BBA_CUDA(h, cudaMemsetAsync(h->d_deleted_count, 0, sizeof(unsigned int), s));
  if (!h->d_tile_epoch || h->tile_epoch_capacity < (N + 31u) / 32u) {
    cudaFree(h->d_tile_epoch);
    h->tile_epoch_capacity = std::max<uint32_t>((h->cfg.max_surfel_count + 31u) / 32u, (N + 31u) / 32u) + 1;
    BBA_CUDA(h, cudaMalloc(&h->d_tile_epoch, sizeof(unsigned int) * h->tile_epoch_capacity));
  }
  bba::SurfelStatsArgs a;
  a.cam = MakeCamera(h);
  a.surfels = h->surfels;
  a.pitch = static_cast<uint32_t>(h->surfel_pitch_bytes / sizeof(float));
  a.n = N;
  a.kfs = h->d_kfs;
  a.radius = h->d_kf_radius;
  a.kf_count = K;
  a.min_observation_count = GetMinObservationCount(h);
  a.queue = h->d_geo_queue;
  a.tile_epoch = h->d_tile_epoch;
  a.tile_shift = 8;
  a.deleted_count = h->d_deleted_count;
  // Multi-GPU: every rank evaluates the surfels of its granule shard (the launch is as expensive as a geometry pass over every
  // keyframe); the two result rows reach the other replicas through peer stores or one all-gather, the deleted counts through a
  // sum all-reduce (which is also the barrier behind the peer stores).  The compaction then runs replicated on identical replicas.
  const int world = h->cfg.world_size, rank = h->cfg.rank;
  const bool peers_mapped = world > 1 && h->peers.count == world - 1;
  a.shard_rank = static_cast<uint32_t>(rank);
  a.shard_world = static_cast<uint32_t>(world);
  ShardSurfels(N, rank, world, &a.local_count, nullptr);
  a.peers = peers_mapped ? h->peers : bba::PeerSet{};
  if (world > 1) {
    if (bba_status st = CheckCollective(h)) return st;
    if (bba_status st = PeerFence(h, s)) return st;   // (e.g. the merges above rewrote whole replicas)
  }
  if (K > 0) {
    bba::LaunchObservationStats(a, h->sm_count, s);
    ++h->launches;
    BBA_CUDA(h, cudaGetLastError());
  }
  // (with no keyframe at all the reference still runs MarkDeletedSurfels on zero counts; not reachable through this API,
  // a BA call without keyframes has nothing to optimise)
  uint32_t deleted_total = 0;
  if (world > 1) {
    if (!peers_mapped && K > 0) {
      uint32_t shard_len;
      ShardSurfels(N, rank, world, nullptr, &shard_len);
      const size_t need = static_cast<size_t>(world) * 2 * shard_len;
      if (need > h->exchange_floats) {
        cudaFree(h->d_exchange);
        h->d_exchange = nullptr;
        uint32_t max_len;
        ShardSurfels(std::max(h->cfg.max_surfel_count, N), 0, world, nullptr, &max_len);
        h->exchange_floats = static_cast<size_t>(world) * bba::kShardRows * max_len;
        BBA_CUDA(h, cudaMalloc(&h->d_exchange, sizeof(float) * h->exchange_floats));
      }
      const size_t slice_floats = static_cast<size_t>(2) * shard_len;
      bba::LaunchPackStatsShard(h->surfels, a.pitch, N, rank, world, shard_len, h->d_exchange + slice_floats * rank, s);
      h->collective(h->collective_user, BBA_COLLECTIVE_ALLGATHER, h->d_exchange, slice_floats * sizeof(float), s);
      bba::LaunchUnpackStatsShards(h->surfels, a.pitch, N, shard_len, world, rank, h->d_exchange, s);
      h->launches += 2;
    }
    // deleted count of this shard as two exactly representable floats (low 12 bits, the rest), summed over the ranks
    if (!h->d_count_xchg) {
      BBA_CUDA(h, cudaMalloc(&h->d_count_xchg, sizeof(float) * 2));
      BBA_CUDA(h, cudaMallocHost(&h->h_count_xchg, sizeof(float) * 2));
    }
    BBA_CUDA(h, cudaMemcpyAsync(h->h_deleted_count, h->d_deleted_count, sizeof(unsigned int), cudaMemcpyDeviceToHost, s));
    BBA_CUDA(h, cudaStreamSynchronize(s));
    h->h_count_xchg[0] = static_cast<float>(*h->h_deleted_count & 0xfffu);
    h->h_count_xchg[1] = static_cast<float>(*h->h_deleted_count >> 12);
    BBA_CUDA(h, cudaMemcpyAsync(h->d_count_xchg, h->h_count_xchg, sizeof(float) * 2, cudaMemcpyHostToDevice, s));
    h->collective(h->collective_user, BBA_COLLECTIVE_ALLREDUCE_SUM, h->d_count_xchg, 2, s);
    BBA_CUDA(h, cudaMemcpyAsync(h->h_count_xchg, h->d_count_xchg, sizeof(float) * 2, cudaMemcpyDeviceToHost, s));
    BBA_CUDA(h, cudaStreamSynchronize(s));
    deleted_total = static_cast<uint32_t>(h->h_count_xchg[0] + 0.5f) + (static_cast<uint32_t>(h->h_count_xchg[1] + 0.5f) << 12);
    h->replicated_pass_pending = true;   // the compaction below rewrites every replica as a whole
  } else {
    BBA_CUDA(h, cudaMemcpyAsync(h->h_deleted_count, h->d_deleted_count, sizeof(unsigned int), cudaMemcpyDeviceToHost, s));
    BBA_CUDA(h, cudaStreamSynchronize(s));   // kernel_delete_surfels.cc:93-96
    deleted_total = *h->h_deleted_count;
  }
  h->staging_pending = false;
  BBA_TRACE("stats done");
  const uint32_t deleted = deleted_total + merged;
  if (deleted_out) *deleted_out = deleted;
  if (deleted > 0) {   // kernel_compact_surfels.cu:167-169
    const uint32_t words = bba::CompactScratchWords(N);
    if (words > h->compact_sums_capacity) {
      cudaFree(h->d_compact_sums);
      h->compact_sums_capacity = std::max(words, bba::CompactScratchWords(std::max(h->cfg.max_surfel_count, N)));
      BBA_CUDA(h, cudaMalloc(&h->d_compact_sums, sizeof(unsigned int) * h->compact_sums_capacity));
    }
    bba::LaunchCompactSurfels(h->surfels, a.pitch, N, deleted, h->d_compact_sums, nullptr, s);   // direct_ba.cc:618: no active flags
    h->launches += 4;
    BBA_CUDA(h, cudaGetLastError());
    h->surfels_size = N - deleted;
  }
  return BBA_OK;
}

// Unknown layout of the PCG solver (direct_ba_pcg.cc:273-309) + the vectors sized for it.
struct PcgLayout {
  bool opt_poses, opt_geometry, opt_depth_intr, opt_color_intr, use_desc;
  uint32_t surfel_start, stride, depth_start, a_index, color_start, unknown_count;
};

bba_status MakePcgLayout(bba_handle h, const bba_ba_options* o, PcgLayout* L) {
  constexpr uint32_t kInvalid = 0xffffffffu;
  const int K = static_cast<int>(h->keyframes.size());
  const uint32_t N = h->surfels_size, P = static_cast<uint32_t>(h->cf_w) * h->cf_h;
  L->opt_depth_intr = o->optimize_depth_intrinsics && h->cfg.use_depth_residuals;   // direct_ba.cc:427-434
  L->opt_color_intr = o->optimize_color_intrinsics && h->cfg.use_descriptor_residuals;
  L->opt_poses = o->optimize_poses != 0;
  L->opt_geometry = o->optimize_geometry != 0;
  L->use_desc = h->cfg.use_descriptor_residuals != 0;
  L->stride = L->use_desc ? 3u : 1u;
  uint32_t cur = 0;
  if (L->opt_poses) cur += 6u * static_cast<uint32_t>(K - 1);
  L->surfel_start = L->depth_start = L->a_index = L->color_start = kInvalid;
  if (L->opt_geometry) { L->surfel_start = cur; cur += L->stride * N; }
  if (L->opt_depth_intr) { L->depth_start = cur; cur += 5u + P; L->a_index = L->depth_start + 4u; }
  if (L->opt_color_intr) { L->color_start = cur; cur += 4u; }
  L->unknown_count = cur;
  if (!h->d_pcg_scalars) {
    BBA_CUDA(h, cudaMalloc(&h->d_pcg_scalars, sizeof(double) * bba::kPcgScalarDoubles));   // scalars + the ordered-sum workspace
    BBA_CUDA(h, cudaMemset(h->d_pcg_scalars, 0, sizeof(double) * bba::kPcgScalarDoubles));
    BBA_CUDA(h, cudaMallocHost(&h->h_pcg_scalars, sizeof(double) * 4));
    BBA_CUDA(h, cudaMallocHost(&h->h_pcg_delta, sizeof(float) * (6 * static_cast<size_t>(h->cfg.max_keyframes) + 16)));
  }
  if (L->unknown_count > h->pcg_capacity) {
    const size_t cap = std::max<size_t>(L->unknown_count, 6 * static_cast<size_t>(h->cfg.max_keyframes) +
                                                              3 * static_cast<size_t>(std::max(h->cfg.max_surfel_count, N)) + 9 + P);
    for (float*& v : h->d_pcg) {
      cudaFree(v);
      v = nullptr;
      BBA_CUDA(h, cudaMalloc(&v, sizeof(float) * (cap + 8)));   // (+ the alpha_d pair that travels with g, multi-GPU)
    }
    h->pcg_capacity = cap;
  }
  return BBA_OK;
}

bba::PcgArgs MakePcgArgs(bba_handle h, const PcgLayout& L, int gauge) {
  bba::PcgArgs a;
  a.cam = MakeCamera(h);
  a.surfels = h->surfels;
  a.pitch = static_cast<uint32_t>(h->surfel_pitch_bytes / sizeof(float));
  a.begin = 0;
  a.n = h->surfels_size;
  a.shard_rank = static_cast<uint32_t>(h->cfg.rank);
  a.shard_world = static_cast<uint32_t>(h->cfg.world_size);
  ShardSurfels(h->surfels_size, h->cfg.rank, h->cfg.world_size, &a.end, nullptr);   // this rank's surfels (all of them on one GPU)
  a.alpha_d_slot = h->cfg.world_size > 1 ? 3 : 1;
  a.kfs = h->d_kfs;
  a.kf_count = static_cast<int>(h->keyframes.size());
  a.gauge_kf = gauge;
  a.opt_poses = L.opt_poses;
  a.opt_geometry = L.opt_geometry;
  a.opt_depth_intr = L.opt_depth_intr;
  a.opt_color_intr = L.opt_color_intr;
  a.surfel_start = L.surfel_start;
  a.surfel_stride = L.stride;
  a.depth_intr_start = L.depth_start;
  a.color_intr_start = L.color_start;
  a.r = h->d_pcg[0];
  a.M = h->d_pcg[1];
  a.p = h->d_pcg[4];
  a.g = h->d_pcg[3];
  a.scalars = h->d_pcg_scalars;
  a.queue = h->d_geo_queue;
  return a;
}

// DirectBA::BundleAdjustmentPCG (direct_ba_pcg.cc:43-819) without the surfel lifecycle branches.
bba_status BundleAdjustPCG(bba_handle h, const bba_ba_options* o, bba_ba_result* res, cudaStream_t s) {
  const int K = static_cast<int>(h->keyframes.size());
  // Multi-GPU: the matrix-free products J^T W F / diag(J^T W J) / J^T W J p are summed over THIS rank's surfels (granule
  // sharding of the geometry step); one sum all-reduce of the vector per product makes every rank hold the full result (a
  // surfel's entries are non-zero on its owner only, pose / intrinsics entries are true sums), and the vector kernels, the
  // scalars and the updates then run replicated and bit-identically on every rank (fixed-order sums, pcg.cu GridOrderedAdd).
  const int world = h->cfg.world_size;
  if (bba_status st = CheckCollective(h)) return st;
  if (world > 1 && o->pcg_gauge_keyframe < 0)
    return Fail(h, BBA_ERR_INVALID_ARGUMENT, "use_pcg with more than one rank needs pcg_gauge_keyframe >= 0 (the reference draws rand() % K)");
  if (K == 0) return Fail(h, BBA_ERR_STATE, "use_pcg: no keyframes");
  const int max_inner = o->pcg_max_inner_iterations > 0 ? o->pcg_max_inner_iterations : 30;
  const int max_keyframes = o->pcg_max_keyframes > 0 ? o->pcg_max_keyframes : 2500;
  if (K > max_keyframes) return Fail(h, BBA_ERR_INVALID_ARGUMENT, "use_pcg: more keyframes than pcg_max_keyframes");   // :232
  if (o->pcg_gauge_keyframe >= K) return Fail(h, BBA_ERR_INVALID_ARGUMENT, "pcg_gauge_keyframe out of range");
  PcgLayout L;
  if (bba_status st = MakePcgLayout(h, o, &L)) return st;
  const bool opt_depth_intr = L.opt_depth_intr, opt_color_intr = L.opt_color_intr, opt_poses = L.opt_poses, opt_geometry = L.opt_geometry;
  const bool use_desc = L.use_desc;
  const uint32_t P = static_cast<uint32_t>(h->cf_w) * h->cf_h;
  const uint64_t launches_before = h->launches;
  const auto t_start = std::chrono::steady_clock::now();
  if (!o->increase_ba_iteration_count && h->ba_iteration_count != h->last_ba_iteration_count) {   // :157-161
    h->last_ba_iteration_count = h->ba_iteration_count;
    uint32_t deleted = 0;
    if (bba_status st = PerformEndTasks(h, s, &deleted, o->do_surfel_updates != 0)) return st;
    res->surfels_deleted += deleted;
  }
  std::vector<int> keyframes_with_new_surfels;

  for (int iteration = 0; iteration < o->max_iterations; ++iteration) {
    if (o->progress_function && !o->progress_function(o->progress_user, iteration)) break;
    ++res->iterations_done;
    // surfel creation (:183-206)
    keyframes_with_new_surfels.clear();
    if (opt_geometry && o->do_surfel_updates) {
      for (int k = 0; k < K; ++k) {
        Keyframe& kf = h->keyframes[k];
        if (kf.activation == BBA_KF_ACTIVE && kf.last_active_in_ba_iteration != h->ba_iteration_count) {
          kf.last_active_in_ba_iteration = h->ba_iteration_count;
          uint32_t created = 0;
          if (bba_status st = CreateSurfelsForKeyframe(h, k, /*filter_new_surfels=*/true, s, &created)) return st;
          res->surfels_created += created;
          keyframes_with_new_surfels.push_back(k);
        } else if (kf.activation == BBA_KF_COVISIBLE_ACTIVE && kf.last_covis_in_ba_iteration != h->ba_iteration_count) {
          kf.last_covis_in_ba_iteration = h->ba_iteration_count;
        }
      }
    }
    const uint32_t N = h->surfels_size;
    if (N > 0) BBA_CUDA(h, cudaMemsetAsync(h->active, bba::kSurfelActiveFlag, N, s));   // :209-212
    if (bba_status st = UploadKeyframes(h, s)) return st;
    BBA_CUDA(h, cudaEventRecord(h->ev[0], s));
    if (opt_geometry && N > 0) {   // UpdateSurfelNormalsCUDA, :215-227
      bba::GeometryArgs g;
      if (bba_status st = BuildGeometryArgs(h, &g, s)) return st;
      bba::LaunchActivationAndNormals(g, h->sm_count, false, true, s);
      ++h->launches;
      if (bba_status st = ExchangeGeometry(h, s)) return st;   // multi-GPU: every replica gets the other shards' normals
    }
    BBA_CUDA(h, cudaEventRecord(h->ev[1], s));

    if (bba_status st = MakePcgLayout(h, o, &L)) return st;   // unknown layout (:273-309)
    const uint32_t surfel_start = L.surfel_start, depth_start = L.depth_start, a_index = L.a_index, color_start = L.color_start;
    const uint32_t unknown_count = L.unknown_count;
    float *pcg_r = h->d_pcg[0], *pcg_M = h->d_pcg[1], *pcg_delta = h->d_pcg[2], *pcg_g = h->d_pcg[3], *pcg_p = h->d_pcg[4];
    const int gauge = o->pcg_gauge_keyframe >= 0 ? o->pcg_gauge_keyframe : (rand() % K);   // :324

    int num_converged = 0;
    if (unknown_count > 0) {
      BBA_CUDA(h, cudaMemsetAsync(pcg_r, 0, sizeof(float) * unknown_count, s));   // :312-313
      BBA_CUDA(h, cudaMemsetAsync(pcg_M, 0, sizeof(float) * unknown_count, s));
      BBA_CUDA(h, cudaMemsetAsync(h->d_pcg_scalars, 0, sizeof(double) * 4, s));
      const bba::PcgArgs a = MakePcgArgs(h, L, gauge);
      bba::LaunchPcgAccumulate(a, h->sm_count, true, s);   // PCGInitCUDA for every keyframe, :336-361
      if (world > 1) {
        h->collective(h->collective_user, BBA_COLLECTIVE_ALLREDUCE_SUM, pcg_r, unknown_count, s);
        h->collective(h->collective_user, BBA_COLLECTIVE_ALLREDUCE_SUM, pcg_M, unknown_count, s);
        h->replicated_pass_pending = false;
      }
      int an = 0, bn = 2;
      bba::LaunchPcgInit2(unknown_count, a_index, h->depth_a, K, pcg_r, pcg_M, pcg_delta, pcg_g, pcg_p, h->d_pcg_scalars, an,
                          h->sm_count, s);   // :363-373
      h->launches += 2;
      float prev_r_norm = std::numeric_limits<float>::infinity();
      int without_improvement = 0;
      for (int step = 0; step < max_inner; ++step) {
        if (step > 0) std::swap(an, bn);   // alpha_n <- beta_n (:386); g was cleared and alpha_d re-armed by PcgStep3Kernel
        bba::LaunchPcgAccumulate(a, h->sm_count, false, s);   // PCGStep1CUDA for every keyframe, :392-419
        if (world > 1) {   // g and this rank's part of alpha_d: one all-reduce
          bba::LaunchPcgPackAlphaD(h->d_pcg_scalars, pcg_g + unknown_count, s);
          h->collective(h->collective_user, BBA_COLLECTIVE_ALLREDUCE_SUM, pcg_g, static_cast<size_t>(unknown_count) + 2, s);
          bba::LaunchPcgUnpackAlphaD(h->d_pcg_scalars, pcg_g + unknown_count, s);
          h->launches += 2;
        }
        BBA_CUDA(h, cudaMemsetAsync(h->d_pcg_scalars + bn, 0, sizeof(double), s));
        bba::LaunchPcgStep2(unknown_count, a_index, pcg_r, pcg_M, pcg_delta, pcg_g, pcg_p, h->d_pcg_scalars, an, bn, h->sm_count, s);
        h->launches += 2;
        BBA_CUDA(h, cudaGetLastError());
        BBA_CUDA(h, cudaMemcpyAsync(h->h_pcg_scalars, h->d_pcg_scalars, sizeof(double) * 4, cudaMemcpyDeviceToHost, s));
        BBA_CUDA(h, cudaStreamSynchronize(s));   // :436-437
        ++res->pcg_inner_iterations_total;
        const float r_norm = std::sqrt(static_cast<float>(h->h_pcg_scalars[bn]));
        res->pcg_last_r_norm = r_norm;
        if (static_cast<double>(r_norm) < static_cast<double>(prev_r_norm) - 1e-3) {   // :442-449
          without_improvement = 0;
        } else if (++without_improvement >= 3) {
          break;
        }
        prev_r_norm = r_norm;
        if (step < max_inner - 1) {   // :456-464
          BBA_CUDA(h, cudaMemsetAsync(h->d_pcg_scalars + 1, 0, sizeof(double), s));
          bba::LaunchPcgStep3(unknown_count, a_index, K, pcg_g, pcg_p, h->d_pcg_scalars, an, bn, h->sm_count, s);
          ++h->launches;
        }
      }
      BBA_CUDA(h, cudaEventRecord(h->ev[2], s));

      // --- apply pcg_delta (:552-638)
      size_t n_host = 0;
      const size_t pose_floats = opt_poses ? 6 * static_cast<size_t>(K - 1) : 0;
      if (pose_floats) BBA_CUDA(h, cudaMemcpyAsync(h->h_pcg_delta, pcg_delta, sizeof(float) * pose_floats, cudaMemcpyDeviceToHost, s));
      n_host = pose_floats;
      float* h_di = h->h_pcg_delta + n_host;
      if (opt_depth_intr) {
        BBA_CUDA(h, cudaMemcpyAsync(h_di, pcg_delta + depth_start, sizeof(float) * 5, cudaMemcpyDeviceToHost, s));
        n_host += 5;
      }
      float* h_ci = h->h_pcg_delta + n_host;
      if (opt_color_intr) BBA_CUDA(h, cudaMemcpyAsync(h_ci, pcg_delta + color_start, sizeof(float) * 4, cudaMemcpyDeviceToHost, s));
      if (opt_geometry && N > 0) {
        bba::LaunchPcgUpdateSurfels(h->surfels, a.pitch, N, use_desc, surfel_start, pcg_delta, s);
        ++h->launches;
        h->replicated_pass_pending = true;   // every rank rewrites its whole replica (PeerFence)
      }
      if (opt_depth_intr) {
        bba::LaunchPcgUpdateCfactor(h->d_cfactor, P, pcg_delta + depth_start + 5, s);
        ++h->launches;
      }
      BBA_CUDA(h, cudaGetLastError());
      BBA_CUDA(h, cudaStreamSynchronize(s));
      if (opt_poses) {
        for (int k = 0; k < K; ++k) {
          if (k == gauge) {
            ++num_converged;
            continue;
          }
          const float* d6 = h->h_pcg_delta + 6 * static_cast<size_t>(k < gauge ? k : k - 1);
          const Pose delta = bba::Exp(d6);
          h->keyframes[k].pose = bba::Compose(h->keyframes[k].pose, delta);   // :569-570
          float lg[6];
          bba::Log(delta, lg);
          if (bba::IsScale1PoseEstimationConverged(lg)) ++num_converged;
        }
      }
      if (opt_depth_intr) {   // :590-612
        const double old_fx_inv = 1. / h->depth_K[0], old_fy_inv = 1. / h->depth_K[1];
        const double old_cx_inv = -(h->depth_K[2] - 0.5) * old_fx_inv, old_cy_inv = -(h->depth_K[3] - 0.5) * old_fy_inv;
        const double new_fx = 1. / (old_fx_inv + h_di[0]);
        const double new_fy = 1. / (old_fy_inv + h_di[1]);
        const double new_cx = -(new_fx * (old_cx_inv + h_di[2])) + 0.5;
        const double new_cy = -(new_fy * (old_cy_inv + h_di[3])) + 0.5;
        h->depth_K[0] = static_cast<float>(new_fx);
        h->depth_K[1] = static_cast<float>(new_fy);
        h->depth_K[2] = static_cast<float>(new_cx);
        h->depth_K[3] = static_cast<float>(new_cy);
        h->depth_a += h_di[4];
      }
      if (opt_color_intr)   // :623-638
        for (int c = 0; c < 4; ++c) h->color_K[c] = static_cast<float>(h->color_K[c] + h_ci[c]);
      // surfel merge + compaction (:644-690) for the keyframes that received new surfels
      if (o->do_surfel_updates && !keyframes_with_new_surfels.empty()) {
        uint32_t merged = 0;
        for (int k : keyframes_with_new_surfels) {
          uint32_t d = 0;
          if (bba_status st = MergeSurfelsForKeyframe(h, k, s, &d)) return st;
          merged += d;
        }
        res->surfels_merged += merged;
        if (bba_status st = CompactSurfels(h, merged, /*with_active=*/true, s)) return st;
      }
    } else {
      BBA_CUDA(h, cudaEventRecord(h->ev[2], s));
      BBA_CUDA(h, cudaStreamSynchronize(s));
      num_converged = opt_poses ? 1 : 0;
    }
    cudaEventElapsedTime(&res->ms_geometry_optimization, h->ev[0], h->ev[1]);   // "BA normals update", :722-727
    cudaEventElapsedTime(&res->ms_pcg, h->ev[1], h->ev[2]);

    if (iteration >= o->min_iterations - 1 && (num_converged == K || !opt_poses)) {   // :757-766
      res->converged = 1;
      break;
    }
    if (o->time_limit_seconds > 0) {
      const double el = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_start).count();
      if (el > o->time_limit_seconds) break;
    }
  }
  if (o->increase_ba_iteration_count) {   // :771-776
    uint32_t deleted = 0;
    if (bba_status st = PerformEndTasks(h, s, &deleted, o->do_surfel_updates != 0)) return st;
    res->surfels_deleted += deleted;
    ++h->ba_iteration_count;
  } else if (o->do_surfel_updates && !keyframes_with_new_surfels.empty()) {
    // :775-815: without the end tasks, the keyframes of the last iteration's creation step are merged (and the map compacted) once more
    uint32_t merged = 0;
    for (int k : keyframes_with_new_surfels) {
      uint32_t d = 0;
      if (bba_status st = MergeSurfelsForKeyframe(h, k, s, &d)) return st;
      merged += d;
    }
    res->surfels_merged += merged;
    if (bba_status st = CompactSurfels(h, merged, /*with_active=*/true, s)) return st;
  }
  res->surfels_size = h->surfels_size;
  res->kernel_launches = h->launches - launches_before;
  return BBA_OK;
}

// The u8 staging plane is shared by every keyframe / frame upload of the handle.  Calls may arrive on different streams (the
// reference's tracking thread and BA thread use their own, bad_slam.cc:73-78,1197-1200): the next user waits until the previous
// copy-to-array has consumed the plane.
bba_status AcquireLumaStaging(bba_handle h, cudaStream_t s) {
  if (!h->luma_staging_free) BBA_CUDA(h, cudaEventCreateWithFlags(&h->luma_staging_free, cudaEventDisableTiming));
  else BBA_CUDA(h, cudaStreamWaitEvent(s, h->luma_staging_free, 0));
  return BBA_OK;
}

// The luma plane (the .w channel of a uchar4 image) as a gather-enabled CUDA array (block-linear: 2-D locality for the sample
// footprints) + a texture with the reference's sampling state (keyframe.cc:67-73).  *array / *tex are created when null and
// refilled otherwise.
bba_status MakeLumaTexture(bba_handle h, const uint8_t* device_rgba, size_t color_pitch, cudaArray_t* array, cudaTextureObject_t* tex_out,
                           cudaStream_t s) {
  const int cw = h->cfg.color_width, ch = h->cfg.color_height;
  if (!h->luma_staging)
    BBA_CUDA(h, cudaMallocPitch(reinterpret_cast<void**>(&h->luma_staging), &h->luma_staging_pitch, cw, ch));
  if (bba_status st = AcquireLumaStaging(h, s)) return st;
  if (!*array) {
    const cudaChannelFormatDesc desc = cudaCreateChannelDesc(8, 0, 0, 0, cudaChannelFormatKindUnsigned);
    BBA_CUDA(h, cudaMallocArray(array, &desc, cw, ch, cudaArrayTextureGather));
  }
  bba::LaunchExtractLuma(device_rgba, color_pitch, h->luma_staging, h->luma_staging_pitch, cw, ch, s);
  ++h->launches;
  BBA_CUDA(h, cudaGetLastError());
  BBA_CUDA(h, cudaMemcpy2DToArrayAsync(*array, 0, 0, h->luma_staging, h->luma_staging_pitch, cw, ch, cudaMemcpyDeviceToDevice, s));
  BBA_CUDA(h, cudaEventRecord(h->luma_staging_free, s));
  if (!*tex_out) {
    cudaResourceDesc res;
    std::memset(&res, 0, sizeof(res));
    res.resType = cudaResourceTypeArray;
    res.res.array.array = *array;
    cudaTextureDesc tex;
    std::memset(&tex, 0, sizeof(tex));
    tex.addressMode[0] = cudaAddressModeClamp;
    tex.addressMode[1] = cudaAddressModeClamp;
    tex.filterMode = cudaFilterModeLinear;
    tex.readMode = cudaReadModeNormalizedFloat;
    tex.normalizedCoords = 0;
    BBA_CUDA(h, cudaCreateTextureObject(tex_out, &res, &tex, nullptr));
  }
  return BBA_OK;
}

// ---- image-pair odometry (bba_track_frame_pairwise) --------------------------------------------------------------------
void FreeOdometry(bba_handle h) {
  auto& o = h->odo;
  for (int f = 0; f < 2; ++f) {
    if (o.gradmag_tex[f]) cudaDestroyTextureObject(o.gradmag_tex[f]);
    cudaFree(o.gradmag[f]);
    o.gradmag_tex[f] = 0;
    o.gradmag[f] = nullptr;
    for (int s = 0; s < bba::odom::kMaxScales; ++s) {
      bba::odom::Image& im = o.image[f][s];
      if (im.color_tex) cudaDestroyTextureObject(im.color_tex);
      cudaFree(im.depth);
      if (o.owns_normals[f][s]) cudaFree(im.normals);
      cudaFree(im.color);
      im = bba::odom::Image{};
      o.owns_normals[f][s] = false;
    }
  }
  cudaFree(o.d_acc);
  cudaFree(o.d_barrier);
  cudaFree(o.d_result);
  if (o.h_result) cudaFreeHost(o.h_result);
  o.d_acc = nullptr; o.d_barrier = nullptr; o.d_result = nullptr; o.h_result = nullptr;
  o.num_scales = 0;
  o.last_num_scales = 0;
}

// A u8 plane in pitched device memory as a texture with the sampler state of CUDABuffer::CreateTextureObject as the reference
// calls it for the pyramid colour planes (pairwise_frame_tracking.cc:57-79): clamp, linear, normalised float, unnormalised coordinates.
bba_status MakePitchedU8Texture(bba_handle h, uint8_t* data, size_t pitch, int w, int ht, cudaTextureObject_t* out) {
  cudaResourceDesc res;
  std::memset(&res, 0, sizeof(res));
  res.resType = cudaResourceTypePitch2D;
  res.res.pitch2D.devPtr = data;
  res.res.pitch2D.desc = cudaCreateChannelDesc(8, 0, 0, 0, cudaChannelFormatKindUnsigned);
  res.res.pitch2D.width = w;
  res.res.pitch2D.height = ht;
  res.res.pitch2D.pitchInBytes = pitch;
  cudaTextureDesc tex;
  std::memset(&tex, 0, sizeof(tex));
  tex.addressMode[0] = cudaAddressModeClamp;
  tex.addressMode[1] = cudaAddressModeClamp;
  tex.filterMode = cudaFilterModeLinear;
  tex.readMode = cudaReadModeNormalizedFloat;
  tex.normalizedCoords = 0;
  BBA_CUDA(h, cudaCreateTextureObject(out, &res, &tex, nullptr));
  return BBA_OK;
}

// PairwiseFrameTrackingBuffers + CreatePairwiseTrackingInputBuffersAndTextures (pairwise_frame_tracking.cc:39-151)
bba_status EnsureOdometry(bba_handle h, int num_scales) {
  auto& o = h->odo;
  if (o.num_scales >= num_scales) return BBA_OK;
  FreeOdometry(h);
  const int cw = h->cfg.color_width, ch = h->cfg.color_height;
  for (int f = 0; f < 2; ++f) {
    BBA_CUDA(h, cudaMallocPitch(reinterpret_cast<void**>(&o.gradmag[f]), &o.gradmag_pitch[f], cw, ch));
    if (bba_status st = MakePitchedU8Texture(h, o.gradmag[f], o.gradmag_pitch[f], cw, ch, &o.gradmag_tex[f])) return st;
  }
  for (int s = 0; s < num_scales; ++s) {
    // pairwise_frame_tracking.cc:51-53: int scale_width = depth_width / pow(2, scale)
    o.w[s] = static_cast<int>(h->cfg.depth_width / std::pow(2, s));
    o.h[s] = static_cast<int>(h->cfg.depth_height / std::pow(2, s));
    if (o.w[s] < 1 || o.h[s] < 1) return Fail(h, BBA_ERR_INVALID_ARGUMENT, "bba_track_frame_pairwise: too many pyramid levels for this image size");
    for (int f = 0; f < 2; ++f) {
      bba::odom::Image& im = o.image[f][s];
      size_t pitch = 0;
      BBA_CUDA(h, cudaMallocPitch(reinterpret_cast<void**>(&im.depth), &pitch, sizeof(float) * o.w[s], o.h[s]));
      im.depth_pitch = static_cast<uint32_t>(pitch / sizeof(float));
      if (s >= 1) {   // level 0 uses the caller's normal images
        BBA_CUDA(h, cudaMallocPitch(reinterpret_cast<void**>(&im.normals), &pitch, sizeof(uint16_t) * o.w[s], o.h[s]));
        im.normals_pitch = static_cast<uint32_t>(pitch);
        o.owns_normals[f][s] = true;
      }
      BBA_CUDA(h, cudaMallocPitch(reinterpret_cast<void**>(&im.color), &pitch, o.w[s], o.h[s]));
      im.color_pitch = static_cast<uint32_t>(pitch);
      if (bba_status st = MakePitchedU8Texture(h, im.color, pitch, o.w[s], o.h[s], &im.color_tex)) return st;
    }
  }
  BBA_CUDA(h, cudaMalloc(&o.d_acc, sizeof(double) * 96));
  BBA_CUDA(h, cudaMalloc(&o.d_barrier, sizeof(unsigned int) * 2));
  BBA_CUDA(h, cudaMalloc(&o.d_result, sizeof(bba::odom::TrackResult)));
  BBA_CUDA(h, cudaMallocHost(&o.h_result, sizeof(bba::odom::TrackResult)));
  o.num_scales = num_scales;
  return BBA_OK;
}

// The camera model of one pyramid level: PinholeCamera4f::Scaled (libvis camera.h:1696-1705, 1086-1097: all four parameters
// times the factor, width = factor * width + 0.5) through the builders of surfel_projection.h:42-124.
bba::odom::LevelCamera MakeLevelCamera(bba_handle h, int scale, int level_w, int level_h) {
  bba::odom::LevelCamera c;
  const float scaling_factor = static_cast<float>(std::pow(2, scale));
  const float df = static_cast<float>(1.f / scaling_factor);   // depth_camera.Scaled(1.f / scaling_factor)
  const float cf = static_cast<float>((h->cfg.depth_width == h->cfg.color_width) ? (1.f / scaling_factor) : (2.f / scaling_factor));
  const float dK[4] = {h->depth_K[0] * df, h->depth_K[1] * df, h->depth_K[2] * df, h->depth_K[3] * df};
  const float cK[4] = {h->color_K[0] * cf, h->color_K[1] * cf, h->color_K[2] * cf, h->color_K[3] * cf};
  c.w = level_w; c.h = level_h;
  c.fx = dK[0]; c.fy = dK[1]; c.cx = dK[2]; c.cy = dK[3];
  c.fx_inv = 1.0f / dK[0];
  c.fy_inv = 1.0f / dK[1];
  c.cx_inv = -(dK[2] - 0.5f) * c.fx_inv;
  c.cy_inv = -(dK[3] - 0.5f) * c.fy_inv;
  c.d2c_fx = cK[0] / dK[0];
  c.d2c_cx = -1 * cK[0] * dK[2] / dK[0] + cK[2];
  c.d2c_fy = cK[1] / dK[1];
  c.d2c_cy = -1 * cK[1] * dK[3] / dK[1] + cK[3];
  c.cw = static_cast<int>(static_cast<double>(cf) * h->cfg.color_width + 0.5f);
  c.ch = static_cast<int>(static_cast<double>(cf) * h->cfg.color_height + 0.5f);
  c.cfx = cK[0]; c.cfy = cK[1];
  return c;
}

bba_status AddKeyframeCommon(bba_handle h, Keyframe&& kf, const uint8_t* device_rgba, size_t color_pitch, const float pose[7],
                             float min_depth, float max_depth, cudaStream_t s, int* out_id) {
  if (static_cast<int>(h->keyframes.size()) >= h->cfg.max_keyframes) return Fail(h, BBA_ERR_STATE, "max_keyframes exceeded");
  // (development switch for the locality A/B of tools/ab_locality.py: every keyframe samples keyframe 0's luma array)
  static const bool alias_luma = std::getenv("BADBA_ALIAS_LUMA") != nullptr;
  if (alias_luma && !h->keyframes.empty()) {
    kf.tex = h->keyframes[0].tex;
    kf.tex_alias = true;
  } else if (bba_status st = MakeLumaTexture(h, device_rgba, color_pitch, &kf.luma, &kf.tex, s)) {
    return st;
  }
  kf.pose = PoseFromArray(pose);
  kf.activation = BBA_KF_ACTIVE;   // keyframe.cc:75
  kf.min_depth = min_depth;
  kf.max_depth = max_depth;
  MakeFrustum(&kf.frustum, h->depth_K, h->cfg.depth_width, h->cfg.depth_height, min_depth, max_depth, kf.pose);
  const int id = static_cast<int>(h->keyframes.size());
  // DetermineNewKeyframeCoVisibility, direct_ba.cc:231-249
  for (int k = 0; k < id; ++k) {
    Keyframe& other = h->keyframes[k];
    Frustum other_frustum;
    MakeFrustum(&other_frustum, h->depth_K, h->cfg.depth_width, h->cfg.depth_height, other.min_depth, other.max_depth, other.pose);
    if (FrustaIntersect(kf.frustum, other_frustum)) {
      kf.covis.push_back(k);
      other.covis.push_back(id);
      if (other.activation == BBA_KF_INACTIVE) other.activation = BBA_KF_COVISIBLE_ACTIVE;
    }
  }
  h->keyframes.push_back(std::move(kf));
  if (out_id) *out_id = id;
  return BBA_OK;
}

}  // namespace

extern "C" {

int bba_abi_version(void) { return BBA_ABI_VERSION; }

const char* bba_last_error(bba_handle h) { return h ? h->error.c_str() : "null handle"; }

bba_status bba_create(const bba_config* cfg, bba_handle* out) {
  if (!cfg || !out) return BBA_ERR_INVALID_ARGUMENT;
  *out = nullptr;
  if (cfg->depth_width <= 0 || cfg->depth_height <= 0 || cfg->color_width <= 0 || cfg->color_height <= 0 ||
      cfg->sparse_surfel_cell_size <= 0 || cfg->max_keyframes <= 0 || cfg->world_size <= 0 || cfg->rank < 0 ||
      cfg->rank >= cfg->world_size || (!cfg->use_depth_residuals && !cfg->use_descriptor_residuals))
    return BBA_ERR_INVALID_ARGUMENT;
  int device_count = 0;
  if (cudaGetDeviceCount(&device_count) != cudaSuccess || device_count == 0) {
    cudaGetLastError();
    return BBA_ERR_NO_DEVICE;   // no CPU fallback exists, by design
  }
  bba_handle h = new bba_context();
  h->cfg = *cfg;
  std::memcpy(h->depth_K, cfg->depth_intrinsics, sizeof(h->depth_K));
  std::memcpy(h->color_K, cfg->color_intrinsics, sizeof(h->color_K));
  h->cf_w = (cfg->depth_width - 1) / cfg->sparse_surfel_cell_size + 1;    // direct_ba.cc:110-113
  h->cf_h = (cfg->depth_height - 1) / cfg->sparse_surfel_cell_size + 1;
  auto fail = [&](const char* what, cudaError_t e) {
    std::fprintf(stderr, "bba_create: %s: %s\n", what, cudaGetErrorString(e));
    bba_destroy(h);
    return BBA_ERR_CUDA;
  };
#define CREATE_TRY(expr)                           \
  do {                                             \
    cudaError_t e__ = (expr);                      \
    if (e__ != cudaSuccess) return fail(#expr, e__); \
  } while (0)
  CREATE_TRY(cudaSetDevice(cfg->device));
  cudaDeviceProp prop;
  CREATE_TRY(cudaGetDeviceProperties(&prop, cfg->device));
  h->sm_count = prop.multiProcessorCount;
  const size_t K = static_cast<size_t>(cfg->max_keyframes);
  CREATE_TRY(cudaMalloc(&h->d_cfactor, sizeof(float) * h->cf_w * h->cf_h));
  CREATE_TRY(cudaMemset(h->d_cfactor, 0, sizeof(float) * h->cf_w * h->cf_h));
  CREATE_TRY(cudaMalloc(&h->d_kfs, sizeof(KfDevice) * K));
  CREATE_TRY(cudaMalloc(&h->d_work_records, sizeof(KfDevice) * K));
  CREATE_TRY(cudaMalloc(&h->d_pose_est, sizeof(float) * 7 * K));
  CREATE_TRY(cudaMalloc(&h->d_acc, sizeof(double) * bba::kPoseAccSize * K));
  CREATE_TRY(cudaMemset(h->d_acc, 0, sizeof(double) * bba::kPoseAccSize * K));
  CREATE_TRY(cudaMalloc(&h->d_stage_counts, sizeof(unsigned long long) * 2 * K));
  CREATE_TRY(cudaMemset(h->d_stage_counts, 0, sizeof(unsigned long long) * 2 * K));
  CREATE_TRY(cudaMalloc(&h->d_work[0], sizeof(int) * K));
  CREATE_TRY(cudaMalloc(&h->d_work[1], sizeof(int) * K));
  CREATE_TRY(cudaMalloc(&h->d_count, sizeof(int) * 2));
  CREATE_TRY(cudaMalloc(&h->d_iterations, sizeof(int) * K));
  CREATE_TRY(cudaMalloc(&h->d_converged, sizeof(int) * K));
  CREATE_TRY(cudaMalloc(&h->d_first_stats, sizeof(double) * 8 * K));
  CREATE_TRY(cudaMemset(h->d_first_stats, 0, sizeof(double) * 8 * K));
  CREATE_TRY(cudaMalloc(&h->d_geo_list, sizeof(int) * K));
  CREATE_TRY(cudaMalloc(&h->d_geo_queue, sizeof(unsigned int)));
  CREATE_TRY(cudaMalloc(&h->d_pose_pack, sizeof(float) * bba::kPoseSlot * K));
  CREATE_TRY(cudaMallocHost(&h->h_pose_pack, sizeof(float) * bba::kPoseSlot * K));
  CREATE_TRY(cudaMalloc(&h->d_local_ids, sizeof(int) * K));
  CREATE_TRY(cudaMalloc(&h->d_queue, sizeof(unsigned int)));
  CREATE_TRY(cudaMemset(h->d_queue, 0, sizeof(unsigned int)));
  CREATE_TRY(cudaMalloc(&h->d_totals, sizeof(unsigned long long) * 8));
  CREATE_TRY(cudaMemset(h->d_totals, 0, sizeof(unsigned long long) * 8));
  {
    int* flag = nullptr;
    CREATE_TRY(cudaHostAlloc(&flag, sizeof(int) * 4, cudaHostAllocMapped));
    flag[0] = flag[1] = flag[2] = flag[3] = 0;
    h->h_flag = flag;
    CREATE_TRY(cudaHostGetDevicePointer(&h->d_flag, flag, 0));
  }
  CREATE_TRY(cudaMallocHost(&h->h_totals, sizeof(unsigned long long) * 8));
  std::memset(&h->profile, 0, sizeof(h->profile));
  for (auto& e : h->prof_ev) e = nullptr;
  for (auto& e : h->prof_ev) CREATE_TRY(cudaEventCreate(&e));
  CREATE_TRY(cudaMallocHost(&h->h_kfs, sizeof(KfDevice) * K));
  CREATE_TRY(cudaMallocHost(&h->h_pose_est, sizeof(float) * 7 * K));
  CREATE_TRY(cudaMallocHost(&h->h_work, sizeof(int) * (K + 2)));
  CREATE_TRY(cudaMallocHost(&h->h_geo_list, sizeof(int) * K));
  CREATE_TRY(cudaMallocHost(&h->h_iterations, sizeof(int) * K));
  CREATE_TRY(cudaMallocHost(&h->h_converged, sizeof(int) * K));
  CREATE_TRY(cudaMallocHost(&h->h_first_stats, sizeof(double) * 8 * K));
  CREATE_TRY(cudaMallocHost(&h->h_acc, sizeof(double) * (bba::kPoseAccSize + 2)));
  CREATE_TRY(cudaEventCreateWithFlags(&h->staging_event, cudaEventDisableTiming));
  for (auto& e : h->ev) CREATE_TRY(cudaEventCreate(&e));
#undef CREATE_TRY
  h->keyframes.reserve(K);
  *out = h;
  return BBA_OK;
}

void bba_destroy(bba_handle h) {
  if (!h) return;
  cudaDeviceSynchronize();
  for (Keyframe& kf : h->keyframes) {
    if (kf.tex && !kf.tex_alias) cudaDestroyTextureObject(kf.tex);
    if (kf.luma) cudaFreeArray(kf.luma);
    for (void* p : kf.owned) cudaFree(p);
    cudaFree(kf.owned_rgba);
  }
  cudaFree(h->owned_surfels);
  cudaFree(h->owned_active);
  cudaFree(h->d_cfactor);
  cudaFree(h->color_staging);
  cudaFree(h->luma_staging);
  if (h->luma_staging_free) cudaEventDestroy(h->luma_staging_free);
  cudaFree(h->d_kfs);
  cudaFree(h->d_work_records);
  cudaFree(h->d_frames);
  cudaFree(h->d_pose_est);
  cudaFree(h->d_acc);
  cudaFree(h->d_stage_counts);
  cudaFree(h->d_work[0]);
  cudaFree(h->d_work[1]);
  cudaFree(h->d_count);
  cudaFree(h->d_iterations);
  cudaFree(h->d_converged);
  cudaFree(h->d_first_stats);
  cudaFree(h->d_geo_list);
  cudaFree(h->d_totals);
  cudaFree(h->d_queue);
  cudaFree(h->d_geo_queue);
  cudaFree(h->d_exchange);
  cudaFree(h->d_pose_pack);
  cudaFreeHost(h->h_pose_pack);
  cudaFree(h->d_local_ids);
  cudaFree(h->d_tile_epoch);
  cudaFree(h->d_intr);
  cudaFree(h->d_intr_sums);
  cudaFree(h->d_all_list);
  cudaFreeHost(h->h_intr_sums);
  cudaFreeHost(h->h_intr_x1);
  UnmapPeers(h);
  cudaFree(h->d_barrier);
  cudaFree(h->d_sup);
  cudaFree(h->d_cell_bits);
  cudaFree(h->d_flags);
  cudaFree(h->d_scan_out);
  cudaFree(h->d_scan_sums);
  cudaFree(h->d_covis);
  cudaFreeHost(h->h_covis);
  cudaFree(h->d_kf_radius);
  cudaFreeHost(h->h_kf_radius);
  cudaFree(h->d_deleted_count);
  cudaFree(h->d_count_xchg);
  if (h->h_count_xchg) cudaFreeHost(h->h_count_xchg);
  cudaFreeHost(h->h_deleted_count);
  cudaFree(h->d_compact_sums);
  cudaFree(h->d_min_max);
  cudaFreeHost(h->h_min_max);
  FreeOdometry(h);
  if (h->scratch_tex) cudaDestroyTextureObject(h->scratch_tex);
  if (h->scratch_luma) cudaFreeArray(h->scratch_luma);
  for (float* v : h->d_pcg) cudaFree(v);
  cudaFree(h->d_pcg_scalars);
  cudaFreeHost(h->h_pcg_scalars);
  cudaFreeHost(h->h_pcg_delta);
  if (h->h_flag) cudaFreeHost(const_cast<int*>(h->h_flag));
  cudaFreeHost(h->h_totals);
  for (auto& e : h->prof_ev)
    if (e) cudaEventDestroy(e);
  cudaFreeHost(h->h_kfs);
  cudaFreeHost(h->h_pose_est);
  cudaFreeHost(h->h_work);
  cudaFreeHost(h->h_geo_list);
  cudaFreeHost(h->h_iterations);
  cudaFreeHost(h->h_converged);
  cudaFreeHost(h->h_first_stats);
  cudaFreeHost(h->h_acc);
  if (h->staging_event) cudaEventDestroy(h->staging_event);
  for (auto& e : h->ev)
    if (e) cudaEventDestroy(e);
  delete h;
}

bba_status bba_set_surfels(bba_handle h, float* device_surfels, size_t pitch_bytes, uint32_t surfels_size) {
  if (h && (device_surfels != h->surfels || pitch_bytes != h->surfel_pitch_bytes)) UnmapPeers(h);
  if (!h) return BBA_ERR_INVALID_ARGUMENT;
  if (!device_surfels || pitch_bytes % 16 != 0 || (reinterpret_cast<uintptr_t>(device_surfels) & 15) != 0 ||
      pitch_bytes < static_cast<size_t>((surfels_size + 3) / 4) * 16 || surfels_size > h->cfg.max_surfel_count)
    return Fail(h, BBA_ERR_INVALID_ARGUMENT,
                "surfel buffer must be 16-byte aligned with a row pitch that is a multiple of 16 bytes and holds surfels_size floats");
  h->surfels = device_surfels;
  h->surfel_pitch_bytes = pitch_bytes;
  h->surfels_size = surfels_size;
  return BBA_OK;
}

bba_status bba_set_active_flags(bba_handle h, uint8_t* device_flags) {
  if (h && device_flags != h->active) UnmapPeers(h);
  if (!h || !device_flags) return BBA_ERR_INVALID_ARGUMENT;
  h->active = device_flags;
  return BBA_OK;
}

bba_status bba_set_surfels_host(bba_handle h, const float* host_surfels, size_t pitch_bytes, uint32_t surfels_size, void* stream) {
  if (!h || !host_surfels) return BBA_ERR_INVALID_ARGUMENT;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (!h->owned_surfels) {
    const size_t pitch = (static_cast<size_t>(h->cfg.max_surfel_count) * 4 + 511) / 512 * 512;
    BBA_CUDA(h, cudaMalloc(&h->owned_surfels, pitch * bba::kSurfelRowCount));
    BBA_CUDA(h, cudaMalloc(&h->owned_active, h->cfg.max_surfel_count));
    BBA_CUDA(h, cudaMemsetAsync(h->owned_active, 0, h->cfg.max_surfel_count, s));
    h->owned_surfel_pitch = pitch;
  }
  if (surfels_size > h->cfg.max_surfel_count || pitch_bytes < static_cast<size_t>(surfels_size) * 4)
    return Fail(h, BBA_ERR_INVALID_ARGUMENT, "surfels_size exceeds max_surfel_count or the host pitch");
  // only the 8 data rows are inputs (kSurfelDataAttributeCount, kernels.cuh:89); rows 8-16 are scratch
  BBA_CUDA(h, cudaMemcpy2DAsync(h->owned_surfels, h->owned_surfel_pitch, host_surfels, pitch_bytes,
                                static_cast<size_t>(surfels_size) * 4, 8, cudaMemcpyHostToDevice, s));
  if (bba_status st = bba_set_surfels(h, h->owned_surfels, h->owned_surfel_pitch, surfels_size)) return st;
  return bba_set_active_flags(h, h->owned_active);
}

bba_status bba_get_surfels_host(bba_handle h, float* host_surfels, size_t pitch_bytes, int rows, void* stream) {
  if (!h || !host_surfels || rows < 1 || rows > bba::kSurfelRowCount) return BBA_ERR_INVALID_ARGUMENT;
  if (bba_status st = CheckSurfels(h)) return st;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  BBA_CUDA(h, cudaMemcpy2DAsync(host_surfels, pitch_bytes, h->surfels, h->surfel_pitch_bytes,
                                static_cast<size_t>(h->surfels_size) * 4, rows, cudaMemcpyDeviceToHost, s));
  BBA_CUDA(h, cudaStreamSynchronize(s));
  return BBA_OK;
}

bba_status bba_get_active_flags_host(bba_handle h, uint8_t* host_flags, void* stream) {
  if (!h || !host_flags) return BBA_ERR_INVALID_ARGUMENT;
  if (bba_status st = CheckSurfels(h)) return st;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  BBA_CUDA(h, cudaMemcpyAsync(host_flags, h->active, h->surfels_size, cudaMemcpyDeviceToHost, s));
  BBA_CUDA(h, cudaStreamSynchronize(s));
  return BBA_OK;
}

bba_status bba_get_surfels_device(bba_handle h, float** device_surfels, size_t* pitch_bytes, uint32_t* surfels_size) {
  if (!h) return BBA_ERR_INVALID_ARGUMENT;
  if (device_surfels) *device_surfels = h->surfels;
  if (pitch_bytes) *pitch_bytes = h->surfel_pitch_bytes;
  if (surfels_size) *surfels_size = h->surfels_size;
  return BBA_OK;
}

bba_status bba_add_keyframe(bba_handle h, const uint16_t* device_depth, size_t depth_pitch, const uint16_t* device_normals,
                            size_t normals_pitch, const uint16_t* device_radius, size_t radius_pitch,
                            const uint8_t* device_color_rgba, size_t color_pitch, const float global_T_frame[7], float min_depth,
                            float max_depth, void* stream, int* out_keyframe_id) {
  if (!h || !device_depth || !device_normals || !device_color_rgba || !global_T_frame) return BBA_ERR_INVALID_ARGUMENT;
  if (depth_pitch < static_cast<size_t>(h->cfg.depth_width) * 2 || normals_pitch < static_cast<size_t>(h->cfg.depth_width) * 2 ||
      color_pitch < static_cast<size_t>(h->cfg.color_width) * 4 || depth_pitch > 0xffffffffull || normals_pitch > 0xffffffffull)
    return Fail(h, BBA_ERR_INVALID_ARGUMENT, "keyframe buffer pitch too small");
  Keyframe kf;
  kf.depth = device_depth; kf.depth_pitch = depth_pitch;
  kf.normals = device_normals; kf.normals_pitch = normals_pitch;
  kf.radius = device_radius; kf.radius_pitch = radius_pitch;
  kf.rgba = device_color_rgba; kf.rgba_pitch = color_pitch;
  return AddKeyframeCommon(h, std::move(kf), device_color_rgba, color_pitch, global_T_frame, min_depth, max_depth,
                           static_cast<cudaStream_t>(stream), out_keyframe_id);
}

bba_status bba_add_keyframe_host(bba_handle h, const uint16_t* host_depth, const uint16_t* host_normals, const uint16_t* host_radius,
                                 const uint8_t* host_color_rgba, const float global_T_frame[7], float min_depth, float max_depth,
                                 void* stream, int* out_keyframe_id) {
  if (!h || !host_depth || !host_normals || !host_color_rgba || !global_T_frame) return BBA_ERR_INVALID_ARGUMENT;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int w = h->cfg.depth_width, hh = h->cfg.depth_height, cw = h->cfg.color_width, ch = h->cfg.color_height;
  Keyframe kf;
  size_t pitch = 0;
  const uint16_t* srcs[3] = {host_depth, host_normals, host_radius};
  for (int i = 0; i < 3; ++i) {
    if (!srcs[i]) continue;
    BBA_CUDA(h, cudaMallocPitch(&kf.owned[i], &pitch, static_cast<size_t>(w) * 2, hh));
    BBA_CUDA(h, cudaMemcpy2DAsync(kf.owned[i], pitch, srcs[i], static_cast<size_t>(w) * 2, static_cast<size_t>(w) * 2, hh,
                                  cudaMemcpyHostToDevice, s));
  }
  kf.depth = static_cast<const uint16_t*>(kf.owned[0]); kf.depth_pitch = pitch;
  kf.normals = static_cast<const uint16_t*>(kf.owned[1]); kf.normals_pitch = pitch;
  kf.radius = static_cast<const uint16_t*>(kf.owned[2]); kf.radius_pitch = pitch;
  // the colour image: the luma plane is derived from it; the copy is kept for the colours of surfels created later
  uint8_t* tmp = nullptr;
  size_t tmp_pitch = 0;
  BBA_CUDA(h, cudaMallocPitch(reinterpret_cast<void**>(&tmp), &tmp_pitch, static_cast<size_t>(cw) * 4, ch));
  BBA_CUDA(h, cudaMemcpy2DAsync(tmp, tmp_pitch, host_color_rgba, static_cast<size_t>(cw) * 4, static_cast<size_t>(cw) * 4, ch,
                                cudaMemcpyHostToDevice, s));
  kf.owned_rgba = tmp;
  kf.rgba = tmp;
  kf.rgba_pitch = tmp_pitch;
  return AddKeyframeCommon(h, std::move(kf), tmp, tmp_pitch, global_T_frame, min_depth, max_depth, s, out_keyframe_id);
}

// ---- host-side building blocks, callable without a device (the CPU test-suite checks them against the oracle) ----
void bba_host_se3_exp(const float a[6], float out[7]) { PoseToArray(bba::Exp(a), out); }
void bba_host_se3_log(const float T[7], float out[6]) { bba::Log(PoseFromArray(T), out); }
void bba_host_se3_compose(const float A[7], const float B[7], float out[7]) { PoseToArray(bba::Compose(PoseFromArray(A), PoseFromArray(B)), out); }
void bba_host_se3_inverse(const float A[7], float out[7]) { PoseToArray(bba::Inverse(PoseFromArray(A)), out); }
int bba_host_pose_update_converged(const float x[6]) { return bba::IsScale1PoseEstimationConverged(x) ? 1 : 0; }
int bba_host_solve_ldlt(int n, const double* upper, const double* b, double* x) {
  if (!upper || !b || !x) return 0;
  if (n == 4) bba::SolveLDLT<4>(upper, b, x);
  else if (n == 5) bba::SolveLDLT<5>(upper, b, x);
  else if (n == 6) bba::SolveLDLT<6>(upper, b, x);
  else return 0;
  return 1;
}
int bba_host_frusta_intersect(const float depth_intrinsics[4], int width, int height, const float global_T_frame_a[7], float min_depth_a,
                              float max_depth_a, const float global_T_frame_b[7], float min_depth_b, float max_depth_b) {
  Frustum a, b;
  MakeFrustum(&a, depth_intrinsics, width, height, min_depth_a, max_depth_a, PoseFromArray(global_T_frame_a));
  MakeFrustum(&b, depth_intrinsics, width, height, min_depth_b, max_depth_b, PoseFromArray(global_T_frame_b));
  return FrustaIntersect(a, b) ? 1 : 0;
}

// Constant-motion model of the odometry front end.  The stored transforms and their inverses are two lists that are updated side
// by side (never re-derived from each other), like base_kf_tr_frame_ / frame_tr_base_kf_ of the reference; products associate
// left to right like its `a * b * c`.
namespace {
const float kIdentityPose[7] = {0.f, 0.f, 0.f, 1.f, 0.f, 0.f, 0.f};
void CopyPose(const float* src, float* dst) { for (int i = 0; i < 7; ++i) dst[i] = src[i]; }
}  // namespace

void bba_host_motion_model_clear(bba_motion_model* m, const float last_kf_frame_T_global[7], const float global_T_frame[7]) {   // bad_slam.cc:542-565
  if (!m) return;
  m->count = 1;
  if (!last_kf_frame_T_global || !global_T_frame) {
    CopyPose(kIdentityPose, m->base_kf_tr_frame[0]);
    CopyPose(kIdentityPose, m->frame_tr_base_kf[0]);
    return;
  }
  const Pose rel = bba::Compose(PoseFromArray(last_kf_frame_T_global), PoseFromArray(global_T_frame));
  PoseToArray(rel, m->base_kf_tr_frame[0]);
  PoseToArray(bba::Inverse(rel), m->frame_tr_base_kf[0]);
}

int bba_host_motion_model_predict(const bba_motion_model* m, int use_motion_model, float e1[7], float e2[7]) {   // bad_slam.cc:767-827
  if (!m || !e1 || !e2 || m->count < 1 || m->count > 3) return 0;
  const int n = m->count;
  const Pose last = PoseFromArray(m->base_kf_tr_frame[n - 1]);
  if (!use_motion_model) {
    PoseToArray(last, e1);
    PoseToArray(last, e2);
    return 1;
  }
  // the motion of the last step applied once more
  Pose first = last;
  if (n >= 2) first = bba::Compose(bba::Compose(last, PoseFromArray(m->frame_tr_base_kf[n - 2])), last);
  PoseToArray(first, e1);
  // the motion of the step before, applied twice to the frame before the last: an outlier in the last frame does not enter
  if (n >= 3) {
    const Pose step = bba::Compose(PoseFromArray(m->frame_tr_base_kf[n - 3]), PoseFromArray(m->base_kf_tr_frame[n - 2]));
    PoseToArray(bba::Compose(bba::Compose(PoseFromArray(m->base_kf_tr_frame[n - 2]), step), step), e2);
  } else {
    PoseToArray(first, e2);
  }
  return 1;
}

void bba_host_motion_model_push(bba_motion_model* m, const float estimate[7]) {   // bad_slam.cc:949-954
  if (!m || !estimate) return;
  if (m->count < 0 || m->count > 3) m->count = 0;
  if (m->count == 3) {
    for (int i = 0; i < 2; ++i) {
      CopyPose(m->base_kf_tr_frame[i + 1], m->base_kf_tr_frame[i]);
      CopyPose(m->frame_tr_base_kf[i + 1], m->frame_tr_base_kf[i]);
    }
    m->count = 2;
  }
  CopyPose(estimate, m->base_kf_tr_frame[m->count]);
  PoseToArray(bba::Inverse(PoseFromArray(estimate)), m->frame_tr_base_kf[m->count]);
  ++m->count;
}

void bba_host_motion_model_rebase(bba_motion_model* m) {   // bad_slam.cc:1057-1068
  if (!m) return;
  if (m->count < 0 || m->count > 3) m->count = 0;
  const int n = m->count;
  if (n == 0) {
    m->count = 1;
  } else {
    const Pose last = PoseFromArray(m->base_kf_tr_frame[n - 1]);
    const Pose last_inv = PoseFromArray(m->frame_tr_base_kf[n - 1]);
    for (int i = 0; i + 1 < n; ++i) {
      PoseToArray(bba::Compose(PoseFromArray(m->frame_tr_base_kf[i]), last), m->frame_tr_base_kf[i]);
      PoseToArray(bba::Compose(last_inv, PoseFromArray(m->base_kf_tr_frame[i])), m->base_kf_tr_frame[i]);
    }
  }
  CopyPose(kIdentityPose, m->base_kf_tr_frame[m->count - 1]);
  CopyPose(kIdentityPose, m->frame_tr_base_kf[m->count - 1]);
}

int bba_keyframe_count(bba_handle h) { return h ? static_cast<int>(h->keyframes.size()) : 0; }

#define CHECK_KF(h, id)                                                                   \
  if (!(h)) return BBA_ERR_INVALID_ARGUMENT;                                              \
  if ((id) < 0 || (id) >= static_cast<int>((h)->keyframes.size())) return Fail(h, BBA_ERR_INVALID_ARGUMENT, "bad keyframe id")

bba_status bba_set_keyframe_pose(bba_handle h, int id, const float p[7]) {
  CHECK_KF(h, id);
  h->keyframes[id].pose = PoseFromArray(p);
  return BBA_OK;
}
bba_status bba_get_keyframe_pose(bba_handle h, int id, float p[7]) {
  CHECK_KF(h, id);
  PoseToArray(h->keyframes[id].pose, p);
  return BBA_OK;
}
bba_status bba_set_keyframe_activation(bba_handle h, int id, int activation) {
  CHECK_KF(h, id);
  if (activation < 0 || activation > 2) return Fail(h, BBA_ERR_INVALID_ARGUMENT, "bad activation");
  h->keyframes[id].activation = activation;
  return BBA_OK;
}
bba_status bba_get_keyframe_activation(bba_handle h, int id, int* activation) {
  CHECK_KF(h, id);
  *activation = h->keyframes[id].activation;
  return BBA_OK;
}
bba_status bba_set_keyframe_states(bba_handle h, int count, const float* poses, const int* activation) {
  if (!h || count < 0 || count > static_cast<int>(h->keyframes.size())) return BBA_ERR_INVALID_ARGUMENT;
  for (int k = 0; k < count; ++k) {
    if (poses) h->keyframes[k].pose = PoseFromArray(poses + 7 * k);
    if (activation) {
      if (activation[k] < 0 || activation[k] > 2) return Fail(h, BBA_ERR_INVALID_ARGUMENT, "bad activation");
      h->keyframes[k].activation = activation[k];
    }
  }
  return BBA_OK;
}
bba_status bba_get_keyframe_states(bba_handle h, int count, float* poses, int* activation) {
  if (!h || count < 0 || count > static_cast<int>(h->keyframes.size())) return BBA_ERR_INVALID_ARGUMENT;
  for (int k = 0; k < count; ++k) {
    if (poses) PoseToArray(h->keyframes[k].pose, poses + 7 * k);
    if (activation) activation[k] = h->keyframes[k].activation;
  }
  return BBA_OK;
}
bba_status bba_get_covisibility(bba_handle h, int id, uint8_t* out_row) {
  CHECK_KF(h, id);
  std::memset(out_row, 0, h->keyframes.size());
  for (int o : h->keyframes[id].covis) out_row[o] = 1;
  return BBA_OK;
}

bba_status bba_set_intrinsics(bba_handle h, const float d[4], const float c[4], float a) {
  if (!h) return BBA_ERR_INVALID_ARGUMENT;
  if (d) std::memcpy(h->depth_K, d, sizeof(h->depth_K));
  if (c) std::memcpy(h->color_K, c, sizeof(h->color_K));
  h->depth_a = a;
  return BBA_OK;
}
bba_status bba_set_residual_types(bba_handle h, int use_depth_residuals, int use_descriptor_residuals) {
  if (!h) return BBA_ERR_INVALID_ARGUMENT;
  if (!use_depth_residuals && !use_descriptor_residuals)
    return Fail(h, BBA_ERR_INVALID_ARGUMENT, "bba_set_residual_types: at least one residual type must stay enabled");
  h->cfg.use_depth_residuals = use_depth_residuals != 0;
  h->cfg.use_descriptor_residuals = use_descriptor_residuals != 0;
  return BBA_OK;
}
bba_status bba_get_residual_types(bba_handle h, int* use_depth_residuals, int* use_descriptor_residuals) {
  if (!h) return BBA_ERR_INVALID_ARGUMENT;
  if (use_depth_residuals) *use_depth_residuals = h->cfg.use_depth_residuals;
  if (use_descriptor_residuals) *use_descriptor_residuals = h->cfg.use_descriptor_residuals;
  return BBA_OK;
}
bba_status bba_get_intrinsics(bba_handle h, float d[4], float c[4], float* a) {
  if (!h) return BBA_ERR_INVALID_ARGUMENT;
  if (d) std::memcpy(d, h->depth_K, sizeof(h->depth_K));
  if (c) std::memcpy(c, h->color_K, sizeof(h->color_K));
  if (a) *a = h->depth_a;
  return BBA_OK;
}
bba_status bba_cfactor_size(bba_handle h, int* w, int* hh) {
  if (!h) return BBA_ERR_INVALID_ARGUMENT;
  if (w) *w = h->cf_w;
  if (hh) *hh = h->cf_h;
  return BBA_OK;
}
bba_status bba_set_cfactor_host(bba_handle h, const float* host, void* stream) {
  if (!h || !host) return BBA_ERR_INVALID_ARGUMENT;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  BBA_CUDA(h, cudaMemcpyAsync(h->d_cfactor, host, sizeof(float) * h->cf_w * h->cf_h, cudaMemcpyHostToDevice, s));
  BBA_CUDA(h, cudaStreamSynchronize(s));
  return BBA_OK;
}
bba_status bba_get_cfactor_host(bba_handle h, float* host, void* stream) {
  if (!h || !host) return BBA_ERR_INVALID_ARGUMENT;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  BBA_CUDA(h, cudaMemcpyAsync(host, h->d_cfactor, sizeof(float) * h->cf_w * h->cf_h, cudaMemcpyDeviceToHost, s));
  BBA_CUDA(h, cudaStreamSynchronize(s));
  return BBA_OK;
}

bba_status bba_accumulate_pose_coeffs(bba_handle h, int id, const float pose[7], bba_pose_coeffs* out, void* stream) {
  CHECK_KF(h, id);
  if (!pose || !out) return BBA_ERR_INVALID_ARGUMENT;
  if (bba_status st = CheckSurfels(h)) return st;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int K = static_cast<int>(h->keyframes.size());
  if (bba_status st = WaitStaging(h)) return st;
  for (int k = 0; k < K; ++k) FillKfDevice(h->keyframes[k], h->keyframes[k].pose, h->h_kfs + k);
  FillKfDevice(h->keyframes[id], PoseFromArray(pose), h->h_kfs + id);
  h->h_work[0] = id;
  h->h_work[h->cfg.max_keyframes] = 1;
  BBA_CUDA(h, cudaMemcpyAsync(h->d_kfs, h->h_kfs, sizeof(KfDevice) * K, cudaMemcpyHostToDevice, s));
  BBA_CUDA(h, cudaMemcpyAsync(h->d_work[0], h->h_work, sizeof(int), cudaMemcpyHostToDevice, s));
  BBA_CUDA(h, cudaMemcpyAsync(h->d_count, h->h_work + h->cfg.max_keyframes, sizeof(int), cudaMemcpyHostToDevice, s));
  BBA_CUDA(h, cudaMemsetAsync(h->d_acc + static_cast<size_t>(id) * bba::kPoseAccSize, 0, sizeof(double) * bba::kPoseAccSize, s));
  BBA_CUDA(h, cudaMemsetAsync(h->d_stage_counts + 2 * id, 0, sizeof(unsigned long long) * 2, s));
  bba::PoseAccumulateArgs acc;
  acc.cam = MakeCamera(h);
  acc.surfels = h->surfels;
  acc.pitch = static_cast<uint32_t>(h->surfel_pitch_bytes / sizeof(float));
  acc.n = h->surfels_size;
  acc.kfs = h->d_kfs;
  acc.work_records = h->d_work_records;
  acc.frames = nullptr;
  acc.frames_pitch = 0;
  acc.acc = h->d_acc;
  acc.stage_counts = h->d_stage_counts;
  acc.queue = h->d_queue;
  BBA_CUDA(h, cudaMemsetAsync(h->d_queue, 0, sizeof(unsigned int), s));
  acc.work_list = h->d_work[0];
  acc.work_count = h->d_count;
  if (h->surfels_size > 0) {
    bba::LaunchPoseAccumulate(acc, h->sm_count, /*with_stats=*/true, 1, s);
    h->launches += 2;   // record packing + the kernel
  }
  BBA_CUDA(h, cudaGetLastError());
  BBA_CUDA(h, cudaMemcpyAsync(h->h_acc, h->d_acc + static_cast<size_t>(id) * bba::kPoseAccSize, sizeof(double) * bba::kPoseAccSize,
                              cudaMemcpyDeviceToHost, s));
  BBA_CUDA(h, cudaMemcpyAsync(h->h_acc + bba::kPoseAccSize, h->d_stage_counts + 2 * id, sizeof(unsigned long long) * 2,
                              cudaMemcpyDeviceToHost, s));
  BBA_CUDA(h, cudaMemsetAsync(h->d_acc + static_cast<size_t>(id) * bba::kPoseAccSize, 0, sizeof(double) * bba::kPoseAccSize, s));
  BBA_CUDA(h, cudaMemsetAsync(h->d_stage_counts + 2 * id, 0, sizeof(unsigned long long) * 2, s));
  BBA_CUDA(h, cudaStreamSynchronize(s));
  h->staging_pending = false;
  for (int i = 0; i < 21; ++i) out->H[i] = static_cast<float>(h->h_acc[i]);
  for (int i = 0; i < 6; ++i) out->b[i] = static_cast<float>(h->h_acc[21 + i]);
  unsigned long long sc[2];
  std::memcpy(sc, h->h_acc + bba::kPoseAccSize, sizeof(sc));
  out->n_pair = h->surfels_size;
  out->n_inimg = sc[0];
  out->n_depthok = sc[1];
  out->n_assoc = static_cast<uint64_t>(h->h_acc[27] + 0.5);
  out->n_photo = static_cast<uint64_t>(h->h_acc[28] + 0.5);
  out->cost_depth = h->h_acc[29];
  out->cost_desc1 = h->h_acc[30];
  out->cost_desc2 = h->h_acc[31];
  return BBA_OK;
}

bba_status bba_estimate_frame_pose(bba_handle h, int id, const float init[7], float out[7], int* iterations, int* converged,
                                   void* stream) {
  CHECK_KF(h, id);
  if (!init || !out) return BBA_ERR_INVALID_ARGUMENT;
  if (bba_status st = CheckSurfels(h)) return st;
  std::vector<int> ids(1, id);
  std::vector<Pose> poses(1, PoseFromArray(init));
  if (bba_status st = RunPoseStep(h, ids, poses, 30, static_cast<cudaStream_t>(stream))) return st;
  std::memcpy(out, h->h_pose_est + 7 * id, sizeof(float) * 7);
  if (iterations) *iterations = h->h_iterations[id];
  if (converged) *converged = h->h_converged[id];
  return BBA_OK;
}

bba_status bba_estimate_frame_pose_for_frame(bba_handle h, const uint16_t* device_depth, size_t depth_pitch,
                                             const uint16_t* device_normals, size_t normals_pitch,
                                             const uint8_t* device_color_rgba, size_t color_pitch, const float init[7], float out[7],
                                             int* iterations, int* converged, void* stream) {
  if (!h || !device_depth || !device_normals || !device_color_rgba || !init || !out) return BBA_ERR_INVALID_ARGUMENT;
  if (depth_pitch < static_cast<size_t>(h->cfg.depth_width) * 2 || normals_pitch < static_cast<size_t>(h->cfg.depth_width) * 2 ||
      color_pitch < static_cast<size_t>(h->cfg.color_width) * 4 || depth_pitch > 0xffffffffull || normals_pitch > 0xffffffffull)
    return Fail(h, BBA_ERR_INVALID_ARGUMENT, "frame buffer pitch too small");
  if (bba_status st = CheckSurfels(h)) return st;
  const int id = static_cast<int>(h->keyframes.size());
  if (id >= h->cfg.max_keyframes)
    return Fail(h, BBA_ERR_STATE, "bba_estimate_frame_pose_for_frame needs one free keyframe slot (max_keyframes reached)");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (bba_status st = MakeLumaTexture(h, device_color_rgba, color_pitch, &h->scratch_luma, &h->scratch_tex, s)) return st;
  // The frame rides through the pose step as a temporary entry behind the keyframes: it takes part in nothing else
  // (no co-visibility, no activation state) and is removed again before the call returns.
  Keyframe frame{};
  frame.depth = device_depth; frame.depth_pitch = depth_pitch;
  frame.normals = device_normals; frame.normals_pitch = normals_pitch;
  frame.tex = h->scratch_tex;
  frame.pose = PoseFromArray(init);
  frame.activation = BBA_KF_ACTIVE;
  h->keyframes.push_back(frame);
  std::vector<int> ids(1, id);
  std::vector<Pose> poses(1, PoseFromArray(init));
  const bba_status st = RunPoseStep(h, ids, poses, 30, s);
  h->keyframes.pop_back();
  if (id < static_cast<int>(h->kf_cost.size())) h->kf_cost[id] = 0.f;   // the slot's cost statistics belong to a future keyframe
  if (st) return st;
  std::memcpy(out, h->h_pose_est + 7 * id, sizeof(float) * 7);
  if (iterations) *iterations = h->h_iterations[id];
  if (converged) *converged = h->h_converged[id];
  return BBA_OK;
}

namespace {

// Fills the pyramids of both frames for the given options (stages 1-3 of odometry.cuh) and the level descriptors in h->odo.level.
bba_status BuildOdometryPyramids(bba_handle h, const bba_odometry_options& o, const Keyframe& base, const uint16_t* trk_depth, size_t trk_depth_pitch,
                                 const uint16_t* trk_normals, size_t trk_normals_pitch, cudaStream_t s) {
  namespace od = bba::odom;
  auto& st = h->odo;
  const int S = o.num_scales;
  od::BrightnessArgs br{};
  br.luma_tex[0] = base.tex; br.luma_tex[1] = h->scratch_tex;
  for (int f = 0; f < 2; ++f) { br.out[f] = st.gradmag[f]; br.out_pitch[f] = static_cast<uint32_t>(st.gradmag_pitch[f]); }
  br.w = h->cfg.color_width; br.h = h->cfg.color_height;
  br.use_gradmag = o.use_gradmag;
  od::LaunchBrightness(br, s);
  ++h->launches;

  // level images as seen by the kernels: level 0 normals are the keyframe's / the frame's own buffers
  od::Image img[2][od::kMaxScales];
  for (int f = 0; f < 2; ++f)
    for (int l = 0; l < S; ++l) img[f][l] = st.image[f][l];
  img[0][0].normals = const_cast<uint16_t*>(base.normals); img[0][0].normals_pitch = static_cast<uint32_t>(base.normals_pitch);
  img[1][0].normals = const_cast<uint16_t*>(trk_normals);  img[1][0].normals_pitch = static_cast<uint32_t>(trk_normals_pitch);

  const bba::CameraParams cam = MakeCamera(h);
  od::Level0Args l0{};
  l0.raw_depth[0] = base.depth; l0.raw_depth_pitch[0] = static_cast<uint32_t>(base.depth_pitch);
  l0.raw_depth[1] = trk_depth;  l0.raw_depth_pitch[1] = static_cast<uint32_t>(trk_depth_pitch);
  l0.raw_normals = trk_normals; l0.raw_normals_pitch = static_cast<uint32_t>(trk_normals_pitch);
  l0.gradmag_tex[0] = st.gradmag_tex[0]; l0.gradmag_tex[1] = st.gradmag_tex[1];
  l0.out[0] = img[0][0];
  l0.skip_level0 = o.use_pyramid_level_0 ? 0 : 1;
  l0.out[1] = l0.skip_level0 ? img[1][1] : img[1][0];
  l0.w = st.w[0]; l0.h = st.h[0];
  l0.out_w = l0.skip_level0 ? st.w[1] : st.w[0];
  l0.out_h = l0.skip_level0 ? st.h[1] : st.h[0];
  l0.d2c_fx = cam.d2c_fx; l0.d2c_fy = cam.d2c_fy; l0.d2c_cx = cam.d2c_cx; l0.d2c_cy = cam.d2c_cy;
  l0.cw = cam.cw; l0.ch = cam.ch;
  l0.a = cam.a; l0.raw_to_float = cam.raw_to_float; l0.cfactor = cam.cfactor; l0.cf_w = cam.cf_w; l0.cell = cam.cell;
  l0.downsample_color = h->cfg.depth_width == h->cfg.color_width;
  od::LaunchLevel0(l0, s);
  ++h->launches;

  for (int l = 1; l < S; ++l) {
    // pairwise_frame_tracking.cc:325-347: the tracked image from level 2 on (level 1 too when level 0 is in use), the base always
    od::DownsampleArgs d{};
    d.in[0] = img[0][l - 1]; d.out[0] = img[0][l];
    d.count = 1;
    if (l >= 2 || o.use_pyramid_level_0) {
      d.in[1] = img[1][l - 1]; d.out[1] = img[1][l];
      d.count = 2;
    }
    d.w = st.w[l]; d.h = st.h[l];
    d.in_w = st.w[l - 1]; d.in_h = st.h[l - 1];
    od::LaunchDownsample(d, s);
    ++h->launches;
  }
  for (int l = 0; l < S; ++l) {
    st.level[l].cam = MakeLevelCamera(h, l, st.w[l], st.h[l]);
    st.level[l].base = img[0][l];
    st.level[l].tracked = img[1][l];
  }
  st.last_num_scales = S;
  st.last_first_scale = o.use_pyramid_level_0 ? 0 : 1;
  BBA_CUDA(h, cudaGetLastError());
  return BBA_OK;
}

bba_status LaunchOdometryKernel(bba_handle h, int num_scales, int first_scale, int max_iterations, int use_gradmag, int test_different,
                                int debug_scale, const float init1[7], const float init2[7], cudaStream_t s) {
  namespace od = bba::odom;
  auto& st = h->odo;
  od::TrackArgs a{};
  for (int l = 0; l < num_scales; ++l) a.level[l] = st.level[l];
  a.num_scales = num_scales;
  a.first_scale = first_scale;
  a.max_iterations = max_iterations;
  a.use_depth = h->cfg.use_depth_residuals;
  a.use_desc = h->cfg.use_descriptor_residuals;
  a.use_gradmag = use_gradmag;
  a.test_different_initial_estimates = test_different;
  a.debug_scale = debug_scale;
  a.baseline_fx = h->cfg.baseline_fx;
  std::memcpy(a.init1, init1, sizeof(float) * 7);
  std::memcpy(a.init2, init2, sizeof(float) * 7);
  a.acc = st.d_acc;
  a.barrier = st.d_barrier;
  a.result = st.d_result;
  BBA_CUDA(h, cudaMemsetAsync(st.d_acc, 0, sizeof(double) * 96, s));
  BBA_CUDA(h, cudaMemsetAsync(st.d_barrier, 0, sizeof(unsigned int) * 2, s));
  BBA_CUDA(h, cudaMemsetAsync(st.d_result, 0, sizeof(od::TrackResult), s));
  od::LaunchTrack(a, h->sm_count, s);
  ++h->launches;
  BBA_CUDA(h, cudaGetLastError());
  BBA_CUDA(h, cudaMemcpyAsync(st.h_result, st.d_result, sizeof(od::TrackResult), cudaMemcpyDeviceToHost, s));
  BBA_CUDA(h, cudaStreamSynchronize(s));
  if (st.h_result->barrier_timeout) return Fail(h, BBA_ERR_CUDA, "odometry kernel: grid barrier timed out");
  return BBA_OK;
}

}  // namespace

bba_status bba_track_frame_pairwise(bba_handle h, const bba_odometry_options* o, int base_keyframe_id,
                                    const uint16_t* device_depth, size_t depth_pitch, const uint16_t* device_normals, size_t normals_pitch,
                                    const uint8_t* device_color_rgba, size_t color_pitch, const float init1[7], const float init2[7],
                                    float out[7], bba_odometry_result* result, void* stream) {
  if (!h || !o || !device_depth || !device_normals || !device_color_rgba || !init1 || !out) return h ? Fail(h, BBA_ERR_INVALID_ARGUMENT, "bba_track_frame_pairwise: null argument") : BBA_ERR_INVALID_ARGUMENT;
  if (base_keyframe_id < 0 || base_keyframe_id >= static_cast<int>(h->keyframes.size()))
    return Fail(h, BBA_ERR_INVALID_ARGUMENT, "bba_track_frame_pairwise: no such keyframe");
  if (o->num_scales < 1 || o->num_scales > bba::odom::kMaxScales || (!o->use_pyramid_level_0 && o->num_scales < 2))
    return Fail(h, BBA_ERR_INVALID_ARGUMENT, "bba_track_frame_pairwise: num_scales must be 1..8 (>= 2 without pyramid level 0)");
  if (depth_pitch < static_cast<size_t>(h->cfg.depth_width) * 2 || normals_pitch < static_cast<size_t>(h->cfg.depth_width) * 2 ||
      color_pitch < static_cast<size_t>(h->cfg.color_width) * 4 || depth_pitch > 0xffffffffull || normals_pitch > 0xffffffffull ||
      ((depth_pitch | normals_pitch) & 1u))
    return Fail(h, BBA_ERR_INVALID_ARGUMENT, "bba_track_frame_pairwise: bad frame buffer pitch");
  // pairwise_frame_tracking.cc:300-306 (LOG(FATAL) in the reference)
  if (!o->use_pyramid_level_0 && h->cfg.depth_width != h->cfg.color_width && h->cfg.depth_width != 2 * h->cfg.color_width)
    return Fail(h, BBA_ERR_UNSUPPORTED, "The chosen depth / color pyramid level combination is not supported here.");
  if (o->test_different_initial_estimates && !init2)
    return Fail(h, BBA_ERR_INVALID_ARGUMENT, "bba_track_frame_pairwise: test_different_initial_estimates needs the second estimate");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const uint64_t launches_before = h->launches;
  if (bba_status st = EnsureOdometry(h, o->num_scales)) return st;
  if (bba_status st = MakeLumaTexture(h, device_color_rgba, color_pitch, &h->scratch_luma, &h->scratch_tex, s)) return st;
  const Keyframe& base = h->keyframes[base_keyframe_id];
  if (bba_status st = BuildOdometryPyramids(h, *o, base, device_depth, depth_pitch, device_normals, normals_pitch, s)) return st;
  const int max_it = o->max_iterations_per_scale > 0 ? o->max_iterations_per_scale : 30;
  if (bba_status st = LaunchOdometryKernel(h, o->num_scales, o->use_pyramid_level_0 ? 0 : 1, max_it, o->use_gradmag ? 1 : 0,
                                           o->test_different_initial_estimates ? 1 : 0, -1, init1, init2 ? init2 : init1, s))
    return st;
  const bba::odom::TrackResult& r = *h->odo.h_result;
  std::memcpy(out, r.base_T_frame, sizeof(float) * 7);
  if (result) {
    for (int i = 0; i < 8; ++i) {
      result->iterations[i] = r.iterations[i];
      result->chose_initial[i] = i < o->num_scales ? r.chose_initial[i] : -1;
    }
    result->residual_count = r.residual_count;
    result->residual_sum = r.residual_sum;
    result->passes = r.passes;
    result->kernel_launches = static_cast<uint32_t>(h->launches - launches_before);
  }
  return BBA_OK;
}

bba_status bba_odometry_get_level(bba_handle h, int which, int scale, float* host_depth, uint16_t* host_normals, uint8_t* host_color,
                                  int* width, int* height, void* stream) {
  if (!h) return BBA_ERR_INVALID_ARGUMENT;
  auto& st = h->odo;
  if (which < 0 || which > 1 || scale < 0 || scale >= st.last_num_scales || (which == 1 && scale < st.last_first_scale))
    return Fail(h, BBA_ERR_STATE, "bba_odometry_get_level: this level was not built by the last bba_track_frame_pairwise call");
  const bba::odom::Image& im = which ? st.level[scale].tracked : st.level[scale].base;
  const int w = st.w[scale], ht = st.h[scale];
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (host_depth) BBA_CUDA(h, cudaMemcpy2DAsync(host_depth, sizeof(float) * w, im.depth, sizeof(float) * im.depth_pitch, sizeof(float) * w, ht, cudaMemcpyDeviceToHost, s));
  if (host_normals) BBA_CUDA(h, cudaMemcpy2DAsync(host_normals, sizeof(uint16_t) * w, im.normals, im.normals_pitch, sizeof(uint16_t) * w, ht, cudaMemcpyDeviceToHost, s));
  if (host_color) BBA_CUDA(h, cudaMemcpy2DAsync(host_color, w, im.color, im.color_pitch, w, ht, cudaMemcpyDeviceToHost, s));
  BBA_CUDA(h, cudaStreamSynchronize(s));
  if (width) *width = w;
  if (height) *height = ht;
  return BBA_OK;
}

bba_status bba_odometry_debug_coeffs(bba_handle h, int scale, int use_gradmag, const float pose_a[7], const float pose_b[7], float H[21],
                                     float b[6], uint32_t* residual_count, float* residual_sum, uint32_t counts[2], float costs[2], void* stream) {
  if (!h || !pose_a) return BBA_ERR_INVALID_ARGUMENT;
  auto& st = h->odo;
  if (scale < st.last_first_scale || scale >= st.last_num_scales)
    return Fail(h, BBA_ERR_STATE, "bba_odometry_debug_coeffs: this level was not built by the last bba_track_frame_pairwise call");
  if (bba_status s2 = LaunchOdometryKernel(h, st.last_num_scales, st.last_first_scale, 1, use_gradmag ? 1 : 0, 0, scale, pose_a,
                                           pose_b ? pose_b : pose_a, static_cast<cudaStream_t>(stream)))
    return s2;
  const double* d = st.h_result->debug;
  if (H) for (int i = 0; i < 21; ++i) H[i] = static_cast<float>(d[i]);
  if (b) for (int i = 0; i < 6; ++i) b[i] = static_cast<float>(d[21 + i]);
  if (residual_count) *residual_count = static_cast<uint32_t>(d[27] + 0.5);
  if (residual_sum) *residual_sum = static_cast<float>(d[28]);
  if (counts) { counts[0] = static_cast<uint32_t>(d[32] + 0.5); counts[1] = static_cast<uint32_t>(d[34] + 0.5); }
  if (costs) { costs[0] = static_cast<float>(d[33]); costs[1] = static_cast<float>(d[35]); }
  return BBA_OK;
}

bba_status bba_preprocess_frame(bba_handle h, const bba_preprocess_options* o,
                                const uint16_t* device_raw_depth, size_t raw_depth_pitch,
                                const uint8_t* device_rgb, size_t rgb_pitch,
                                uint16_t* device_depth, size_t depth_pitch,
                                uint16_t* device_normals, size_t normals_pitch,
                                uint16_t* device_radius, size_t radius_pitch,
                                uint8_t* device_color_rgba, size_t color_pitch,
                                float* min_depth, float* max_depth, void* stream) {
  if (!h || !o || !device_raw_depth || !device_depth || !device_normals || !device_radius) return h ? Fail(h, BBA_ERR_INVALID_ARGUMENT, "bba_preprocess_frame: null argument") : BBA_ERR_INVALID_ARGUMENT;
  if ((device_rgb == nullptr) != (device_color_rgba == nullptr))
    return Fail(h, BBA_ERR_INVALID_ARGUMENT, "bba_preprocess_frame: rgb input and rgba output go together");
  if ((raw_depth_pitch | depth_pitch | normals_pitch | radius_pitch) & 1u)
    return Fail(h, BBA_ERR_INVALID_ARGUMENT, "bba_preprocess_frame: u16 image pitches must be even");
  if (device_color_rgba && ((color_pitch & 3u) || (reinterpret_cast<uintptr_t>(device_color_rgba) & 3u)))
    return Fail(h, BBA_ERR_INVALID_ARGUMENT, "bba_preprocess_frame: the rgba image must be 4-byte aligned");
  if (device_depth == device_raw_depth)
    return Fail(h, BBA_ERR_INVALID_ARGUMENT, "bba_preprocess_frame: in-place filtering is not possible (tiles read their neighbours' raw depth)");
  // BilateralFilteringAndDepthCutoffCUDA (cuda_depth_processing.cu:100-128)
  const int radius = static_cast<int>(o->bilateral_filter_radius_factor * o->bilateral_filter_sigma_xy + 0.5f);
  if (radius < 0 || radius > bba::pre::kMaxFilterRadius)
    return Fail(h, BBA_ERR_INVALID_ARGUMENT, "bba_preprocess_frame: bilateral filter radius outside [0, 16]");
  if (!(o->bilateral_filter_sigma_xy > 0.f) || !(o->bilateral_filter_sigma_inv_depth > 0.f) || !(o->max_depth > 0.f))
    return Fail(h, BBA_ERR_INVALID_ARGUMENT, "bba_preprocess_frame: sigma_xy, sigma_inv_depth and max_depth must be positive");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (!h->d_min_max) {
    BBA_CUDA(h, cudaMalloc(&h->d_min_max, 2 * sizeof(float)));
    BBA_CUDA(h, cudaMallocHost(&h->h_min_max, 2 * sizeof(float)));
  }
  const bba::CameraParams cam = MakeCamera(h);
  bba::pre::FrameArgs f{};
  f.w = cam.w; f.h = cam.h;
  f.fx_inv = cam.fx_inv; f.fy_inv = cam.fy_inv; f.cx_inv = cam.cx_inv; f.cy_inv = cam.cy_inv;
  f.raw_to_float = cam.raw_to_float; f.a = cam.a;
  f.cell = cam.cell; f.cf_w = cam.cf_w; f.cfactor = cam.cfactor;
  f.denom_xy = 2.0f * o->bilateral_filter_sigma_xy * o->bilateral_filter_sigma_xy;
  f.denom_value = 2.0f * o->bilateral_filter_sigma_inv_depth * o->bilateral_filter_sigma_inv_depth;
  f.radius = radius;
  f.radius_squared = radius * radius;
  const float max_raw = o->max_depth / cam.raw_to_float;   // bad_slam.cc:703 (float -> u16 at the call)
  f.max_depth = max_raw >= 65535.f ? static_cast<uint16_t>(65535) : static_cast<uint16_t>(max_raw);
  f.raw_depth = device_raw_depth; f.raw_pitch = static_cast<uint32_t>(raw_depth_pitch);
  f.out_depth = device_depth; f.out_depth_pitch = static_cast<uint32_t>(depth_pitch);
  f.out_normals = device_normals; f.out_normals_pitch = static_cast<uint32_t>(normals_pitch);
  f.out_radius = device_radius; f.out_radius_pitch = static_cast<uint32_t>(radius_pitch);
  f.min_max = h->d_min_max;
  f.cw = cam.cw; f.ch = cam.ch;
  f.rgb = device_rgb; f.rgb_pitch = static_cast<uint32_t>(rgb_pitch);
  f.rgba = device_color_rgba; f.rgba_pitch = static_cast<uint32_t>(color_pitch);
  f.tiles_x = (f.w + bba::pre::kTile - 1) / bba::pre::kTile;
  f.tiles_y = (f.h + bba::pre::kTile - 1) / bba::pre::kTile;
  h->launches += bba::LaunchPreprocessFrame(f, s);
  BBA_CUDA(h, cudaGetLastError());
  if (min_depth || max_depth) {   // ComputeMinMaxDepthCUDA returns host values and synchronises (cuda_depth_processing.cu:452-463)
    BBA_CUDA(h, cudaMemcpyAsync(h->h_min_max, h->d_min_max, 2 * sizeof(float), cudaMemcpyDeviceToHost, s));
    BBA_CUDA(h, cudaStreamSynchronize(s));
    if (min_depth) *min_depth = h->h_min_max[0];
    if (max_depth) *max_depth = h->h_min_max[1];
  }
  return BBA_OK;
}

bba_status bba_update_surfel_activation(bba_handle h, void* stream) {
  if (!h) return BBA_ERR_INVALID_ARGUMENT;
  if (bba_status st = CheckSurfels(h)) return st;
  if (h->surfels_size == 0) return BBA_OK;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (bba_status st = UploadKeyframes(h, s)) return st;
  bba::GeometryArgs g;
  if (bba_status st = BuildGeometryArgs(h, &g, s)) return st;
  if (bba_status st = CheckCollective(h)) return st;
  bba::LaunchActivationAndNormals(g, h->sm_count, true, false, s);
  ++h->launches;
  BBA_CUDA(h, cudaGetLastError());
  if (bba_status st = ExchangeGeometry(h, s)) return st;
  return MarkStaging(h, s);
}

bba_status bba_optimize_geometry_iteration(bba_handle h, void* stream) {
  if (!h) return BBA_ERR_INVALID_ARGUMENT;
  if (bba_status st = CheckSurfels(h)) return st;
  if (h->surfels_size == 0) return BBA_OK;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (bba_status st = UploadKeyframes(h, s)) return st;
  bba::GeometryArgs g;
  if (bba_status st = BuildGeometryArgs(h, &g, s)) return st;
  if (bba_status st = CheckCollective(h)) return st;
  bba::LaunchActivationAndNormals(g, h->sm_count, false, true, s);
  bba::LaunchPositionAndDescriptor(g, h->sm_count, s);
  h->launches += 2;
  BBA_CUDA(h, cudaGetLastError());
  if (bba_status st = ExchangeGeometry(h, s)) return st;
  return MarkStaging(h, s);
}

bba_status bba_optimize_intrinsics(bba_handle h, int optimize_depth, int optimize_color, void* stream) {
  if (!h) return BBA_ERR_INVALID_ARGUMENT;
  if (!optimize_depth && !optimize_color) return Fail(h, BBA_ERR_INVALID_ARGUMENT, "nothing to optimise");   // kernel_opt_intrinsics.cc:54
  if (bba_status st = CheckSurfels(h)) return st;
  if (bba_status st = CheckCollective(h)) return st;
  return OptimizeIntrinsics(h, optimize_depth != 0, optimize_color != 0, static_cast<cudaStream_t>(stream));
}

bba_status bba_bundle_adjust(bba_handle h, const bba_ba_options* o, bba_ba_result* res, void* stream) {
  if (!h || !o || !res) return BBA_ERR_INVALID_ARGUMENT;
  std::memset(res, 0, sizeof(*res));
  if (bba_status st = CheckSurfels(h)) return st;
  // (do_surfel_updates with more than one rank: creation / merging / compaction run REPLICATED -- they are deterministic and
  // every rank holds the whole surfel buffer -- while the geometry and pose steps stay sharded; see PeerFence)
  if (o->use_pcg) return BundleAdjustPCG(h, o, res, static_cast<cudaStream_t>(stream));   // direct_ba.cc:436-457
  // direct_ba.cc:427-434
  const bool opt_depth_intr = o->optimize_depth_intrinsics && h->cfg.use_depth_residuals;
  const bool opt_color_intr = o->optimize_color_intrinsics && h->cfg.use_descriptor_residuals;
  if (bba_status st = CheckCollective(h)) return st;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int K = static_cast<int>(h->keyframes.size());
  const uint64_t launches_before = h->launches;
  const auto t_start = std::chrono::steady_clock::now();

  const int fixed_ba_iteration_count = h->ba_iteration_count;
  if (!o->increase_ba_iteration_count && h->ba_iteration_count != h->last_ba_iteration_count) {   // :313-319
    h->last_ba_iteration_count = h->ba_iteration_count;
    uint32_t deleted = 0;
    if (bba_status st = PerformEndTasks(h, s, &deleted, o->do_surfel_updates != 0)) return st;
    res->surfels_deleted += deleted;
  }
  std::vector<int> keyframes_with_new_surfels;

  const bool fixed_window = o->active_keyframe_window_start > 0 || o->active_keyframe_window_end > 0;   // :330-331
  const bool whole_window = !(o->active_keyframe_window_start != 0 || o->active_keyframe_window_end != K - 1);

  BBA_CUDA(h, cudaMemsetAsync(h->active, 0, h->surfels_size, s));   // :338

  for (int iteration = 0; iteration < o->max_iterations; ++iteration) {
    if (o->progress_function && !o->progress_function(o->progress_user, iteration)) break;
    ++res->iterations_done;
    if (fixed_window) {   // :354-372
      for (int k = 0; k < K; ++k)
        h->keyframes[k].activation =
            (k >= o->active_keyframe_window_start && k <= o->active_keyframe_window_end) ? BBA_KF_ACTIVE : BBA_KF_INACTIVE;
      DetermineCovisibleActiveKeyframes(h);
    }

    BBA_TRACE("iteration start");
    // --- surfel creation (:399-430): keyframes that became active for the first time within this BA iteration block
    keyframes_with_new_surfels.clear();
    const uint32_t old_surfels_size = h->surfels_size;
    if (o->optimize_geometry && o->do_surfel_updates) {
      for (int k = 0; k < K; ++k) {
        Keyframe& kf = h->keyframes[k];
        if (kf.activation == BBA_KF_ACTIVE && kf.last_active_in_ba_iteration != fixed_ba_iteration_count) {
          kf.last_active_in_ba_iteration = fixed_ba_iteration_count;
          keyframes_with_new_surfels.push_back(k);
        } else if (kf.activation == BBA_KF_COVISIBLE_ACTIVE && kf.last_covis_in_ba_iteration != fixed_ba_iteration_count) {
          kf.last_covis_in_ba_iteration = fixed_ba_iteration_count;
        }
      }
      for (int k : keyframes_with_new_surfels) {
        uint32_t created = 0;
        if (bba_status st = CreateSurfelsForKeyframe(h, k, /*filter_new_surfels=*/true, s, &created)) return st;
        res->surfels_created += created;
      }
    }

    BBA_TRACE("creation done");
    if (bba_status st = UploadKeyframes(h, s)) return st;
    BBA_TRACE("keyframes uploaded");
    bba::GeometryArgs g;
    if (bba_status st = BuildGeometryArgs(h, &g, s)) return st;

    BBA_TRACE("after creation + upload");
    // --- surfel activation (:432-456) fused with the normal update of the geometry step (:466-485)
    BBA_CUDA(h, cudaEventRecord(h->ev[0], s));
    const bool has_new = o->optimize_geometry && h->surfels_size > old_surfels_size;
    if (has_new)   // new surfels are active (:435-441); only the old ones are re-evaluated below
      BBA_CUDA(h, cudaMemsetAsync(h->active + old_surfels_size, bba::kSurfelActiveFlag, h->surfels_size - old_surfels_size, s));
    if (!whole_window) BBA_CUDA(h, cudaMemsetAsync(h->active, bba::kSurfelActiveFlag, old_surfels_size, s));
    if (h->surfels_size > 0) {
      if (whole_window && has_new) {
        bba::GeometryArgs g_old = g, g_new = g;   // (begin / end are LOCAL indices of this rank's shard)
        g_old.end = LocalCountBelow(old_surfels_size, h->cfg.rank, h->cfg.world_size);
        g_new.begin = g_old.end;
        bba::LaunchActivationAndNormals(g_old, h->sm_count, true, true, s);
        bba::LaunchActivationAndNormals(g_new, h->sm_count, false, true, s);
        h->launches += 2;
      } else if (whole_window) {
        bba::LaunchActivationAndNormals(g, h->sm_count, true, o->optimize_geometry != 0, s);
        ++h->launches;
      } else if (o->optimize_geometry) {
        bba::LaunchActivationAndNormals(g, h->sm_count, false, true, s);
        ++h->launches;
      }
    }
    BBA_CUDA(h, cudaEventRecord(h->ev[1], s));
    if (o->optimize_geometry && h->surfels_size > 0) {
      bba::LaunchPositionAndDescriptor(g, h->sm_count, s);
      ++h->launches;
    }
    BBA_CUDA(h, cudaGetLastError());
    if (bba_status st = ExchangeGeometry(h, s)) return st;   // multi-GPU: all-gather of the updated surfel shards
    BBA_CUDA(h, cudaEventRecord(h->ev[2], s));
    if (bba_status st = MarkStaging(h, s)) return st;

    BBA_TRACE("after geometry");
    // --- surfel merge + compaction (:489-541) for the keyframes that received new surfels
    if (o->do_surfel_updates && !keyframes_with_new_surfels.empty()) {
      uint32_t merged = 0;
      for (int k : keyframes_with_new_surfels) {
        uint32_t d = 0;
        if (bba_status st = MergeSurfelsForKeyframe(h, k, s, &d)) return st;
        merged += d;
      }
      res->surfels_merged += merged;
      if (bba_status st = CompactSurfels(h, merged, /*with_active=*/true, s)) return st;
    }

    BBA_TRACE("before pose step");
    // --- pose optimisation (:543-577): all non-inactive keyframes at once
    int num_converged = 0;
    if (o->optimize_poses) {
      std::vector<int> ids;
      std::vector<Pose> init;
      for (int k = 0; k < K; ++k) {
        if (h->keyframes[k].activation == BBA_KF_INACTIVE) {
          ++num_converged;
          continue;
        }
        ids.push_back(k);
        init.push_back(h->keyframes[k].pose);
      }
      if (bba_status st = RunPoseStep(h, ids, init, 30, s)) return st;
      res->depth_residual_count = 0;
      res->descriptor_residual_count = 0;
      res->cost = 0;
      for (int k : ids) {
        Keyframe& kf = h->keyframes[k];
        const Pose est = PoseFromArray(h->h_pose_est + 7 * k);
        float lg[6];
        bba::Log(bba::Compose(bba::Inverse(kf.pose), est), lg);   // :562-563
        const bool moved = !bba::IsScale1PoseEstimationConverged(lg);
        kf.pose = est;
        if (moved) {
          kf.activation = BBA_KF_ACTIVE;
        } else {
          kf.activation = BBA_KF_INACTIVE;
          ++num_converged;
        }
        res->pose_iterations_total += h->h_iterations[k];
        const double* fs = h->h_first_stats + 8 * k;
        res->depth_residual_count += static_cast<uint64_t>(fs[0] + 0.5);
        res->descriptor_residual_count += 2 * static_cast<uint64_t>(fs[1] + 0.5);
        res->cost += fs[2] + fs[3];
      }
    } else {
      BBA_CUDA(h, cudaStreamSynchronize(s));
    }
    BBA_CUDA(h, cudaEventRecord(h->ev[3], s));
    // --- intrinsics optimisation (:584-624)
    if (opt_depth_intr || opt_color_intr) {
      if (bba_status st = OptimizeIntrinsics(h, opt_depth_intr, opt_color_intr, s)) return st;
      BBA_CUDA(h, cudaEventRecord(h->ev[4], s));
      BBA_CUDA(h, cudaEventSynchronize(h->ev[4]));
      cudaEventElapsedTime(&res->ms_intrinsics_optimization, h->ev[3], h->ev[4]);
    }
    BBA_CUDA(h, cudaEventSynchronize(h->ev[3]));
    cudaEventElapsedTime(&res->ms_surfel_activation, h->ev[0], h->ev[1]);
    cudaEventElapsedTime(&res->ms_geometry_optimization, h->ev[1], h->ev[2]);
    cudaEventElapsedTime(&res->ms_pose_optimization, h->ev[2], h->ev[3]);
    if (h->profiling) {
      h->profile.activation_normals_ms += res->ms_surfel_activation;
      h->profile.position_descriptor_ms += res->ms_geometry_optimization;
      h->profile.geometry_launches += (o->optimize_geometry ? 2 : 1);
    }

    // --- convergence (:693-701)
    if (iteration >= o->min_iterations - 1 && (num_converged == K || !o->optimize_poses)) {
      res->converged = 1;
      break;
    }
    if (o->time_limit_seconds > 0) {   // :704-709
      const double el = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_start).count();
      if (el > o->time_limit_seconds) break;
    }
    DetermineCovisibleActiveKeyframes(h);   // :711-717
  }
  BBA_TRACE("iterations done");
  if (o->increase_ba_iteration_count) {   // :725-735
    uint32_t deleted = 0;
    if (bba_status st = PerformEndTasks(h, s, &deleted, o->do_surfel_updates != 0)) return st;
    res->surfels_deleted += deleted;
    ++h->ba_iteration_count;
  }
  res->surfels_size = h->surfels_size;
  res->kernel_launches = h->launches - launches_before;
  return BBA_OK;
}

bba_status bba_perform_end_tasks(bba_handle h, int do_surfel_updates, uint32_t* deleted, uint32_t* surfels_size, void* stream) {
  if (!h) return BBA_ERR_INVALID_ARGUMENT;
  if (bba_status st = CheckSurfels(h)) return st;
  uint32_t d = 0;
  if (bba_status st = PerformEndTasks(h, static_cast<cudaStream_t>(stream), &d, do_surfel_updates != 0)) return st;
  if (deleted) *deleted = d;
  if (surfels_size) *surfels_size = h->surfels_size;
  return BBA_OK;
}

uint32_t bba_surfels_size(bba_handle h) { return h ? h->surfels_size : 0; }

bba_status bba_get_ba_iteration_counts(bba_handle h, int* ba_iteration_count, int* last_ba_iteration_count) {
  if (!h) return BBA_ERR_INVALID_ARGUMENT;
  if (ba_iteration_count) *ba_iteration_count = h->ba_iteration_count;
  if (last_ba_iteration_count) *last_ba_iteration_count = h->last_ba_iteration_count;
  return BBA_OK;
}
bba_status bba_set_ba_iteration_counts(bba_handle h, int ba_iteration_count, int last_ba_iteration_count) {
  if (!h) return BBA_ERR_INVALID_ARGUMENT;
  h->ba_iteration_count = ba_iteration_count;
  h->last_ba_iteration_count = last_ba_iteration_count;
  return BBA_OK;
}

bba_status bba_create_surfels_for_keyframe(bba_handle h, int id, int filter_new_surfels, uint32_t* created, void* stream) {
  CHECK_KF(h, id);
  if (bba_status st = CheckSurfels(h)) return st;
  uint32_t c = 0;
  if (bba_status st = CreateSurfelsForKeyframe(h, id, filter_new_surfels != 0, static_cast<cudaStream_t>(stream), &c)) return st;
  if (created) *created = c;
  return BBA_OK;
}

bba_status bba_merge_surfels_for_keyframe(bba_handle h, int id, uint32_t* deleted, void* stream) {
  CHECK_KF(h, id);
  if (bba_status st = CheckSurfels(h)) return st;
  uint32_t d = 0;
  if (bba_status st = MergeSurfelsForKeyframe(h, id, static_cast<cudaStream_t>(stream), &d)) return st;
  if (deleted) *deleted = d;
  return BBA_OK;
}

bba_status bba_compact_surfels(bba_handle h, uint32_t free_count, int with_active_flags, uint32_t* surfels_size, void* stream) {
  if (!h) return BBA_ERR_INVALID_ARGUMENT;
  if (bba_status st = CheckSurfels(h)) return st;
  if (free_count > h->surfels_size) return Fail(h, BBA_ERR_INVALID_ARGUMENT, "free_count exceeds surfels_size");
  if (bba_status st = CompactSurfels(h, free_count, with_active_flags != 0, static_cast<cudaStream_t>(stream))) return st;
  if (surfels_size) *surfels_size = h->surfels_size;
  return BBA_OK;
}

bba_status bba_pcg_debug(bba_handle h, const bba_ba_options* o, uint32_t* unknown_count, float* out_r, float* out_M, float* out_p,
                         float* out_g, double out_scalars[2], void* stream) {
  if (!h || !o || !unknown_count) return BBA_ERR_INVALID_ARGUMENT;
  if (bba_status st = CheckSurfels(h)) return st;
  const int K = static_cast<int>(h->keyframes.size());
  if (K == 0) return Fail(h, BBA_ERR_STATE, "no keyframes");
  if (o->pcg_gauge_keyframe < 0 || o->pcg_gauge_keyframe >= K) return Fail(h, BBA_ERR_INVALID_ARGUMENT, "pcg_gauge_keyframe out of range");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  PcgLayout L;
  if (bba_status st = MakePcgLayout(h, o, &L)) return st;
  *unknown_count = L.unknown_count;
  if (!out_r || L.unknown_count == 0) return BBA_OK;
  const uint32_t U = L.unknown_count;
  if (bba_status st = UploadKeyframes(h, s)) return st;
  BBA_CUDA(h, cudaMemsetAsync(h->d_pcg[0], 0, sizeof(float) * U, s));
  BBA_CUDA(h, cudaMemsetAsync(h->d_pcg[1], 0, sizeof(float) * U, s));
  BBA_CUDA(h, cudaMemsetAsync(h->d_pcg_scalars, 0, sizeof(double) * 4, s));
  const bba::PcgArgs a = MakePcgArgs(h, L, o->pcg_gauge_keyframe);
  bba::LaunchPcgAccumulate(a, h->sm_count, true, s);
  BBA_CUDA(h, cudaMemcpyAsync(out_r, h->d_pcg[0], sizeof(float) * U, cudaMemcpyDeviceToHost, s));
  BBA_CUDA(h, cudaMemcpyAsync(out_M, h->d_pcg[1], sizeof(float) * U, cudaMemcpyDeviceToHost, s));
  bba::LaunchPcgInit2(U, L.a_index, h->depth_a, K, h->d_pcg[0], h->d_pcg[1], h->d_pcg[2], h->d_pcg[3], h->d_pcg[4], h->d_pcg_scalars, 0,
                      h->sm_count, s);
  BBA_CUDA(h, cudaMemcpyAsync(out_p, h->d_pcg[4], sizeof(float) * U, cudaMemcpyDeviceToHost, s));
  bba::LaunchPcgAccumulate(a, h->sm_count, false, s);
  h->launches += 3;
  BBA_CUDA(h, cudaGetLastError());
  BBA_CUDA(h, cudaMemcpyAsync(out_g, h->d_pcg[3], sizeof(float) * U, cudaMemcpyDeviceToHost, s));
  BBA_CUDA(h, cudaMemcpyAsync(h->h_pcg_scalars, h->d_pcg_scalars, sizeof(double) * 4, cudaMemcpyDeviceToHost, s));
  BBA_CUDA(h, cudaStreamSynchronize(s));
  out_scalars[0] = h->h_pcg_scalars[0];
  out_scalars[1] = h->h_pcg_scalars[1];
  return MarkStaging(h, s);
}

// ---- NVLink peer replicas ------------------------------------------------------------------------------------------------
namespace {
bba_status AllocationBase(bba_handle h, const void* ptr, void** base) {
  typedef int (*GetRangeFn)(unsigned long long*, size_t*, unsigned long long);
  static GetRangeFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    BBA_CUDA(h, cudaGetDriverEntryPoint("cuMemGetAddressRange", &p, cudaEnableDefault, &q));
    if (!p) return Fail(h, BBA_ERR_CUDA, "cuMemGetAddressRange is not available");
    fn = reinterpret_cast<GetRangeFn>(p);
  }
  unsigned long long b = 0;
  size_t size = 0;
  if (fn(&b, &size, reinterpret_cast<unsigned long long>(ptr)) != 0) return Fail(h, BBA_ERR_CUDA, "cuMemGetAddressRange failed");
  *base = reinterpret_cast<void*>(b);
  return BBA_OK;
}
}  // namespace

bba_status bba_peer_export(bba_handle h, bba_peer_handle* out) {
  if (!h || !out) return BBA_ERR_INVALID_ARGUMENT;
  if (bba_status st = CheckSurfels(h)) return st;
  std::memset(out, 0, sizeof(*out));
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "bba_peer_handle layout");
  void* base = nullptr;
  cudaIpcMemHandle_t ipc;
  if (bba_status st = AllocationBase(h, h->surfels, &base)) return st;
  BBA_CUDA(h, cudaIpcGetMemHandle(&ipc, base));
  std::memcpy(out->surfels_ipc, &ipc, 64);
  out->surfels_offset = static_cast<uint64_t>(reinterpret_cast<const char*>(h->surfels) - static_cast<const char*>(base));
  if (bba_status st = AllocationBase(h, h->active, &base)) return st;
  BBA_CUDA(h, cudaIpcGetMemHandle(&ipc, base));
  std::memcpy(out->active_ipc, &ipc, 64);
  out->active_offset = static_cast<uint64_t>(reinterpret_cast<const char*>(h->active) - static_cast<const char*>(base));
  out->pitch_bytes = h->surfel_pitch_bytes;
  out->surfels_size = h->surfels_size;
  out->rank = h->cfg.rank;
  return BBA_OK;
}

bba_status bba_peer_import(bba_handle h, const bba_peer_handle* all, int count) {
  if (!h || !all) return BBA_ERR_INVALID_ARGUMENT;
  if (count != h->cfg.world_size) return Fail(h, BBA_ERR_INVALID_ARGUMENT, "bba_peer_import: need one handle per rank");
  if (count - 1 > bba::kMaxPeers) return Fail(h, BBA_ERR_UNSUPPORTED, "bba_peer_import: more than 8 ranks");
  if (bba_status st = CheckSurfels(h)) return st;
  UnmapPeers(h);
  bba::PeerSet ps{};
  for (int r = 0; r < count; ++r) {
    if (r == h->cfg.rank) continue;
    const bba_peer_handle& ph = all[r];
    if (ph.rank != r || ph.pitch_bytes != h->surfel_pitch_bytes || ph.surfels_size != h->surfels_size) {
      UnmapPeers(h);
      return Fail(h, BBA_ERR_INVALID_ARGUMENT, "bba_peer_import: replica layout differs between ranks");
    }
    cudaIpcMemHandle_t ipc;
    void* base_s = nullptr;
    std::memcpy(&ipc, ph.surfels_ipc, 64);
    cudaError_t e = cudaIpcOpenMemHandle(&base_s, ipc, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
      UnmapPeers(h);
      return Fail(h, BBA_ERR_CUDA, std::string("cudaIpcOpenMemHandle(surfels): ") + cudaGetErrorString(e));
    }
    h->peer_bases[h->peer_base_count++] = base_s;
    void* base_a = base_s;
    if (std::memcmp(ph.surfels_ipc, ph.active_ipc, 64) != 0) {
      std::memcpy(&ipc, ph.active_ipc, 64);
      e = cudaIpcOpenMemHandle(&base_a, ipc, cudaIpcMemLazyEnablePeerAccess);
      if (e != cudaSuccess) {
        UnmapPeers(h);
        return Fail(h, BBA_ERR_CUDA, std::string("cudaIpcOpenMemHandle(active): ") + cudaGetErrorString(e));
      }
      h->peer_bases[h->peer_base_count++] = base_a;
    }
    ps.surfels[ps.count] = reinterpret_cast<float*>(static_cast<char*>(base_s) + ph.surfels_offset);
    ps.active[ps.count] = reinterpret_cast<uint8_t*>(static_cast<char*>(base_a) + ph.active_offset);
    ++ps.count;
  }
  h->peers = ps;
  return BBA_OK;
}

int bba_peer_count(bba_handle h) { return h ? h->peers.count : 0; }

bba_status bba_mark_replica_rewritten(bba_handle h) {
  if (!h) return BBA_ERR_INVALID_ARGUMENT;
  h->replicated_pass_pending = true;   // -> PeerFence in front of the next kernel with peer stores
  return BBA_OK;
}

bba_status bba_peer_unmap(bba_handle h) {
  if (!h) return BBA_ERR_INVALID_ARGUMENT;
  UnmapPeers(h);
  return BBA_OK;
}

bba_status bba_set_collective(bba_handle h, bba_collective_fn fn, void* user) {
  if (!h) return BBA_ERR_INVALID_ARGUMENT;
  h->collective = fn;
  h->collective_user = user;
  return BBA_OK;
}

int bba_shard_surfel_owner(uint32_t surfel_index, int world_size) {
  return world_size > 1 ? static_cast<int>((surfel_index >> bba::kShardGranuleShift) % static_cast<uint32_t>(world_size)) : 0;
}

uint32_t bba_shard_surfel_local_index(uint32_t surfel_index, int world_size) {
  if (world_size <= 1) return surfel_index;
  const uint32_t g = surfel_index >> bba::kShardGranuleShift;
  return ((g / static_cast<uint32_t>(world_size)) << bba::kShardGranuleShift) | (surfel_index & ((1u << bba::kShardGranuleShift) - 1u));
}

uint32_t bba_shard_slice_length(uint32_t surfels_size, int world_size) {
  uint32_t len = 0;
  ShardSurfels(surfels_size, 0, world_size, nullptr, &len);
  return len;
}

int bba_shard_keyframe_owner(int list_index, int world_size) { return world_size > 1 ? list_index % world_size : 0; }

void bba_balance_keyframes(const float* cost, int count, int world_size, int* owner) {
  if (count > 0 && owner) BalanceWork(cost, count, world_size, owner);
}

uint64_t bba_kernel_launch_count(bba_handle h) { return h ? h->launches : 0; }

bba_status bba_set_profiling(bba_handle h, int enable) {
  if (!h) return BBA_ERR_INVALID_ARGUMENT;
  h->profiling = enable < 0 ? 0 : (enable > 2 ? 2 : enable);
  return BBA_OK;
}

bba_status bba_get_profile(bba_handle h, bba_profile* out, int reset) {
  if (!h || !out) return BBA_ERR_INVALID_ARGUMENT;
  *out = h->profile;
  if (reset) std::memset(&h->profile, 0, sizeof(h->profile));
  return BBA_OK;
}

bba_status bba_update_keyframe_host(bba_handle h, int id, const uint16_t* host_depth, const uint16_t* host_normals,
                                    const uint16_t* host_radius, const uint8_t* host_color_rgba, void* stream) {
  CHECK_KF(h, id);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  Keyframe& kf = h->keyframes[id];
  const int w = h->cfg.depth_width, hh = h->cfg.depth_height, cw = h->cfg.color_width, ch = h->cfg.color_height;
  // The library can only write into buffers it owns (keyframes added with bba_add_keyframe_host); caller-owned
  // device buffers are updated by the caller.
  const uint16_t* srcs[3] = {host_depth, host_normals, host_radius};
  const size_t pitches[3] = {kf.depth_pitch, kf.normals_pitch, kf.radius_pitch};
  for (int i = 0; i < 3; ++i) {
    if (!srcs[i]) continue;
    if (!kf.owned[i]) return Fail(h, BBA_ERR_STATE, "keyframe buffers are caller-owned; update them directly");
    BBA_CUDA(h, cudaMemcpy2DAsync(kf.owned[i], pitches[i], srcs[i], static_cast<size_t>(w) * 2, static_cast<size_t>(w) * 2, hh,
                                  cudaMemcpyHostToDevice, s));
  }
  if (host_color_rgba) {
    uint8_t* dst = static_cast<uint8_t*>(kf.owned_rgba);
    size_t dst_pitch = kf.rgba_pitch;
    if (!dst) {   // caller-owned colour image: only the library's luma array is refreshed, through a staging image
      if (!h->color_staging) {
        BBA_CUDA(h, cudaMallocPitch(reinterpret_cast<void**>(&h->color_staging), &h->color_staging_pitch, static_cast<size_t>(cw) * 4, ch));
      }
      dst = h->color_staging;
      dst_pitch = h->color_staging_pitch;
    }
    BBA_CUDA(h, cudaMemcpy2DAsync(dst, dst_pitch, host_color_rgba, static_cast<size_t>(cw) * 4,
                                  static_cast<size_t>(cw) * 4, ch, cudaMemcpyHostToDevice, s));
    if (bba_status st = AcquireLumaStaging(h, s)) return st;
    bba::LaunchExtractLuma(dst, dst_pitch, h->luma_staging, h->luma_staging_pitch, cw, ch, s);
    ++h->launches;
    BBA_CUDA(h, cudaGetLastError());
    BBA_CUDA(h, cudaMemcpy2DToArrayAsync(kf.luma, 0, 0, h->luma_staging, h->luma_staging_pitch, cw, ch, cudaMemcpyDeviceToDevice, s));
    BBA_CUDA(h, cudaEventRecord(h->luma_staging_free, s));
  }
  return BBA_OK;
}

}  // extern "C"
