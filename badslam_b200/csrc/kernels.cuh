// kernels.cuh -- launch interface between the host orchestration (badba.cu) and the sm_100a kernels.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "device_math.cuh"

namespace bba {

// Accumulator record per keyframe written by the pose kernel: 32 fp64 sums
//   [0..20] H upper triangle row-major, [21..26] b, [27] n_assoc, [28] n_photo,
//   [29] cost_depth, [30] cost_desc1, [31] cost_desc2
// followed (separately) by 2 u64 stage counters {n_inimg, n_depthok} for the byte model.
constexpr int kPoseAccSize = 32;

struct PoseAccumulateArgs {
  CameraParams cam;
  const float* surfels;      // 17-row SoA
  uint32_t pitch;            // floats per row
  uint32_t n;                // surfels_size
  const KfDevice* kfs;
  const int* work_list;      // keyframe ids to evaluate
  const int* work_count;     // device scalar
  const float* frames;       // 9 rows x frames_pitch: per-surfel unpacked normal, gp + t1, gp + t2 (SurfelFramesKernel); may be null
  uint32_t frames_pitch;     // floats per row
  KfDevice* work_records;    // [max_kf] scratch: the work list's KfDevice records in list order (pad = keyframe id), filled by
                             // LaunchPoseAccumulate so that a work group's <= 8 records are ONE contiguous bulk copy
  double* acc;               // [max_kf][32]
  unsigned long long* stage_counts;  // [max_kf][2]
  unsigned int* queue;       // global work-item counter, must be 0 at launch
};

// Persistent, TMA-staged pose residual/Jacobian/Hessian kernel (AccumulatePoseEstimationCoeffsCUDAKernel,
// kernel_opt_pose.cu:251-383, for a whole list of keyframes in one launch).
// with_stats: also accumulate residual costs + the stage counters (iteration 0 of a pose step, profiling, debug API).
// Per-surfel, pose-independent inputs of the descriptor residual, computed once per pose step (the surfels do not move while the
// keyframe poses are optimised): rows 0-2 unpacked + re-normalised normal (util_nvcc_only.cuh:83-95), rows 3-5 / 6-8 the tangent
// points gp + t1 / gp + t2 (cost_function.cuh:115-133).  frames: [9][frames_pitch] floats.
void LaunchSurfelFrames(const float* surfels, uint32_t pitch, uint32_t n, float* frames, uint32_t frames_pitch, cudaStream_t stream);
// max_work: upper bound of *work_count known to the host (sizes the record-packing launch that precedes the kernel).
// args.frames != null selects the variant that stages the precomputed frames instead of the packed normal / radius rows.
void LaunchPoseAccumulate(const PoseAccumulateArgs& args, int sm_count, bool with_stats, int max_work, cudaStream_t stream);

struct PoseSolveArgs {
  KfDevice* kfs;
  float* pose_est;             // [max_kf][7] global_T_frame estimates, updated in place
  double* acc;                 // consumed and re-zeroed
  unsigned long long* stage_counts;
  const int* work_in;          // list consumed by this iteration
  const int* count_in;
  int* work_out;               // list of keyframes that need another iteration
  int* count_out;
  int* iterations;             // [max_kf]
  int* converged;              // [max_kf]
  double* first_stats;         // [max_kf][8]: n_assoc n_photo cost_depth cost_desc1 cost_desc2 n_inimg n_depthok (iteration 0)
  unsigned long long* totals;  // [8] cumulative: kf_evals, n_inimg, n_depthok, n_assoc, n_photo (over all iterations)
  volatile int* host_flag;     // mapped pinned memory: {iterations completed, work items left}
  unsigned int* queue;         // PoseAccumulateKernel's work-item counter, re-armed here
  int iteration;
  int max_iterations;
};
// Device-side Gauss-Newton step for every keyframe in the list (direct_ba_alternating.cc:173-233).
void LaunchPoseSolve(const PoseSolveArgs& args, cudaStream_t stream);

// Replicas of the surfel buffer / active flags on the OTHER ranks of a one-process-per-GPU job, mapped into this process
// (CUDA IPC) and written directly over NVLink by the geometry kernels: the owner of a surfel stores its updated rows into
// every replica, so the "all-gather" of the geometry step is fused into the kernels' own final stores.
constexpr int kMaxPeers = 7;
struct PeerSet {
  int count;                   // 0: no peers mapped (single GPU, or the host-collective exchange is used)
  float* surfels[kMaxPeers];   // same pitch / layout as the local buffer
  uint8_t* active[kMaxPeers];
};

struct GeometryArgs {
  CameraParams cam;
  float* surfels;
  uint32_t pitch;
  uint32_t n;
  uint32_t begin, end;         // range of this rank's LOCAL surfel indices (SurfelShardToGlobal maps them; 0 .. n on one GPU)
  uint32_t shard_rank, shard_world;
  uint8_t* active;
  const KfDevice* kfs;
  const int* kf_list;          // non-inactive keyframes (ascending ids)
  int kf_count;
  unsigned int* queue;         // work-item counter (reset by the launcher)
  unsigned int* tile_epoch;    // [ceil(n / 32)] keyframe groups retired per tile (reset by the launcher)
  int tile_shift;              // log2(surfels per tile), 5..8; chosen by the launcher
  PeerSet peers;
};
// SetSurfelInactive + DetermineActiveSurfels (kernel_surfel_activation.cu:38-79) fused with the normal
// accumulation + update (kernel_opt_geometry.cu:527-597).
void LaunchActivationAndNormals(const GeometryArgs& args, int sm_count, bool determine_activation, bool update_normals, cudaStream_t stream);
// Position (+ descriptor) accumulation and per-surfel solve (kernel_opt_geometry.cu:118-231,273-361 or :417-507).
void LaunchPositionAndDescriptor(const GeometryArgs& args, int sm_count, cudaStream_t stream);

// Multi-GPU surfel sharding: 256-surfel granules are dealt round-robin to the ranks (granule g belongs to rank g % world), so
// that every rank sees the same mix of well- and poorly-observed surfels (surfels are stored in creation order, and the
// cost of a surfel is the number of keyframes that see it).  A rank addresses its surfels through a dense local index.
constexpr uint32_t kShardGranuleShift = 8;
__host__ __device__ inline uint32_t SurfelShardToGlobal(uint32_t local, uint32_t rank, uint32_t world) {
  return world <= 1 ? local : ((((local >> kShardGranuleShift) * world + rank) << kShardGranuleShift) | (local & ((1u << kShardGranuleShift) - 1u)));
}
// Exchange of the shards: 7 rows (x y z normal d1 d2 active-as-float) x shard_len floats per rank, in local index order.
constexpr int kShardRows = 7;
void LaunchPackShard(const float* surfels, uint32_t pitch, const uint8_t* active, uint32_t n, uint32_t rank, uint32_t world,
                     uint32_t shard_len, float* slice, cudaStream_t stream);
void LaunchUnpackShards(float* surfels, uint32_t pitch, uint8_t* active, uint32_t n, uint32_t shard_len, int world, int skip_rank,
                        const float* buffer, cudaStream_t stream);
// Pose results of the locally owned keyframes -> [K][17] floats (zeros elsewhere) for the sum all-reduce.
constexpr int kPoseSlot = 17;   // 7 pose, iterations, converged, 8 first-iteration statistics
void LaunchPackPoseResults(const int* ids, int n, const float* pose_est, const int* iterations, const int* converged,
                           const double* first_stats, float* out, cudaStream_t stream);

// Intrinsics + depth-deformation step (intrinsics.cu; OptimizeIntrinsicsCUDA, kernel_opt_intrinsics.cc:39-281).
constexpr int kIntrinsicsSums = 34;   // A (15) b1 (5) colour H (10) colour b (4), fp64
struct IntrinsicsArgs {
  CameraParams cam;
  const float* surfels;
  uint32_t pitch;
  uint32_t n;
  uint32_t begin, end;         // range of this rank's LOCAL surfel indices (SurfelShardToGlobal)
  uint32_t shard_rank, shard_world;
  const KfDevice* kfs;
  const int* kf_list;          // every keyframe (ascending ids)
  int kf_count;
  unsigned int* queue;         // work-item counter (reset by the launcher)
  double* sums;                // [kIntrinsicsSums]
  float* cell_B;               // [5][cell_count]
  float* cell_D;               // [cell_count]
  float* cell_b2;              // [cell_count]
  float* cell_obs;             // [cell_count] observation count (fp32 so that one sum all-reduce covers everything)
  uint32_t cell_count;
};
void LaunchIntrinsicsAccumulate(const IntrinsicsArgs& a, int sm_count, bool optimize_color, bool optimize_depth, cudaStream_t stream);
void LaunchIntrinsicsSchur(uint32_t cell_count, float* B, float* D, const float* b2, double* sums, cudaStream_t stream);
void LaunchIntrinsicsConvertSums(double* sums, float* head, bool to_float, cudaStream_t stream);
void LaunchIntrinsicsCellUpdate(uint32_t cell_count, const float* obs, const float* B, const float* D, const float* x1,
                                float* cfactor, cudaStream_t stream);

// PCG Gauss-Newton step over all unknowns (pcg.cu; BundleAdjustmentPCG, direct_ba_pcg.cc:43-819).
struct PcgArgs {
  CameraParams cam;
  const float* surfels;
  uint32_t pitch;
  uint32_t begin, end;         // range of this rank's LOCAL surfel indices (SurfelShardToGlobal maps them; 0 .. n on one GPU)
  uint32_t n;                  // surfels_size
  uint32_t shard_rank, shard_world;
  int alpha_d_slot;            // scalars slot that receives this launch's p^T J^T W J p: 1 on one GPU, 3 (exchanged, then added to 1) otherwise
  const KfDevice* kfs;         // every keyframe, ids 0 .. kf_count-1
  int kf_count;
  int gauge_kf;                // keyframe whose pose is fixed (no unknowns), direct_ba_pcg.cc:315-333
  int opt_poses, opt_geometry, opt_depth_intr, opt_color_intr;
  uint32_t surfel_start, surfel_stride;   // first surfel unknown, unknowns per surfel (1 or 3)
  uint32_t depth_intr_start, color_intr_start;
  float* r;                    // INIT
  float* M;                    // INIT
  const float* p;              // STEP1
  float* g;                    // STEP1
  double* scalars;             // [0] / [2] alpha_n, beta_n (swapping roles), [1] alpha_d
  unsigned int* queue;         // work-item counter (reset by the launcher)
};
// Layout of the fp64 scalar block: [0] / [2] alpha_n, beta_n (swapping roles), [1] alpha_d, [3] this rank's part of alpha_d
// (multi-GPU), then the workspace of the fixed-order grid sums of the vector kernels.
constexpr int kPcgPartialsA = 8, kPcgPartialsB = 8 + 2048, kPcgCounters = 8 + 4096, kPcgScalarDoubles = 8 + 4096 + 2;
void LaunchPcgAccumulate(const PcgArgs& a, int sm_count, bool init, cudaStream_t stream);
void LaunchPcgPackAlphaD(const double* scalars, float* tail, cudaStream_t stream);
void LaunchPcgUnpackAlphaD(double* scalars, const float* tail, cudaStream_t stream);
void LaunchPcgInit2(uint32_t n, uint32_t a_index, float a, int kf_count, const float* r, const float* M, float* delta, float* g, float* p,
                    double* scalars, int slot_alpha_n, int sm_count, cudaStream_t stream);
void LaunchPcgStep2(uint32_t n, uint32_t a_index, float* r, const float* M, float* delta, float* g, const float* p, double* scalars,
                    int slot_alpha_n, int slot_beta_n, int sm_count, cudaStream_t stream);
void LaunchPcgStep3(uint32_t n, uint32_t a_index, int kf_count, float* g, float* p, double* scalars, int slot_alpha_n, int slot_beta_n,
                    int sm_count, cudaStream_t stream);
void LaunchPcgUpdateSurfels(float* surfels, uint32_t pitch, uint32_t n, bool use_desc, uint32_t surfel_start, const float* delta,
                            cudaStream_t stream);
void LaunchPcgUpdateCfactor(float* cfactor, uint32_t cells, const float* delta, cudaStream_t stream);

// End-of-BA surfel maintenance (lifecycle.cu; PerformBASchemeEndTasks, direct_ba.cc:566-653).
struct KfRadius {
  const uint16_t* ptr;         // pitched u16 (IEEE half radius^2, keyframe.h radius_buffer)
  uint32_t pitch;              // bytes
  uint32_t pad;
};
struct SurfelStatsArgs {
  CameraParams cam;
  float* surfels;
  uint32_t pitch;
  uint32_t n;
  const KfDevice* kfs;         // every keyframe, ids 0 .. kf_count-1
  const KfRadius* radius;
  int kf_count;
  int min_observation_count;
  unsigned int* queue;
  unsigned int* tile_epoch;
  int tile_shift;              // chosen by the launcher
  unsigned int* deleted_count; // device scalar, += surfels deleted by this launch
  // multi-GPU: this rank handles the surfels of its granule shard (local indices [0, local_count)); with mapped peers the two
  // result rows (x = deletion marker, radius^2) are stored into every replica, like the geometry step's results
  uint32_t local_count, shard_rank, shard_world;
  PeerSet peers;
};
void LaunchObservationStats(SurfelStatsArgs a, int sm_count, cudaStream_t stream);
// Exchange of the end tasks' two result rows through the host collective (no mapped peers): slice = [2][shard_len] floats.
void LaunchPackStatsShard(const float* surfels, uint32_t pitch, uint32_t n, uint32_t rank, uint32_t world, uint32_t shard_len, float* slice,
                          cudaStream_t stream);
void LaunchUnpackStatsShards(float* surfels, uint32_t pitch, uint32_t n, uint32_t shard_len, int world, int skip_rank, const float* buffer,
                             cudaStream_t stream);
uint32_t CompactScratchWords(uint32_t n);   // size of block_sums for LaunchCompactSurfels
// Moves surviving surfels from the tail into the free spots; afterwards the first n - free_count slots are the surfels.
// active != nullptr: the active flags move with them (CompactSurfelsCUDA's adapt_active_surfels).
void LaunchCompactSurfels(float* surfels, uint32_t pitch, uint32_t n, uint32_t free_count, unsigned int* block_sums, uint8_t* active,
                          cudaStream_t stream);

// In-loop surfel lifecycle for ONE keyframe (CreateSurfelsForKeyframe / DetermineSupportingSurfelsAndMergeSurfels).
struct CovisEntry {              // one co-visible keyframe of the keyframe new surfels are created for
  float R[12];                   // covis_T_frame = covis.frame_T_global * keyframe.global_T_frame (direct_ba.cc:365-370)
  const uint16_t* depth;
  const uint16_t* normals;
  uint32_t depth_pitch, normals_pitch;
  uint32_t pad[2];
};
struct LifecycleArgs {
  CameraParams cam;
  float T[12];                   // frame_T_global of the keyframe
  float G[12];                   // global_T_frame
  const uint16_t* depth;
  const uint16_t* normals;
  const uint16_t* radius;
  uint32_t depth_pitch, normals_pitch, radius_pitch;
  cudaTextureObject_t tex;       // luma
  const uint8_t* rgba;           // the keyframe's uchar4 colour image (surfel colours)
  uint32_t rgba_pitch;
  float* surfels;
  uint32_t pitch, n;
  unsigned int* sup;             // [3][cells] supporting surfel indices
  unsigned int* cell_bits;       // [cells]
  uint32_t cells;
  unsigned int* flags;           // [w * h] new-surfel flag per pixel
  const CovisEntry* covis;
  int covis_count;
  int min_observation_count;
  float cell_merge_dist_squared;
  unsigned int* counter;         // device scalar (deleted surfels)
};
void LaunchSupportSurfels(const LifecycleArgs& a, int sm_count, cudaStream_t stream);   // sup[0] only (occupancy for the creation)
void LaunchMergeSurfels(const LifecycleArgs& a, int sm_count, cudaStream_t stream);     // supports + merge, += *counter
void LaunchSeedNewSurfels(const LifecycleArgs& a, bool filter, cudaStream_t stream);    // a.flags after LaunchSupportSurfels
uint32_t ScanScratchWords(uint32_t n);
void LaunchExclusiveScan(const unsigned int* in, uint32_t n, unsigned int* out, unsigned int* block_sums, cudaStream_t stream);
void LaunchCreateSurfels(const LifecycleArgs& a, const unsigned int* index, cudaStream_t stream);

// uchar4 (.w = luma) -> u8 plane.
void LaunchExtractLuma(const uint8_t* rgba, size_t rgba_pitch, uint8_t* luma, size_t luma_pitch, int w, int h, cudaStream_t stream);

}  // namespace bba
