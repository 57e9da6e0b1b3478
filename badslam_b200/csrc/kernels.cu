// kernels.cu -- hand-written sm_100a kernels of the direct-BA hot path.
//
//  * PoseAccumulateKernel: ONE persistent launch evaluates the pose normal equations of a whole LIST of
//    keyframes (the reference launches AccumulatePoseEstimationCoeffsCUDAKernel once per keyframe and
//    Gauss-Newton iteration, kernel_opt_pose.cc:74-88).  Surfel tiles are staged into shared memory by the
//    TMA engine (cp.async.bulk + mbarrier, double-buffered); each warp owns (tile, keyframe) work items,
//    keeps the 21 H + 6 b + 5 bookkeeping sums in registers across the whole tile, and reduces them with a
//    31-shuffle transposed butterfly followed by one fp64 RED per lane (the reference does 27 block-wide CUB
//    reductions + atomics per residual type per 256 surfels, gauss_newton.cuh:59-92).
//  * ActivationNormalsKernel / PositionDescriptorKernel: surfel-major geometry step.  One thread owns one
//    surfel, loops over all non-inactive keyframes with the accumulators in registers and applies the update
//    in the same kernel -- the reference's reset / K x accumulate / update launch chain with 16-72 bytes of
//    read-modify-write per associated pair (kernel_opt_geometry.cc:114-199) becomes one pass with none.
//
// Built with -use_fast_math like the reference (applications/badslam/CMakeLists.txt:74-75).
#include "kernels.cuh"

#include <cuda.h>

#include <algorithm>

namespace bba {

// ------------------------------------------------------------------------------------------------
// mbarrier / bulk-copy (TMA) primitives, raw PTX.

__device__ __forceinline__ uint32_t SmemAddr(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void MbarInit(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(SmemAddr(bar)), "r"(count));
}
__device__ __forceinline__ void FenceBarrierInit() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void MbarArriveExpectTx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(SmemAddr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void MbarArrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(SmemAddr(bar)) : "memory");
}
__device__ __forceinline__ void MbarWait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra.uni WAIT_DONE;\n"
      "bra.uni WAIT_LOOP;\n"
      "WAIT_DONE:\n"
      "}\n" ::"r"(SmemAddr(bar)),
      "r"(parity)
      : "memory");
}
// 1-D bulk copy global -> shared, completion signalled on an mbarrier (TMA engine; SASS UBLKCP).
__device__ __forceinline__ void BulkCopyG2S(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(SmemAddr(smem_dst)),
               "l"(gmem_src), "r"(bytes), "r"(SmemAddr(bar))
               : "memory");
}

// ------------------------------------------------------------------------------------------------

struct KfRegs {
  float T[12];
  const uint16_t* depth;
  const uint16_t* normals;
  cudaTextureObject_t tex;
  uint32_t depth_pitch, normals_pitch;
  int activation;
};

// The same record from shared memory (staged by the TMA engine together with the surfel tile).  Returns the keyframe id (pad).
__device__ __forceinline__ int LoadKfShared(const KfDevice* rec, KfRegs* r) {
  const float4* p = reinterpret_cast<const float4*>(rec);
  const float4 a = p[0], b = p[1], c = p[2];
  r->T[0] = a.x; r->T[1] = a.y; r->T[2] = a.z; r->T[3] = a.w;
  r->T[4] = b.x; r->T[5] = b.y; r->T[6] = b.z; r->T[7] = b.w;
  r->T[8] = c.x; r->T[9] = c.y; r->T[10] = c.z; r->T[11] = c.w;
  const ulonglong2 q = *reinterpret_cast<const ulonglong2*>(p + 3);
  r->depth = reinterpret_cast<const uint16_t*>(q.x);
  r->normals = reinterpret_cast<const uint16_t*>(q.y);
  const ulonglong2 q2 = *reinterpret_cast<const ulonglong2*>(p + 4);
  r->tex = static_cast<cudaTextureObject_t>(q2.x);
  r->depth_pitch = static_cast<uint32_t>(q2.y & 0xffffffffu);
  r->normals_pitch = static_cast<uint32_t>(q2.y >> 32);
  const int2 tail = *reinterpret_cast<const int2*>(p + 5);
  r->activation = tail.x;
  return tail.y;
}

// A texture handle that is the same in every lane, said in a way ptxas can see (a shuffle from lane 0): without it every
// TEX / TLD4 is wrapped in a per-lane "waterfall" loop (R2UR + predicated fetch + BRA.U.ANY, ~8 extra instructions per fetch).
// Must be called by all 32 lanes.
__device__ __forceinline__ cudaTextureObject_t UniformTexture(cudaTextureObject_t tex) {
  const unsigned long long t = tex;
  const unsigned lo = __shfl_sync(0xffffffffu, static_cast<unsigned>(t), 0);
  const unsigned hi = __shfl_sync(0xffffffffu, static_cast<unsigned>(t >> 32), 0);
  return (static_cast<unsigned long long>(hi) << 32) | lo;
}

// H += w J^T J (upper triangle), b += w r J (gauss_newton.cuh:59-92, per thread), with packed fp32x2 instructions
// (fma.rn.f32x2 / mul.rn.f32x2 -> SASS FFMA2 / FMUL2): each instruction updates two adjacent coefficients.  The per-lane
// accumulators are kept in a PAIR-ALIGNED order --
//   0..5  H00 H01 H02 H03 H04 H05 | 6..9 H12 H13 H14 H15 | 10..13 H22 H23 H24 H25 | 14,15 H34 H35 | 16,17 H44 H45 |
//   18..23 b0..b5 | 24 H11  25 H33  26 H55 | 27..31 statistics
// -- so that every row of the upper triangle is a run of (even, odd) column pairs of J plus at most one leading diagonal
// element; AccSlot() maps the order back to the row-major upper triangle + b the solver reads (gauss_newton.cuh:59-92).
// 12 FFMA2 + 3 FMUL2 + 3 FFMA + 1 FMUL per residual instead of 27 FFMA + 7 FMUL; each product / sum is rounded exactly as by the
// scalar instructions.
typedef unsigned long long F32x2;
__device__ __forceinline__ F32x2 Pack2(float lo, float hi) {
  F32x2 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void Unpack2(F32x2 v, float* lo, float* hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(*lo), "=f"(*hi) : "l"(v)); }
__device__ __forceinline__ F32x2 Mul2(F32x2 a, F32x2 b) {
  F32x2 r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ void Fma2(float* lo, float* hi, F32x2 a, F32x2 b) {   // (*lo, *hi) += a * b
  F32x2 c = Pack2(*lo, *hi);
  asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(c) : "l"(a), "l"(b));
  Unpack2(c, lo, hi);
}
__device__ __forceinline__ void AccumulateHbPacked(float (&acc)[kPoseAccSize], F32x2 J01, F32x2 J23, F32x2 J45, float raw, float w) {
  float J[6];
  Unpack2(J01, &J[0], &J[1]);
  Unpack2(J23, &J[2], &J[3]);
  Unpack2(J45, &J[4], &J[5]);
  const F32x2 ww = Pack2(w, w);
  float wj[6];
  Unpack2(Mul2(ww, J01), &wj[0], &wj[1]);
  Unpack2(Mul2(ww, J23), &wj[2], &wj[3]);
  Unpack2(Mul2(ww, J45), &wj[4], &wj[5]);
  const F32x2 d0 = Pack2(wj[0], wj[0]), d1 = Pack2(wj[1], wj[1]), d2 = Pack2(wj[2], wj[2]), d3 = Pack2(wj[3], wj[3]),
              d4 = Pack2(wj[4], wj[4]);
  Fma2(&acc[0], &acc[1], d0, J01);
  Fma2(&acc[2], &acc[3], d0, J23);
  Fma2(&acc[4], &acc[5], d0, J45);
  acc[24] += wj[1] * J[1];
  Fma2(&acc[6], &acc[7], d1, J23);
  Fma2(&acc[8], &acc[9], d1, J45);
  Fma2(&acc[10], &acc[11], d2, J23);
  Fma2(&acc[12], &acc[13], d2, J45);
  acc[25] += wj[3] * J[3];
  Fma2(&acc[14], &acc[15], d3, J45);
  Fma2(&acc[16], &acc[17], d4, J45);
  acc[26] += wj[5] * J[5];
  const float wr = w * raw;
  const F32x2 dr = Pack2(wr, wr);
  Fma2(&acc[18], &acc[19], dr, J01);
  Fma2(&acc[20], &acc[21], dr, J23);
  Fma2(&acc[22], &acc[23], dr, J45);
}
// J reaches the update through the packed registers; taking the diagonal terms from the array instead gives the same sums but a
// different instruction schedule of the pose kernel.
__device__ __forceinline__ void AccumulateHb(float (&acc)[kPoseAccSize], const float (&J)[6], float raw, float w) {
  AccumulateHbPacked(acc, Pack2(J[0], J[1]), Pack2(J[2], J[3]), Pack2(J[4], J[5]), raw, w);
}
// accumulator index in the pair-aligned order -> index in the solver's order (21 upper-triangle coefficients row-major, 6 b, 5 stats)
__device__ __forceinline__ int AccSlot(int lane) {
  //            H00 H01 H02 H03 H04 H05 H12 H13 H14 H15 H22 H23 H24 H25 H34 H35 H44 H45 b0  b1  b2  b3  b4  b5 H11 H33 H55
  constexpr unsigned long long lo = 0x0ull | (1ull << 5) | (2ull << 10) | (3ull << 15) | (4ull << 20) | (5ull << 25) | (7ull << 30) |
                                    (8ull << 35) | (9ull << 40) | (10ull << 45) | (11ull << 50) | (12ull << 55);   // slots 0..11
  constexpr unsigned long long mid = 13ull | (14ull << 5) | (16ull << 10) | (17ull << 15) | (18ull << 20) | (19ull << 25) | (21ull << 30) |
                                     (22ull << 35) | (23ull << 40) | (24ull << 45) | (25ull << 50) | (26ull << 55);   // slots 12..23
  constexpr unsigned long long hi = 6ull | (15ull << 5) | (20ull << 10);                                               // slots 24..26
  if (lane < 12) return static_cast<int>((lo >> (5 * lane)) & 31u);
  if (lane < 24) return static_cast<int>((mid >> (5 * (lane - 12))) & 31u);
  if (lane < 27) return static_cast<int>((hi >> (5 * (lane - 24))) & 31u);
  return lane;
}

constexpr int kPoseThreads = 256;
constexpr int kPoseMinCtas = 2;      // resident CTAs per SM the register allocation is tuned for
constexpr int kPoseUnroll = 1;       // surfels of a chunk evaluated concurrently per lane
constexpr int kPoseChunkShift = 8;   // log2 of the surfels one warp evaluates per (keyframe) sub-item
constexpr int kPoseStagedRows = 7;   // x y z normal radius^2 d1 d2
constexpr int kPoseStagedRowsPre = 14;   // x y z d1 d2 + the 9 frame rows (normal, tangent point 1, tangent point 2)
constexpr int kPoseGroup = 8;        // keyframes per work item

// Work decomposition.  A work ITEM is (group of <= 8 keyframes from the work list) x (tile of TILE surfels); items are
// handed out through a global counter in GROUP-MAJOR order, so at any moment all resident CTAs read the images of the
// same 8-16 keyframes (~12-24 MB: stays in the 126 MB L2) while surfel tiles stream through shared memory via TMA.
// Inside an item the 8 warps steal SUB-ITEMS (keyframe, 256- or 128-surfel chunk) from a shared-memory counter, which
// evens out the very different cost of culled vs. associated chunks.
// STATS: also produce the residual costs and the stage counters of the byte model (the reference computes its
// residual count / cost only in debug mode, kernel_opt_pose.cu:312-320,373-381).
// PRE: the per-surfel frames (unpacked normal, tangent points) are staged instead of the packed normal and the radius.
template <int TILE, bool STATS, bool PRE>
__global__ void __launch_bounds__(kPoseThreads, kPoseMinCtas) PoseAccumulateKernel(const __grid_constant__ PoseAccumulateArgs args) {
  constexpr int kRows = PRE ? kPoseStagedRowsPre : kPoseStagedRows;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  float* stage_base = reinterpret_cast<float*>(smem_raw);   // [2][kRows][TILE]
  __shared__ __align__(16) KfDevice s_kf[2][kPoseGroup];   // the work group's keyframe records, staged with the tile
  __shared__ __align__(8) uint64_t full_bar[2];
  __shared__ unsigned int s_item[2];
  __shared__ int s_sub[2];

  const int n_work = __ldg(args.work_count);
  if (n_work <= 0) return;

  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const uint32_t n_tiles = (args.n + TILE - 1) / TILE;
  const uint32_t n_groups = (n_work + kPoseGroup - 1) / kPoseGroup;
  const uint32_t n_items = n_groups * n_tiles;
  constexpr int kTileShift = (TILE == 1024) ? 10 : (TILE == 512) ? 9 : 8;

  const CameraParams& cam = args.cam;
  constexpr int kRowIds[kPoseStagedRows] = {kRowX, kRowY, kRowZ, kRowNormal, kRowRadiusSq, kRowD1, kRowD2};

  auto issue_tile = [&](uint32_t item, int s) {
    const uint32_t group = item / n_tiles, tile = item - group * n_tiles;
    const uint32_t base = tile * TILE;
    const uint32_t cnt = min(static_cast<uint32_t>(TILE), args.n - base);
    const uint32_t bytes = ((cnt * 4u + 15u) / 16u) * 16u;
    const uint32_t kf_bytes = static_cast<uint32_t>(sizeof(KfDevice)) * min(kPoseGroup, n_work - static_cast<int>(group) * kPoseGroup);
    MbarArriveExpectTx(&full_bar[s], bytes * kRows + kf_bytes);
    BulkCopyG2S(&s_kf[s][0], args.work_records + static_cast<size_t>(group) * kPoseGroup, kf_bytes, &full_bar[s]);
    if (PRE) {
      constexpr int kPreRowIds[5] = {kRowX, kRowY, kRowZ, kRowD1, kRowD2};
#pragma unroll
      for (int r = 0; r < 5; ++r)
        BulkCopyG2S(stage_base + (s * kRows + r) * TILE, args.surfels + static_cast<size_t>(kPreRowIds[r]) * args.pitch + base, bytes,
                    &full_bar[s]);
#pragma unroll
      for (int r = 0; r < 9; ++r)
        BulkCopyG2S(stage_base + (s * kRows + 5 + r) * TILE, args.frames + static_cast<size_t>(r) * args.frames_pitch + base, bytes,
                    &full_bar[s]);
    } else {
#pragma unroll
      for (int r = 0; r < kPoseStagedRows; ++r) {
        BulkCopyG2S(stage_base + (s * kRows + r) * TILE,
                    args.surfels + static_cast<size_t>(kRowIds[r]) * args.pitch + base, bytes, &full_bar[s]);
      }
    }
  };

  // No CTA-wide barrier in the item loop: a warp that has run out of sub-items of stage s moves on to stage s ^ 1 at once.
  // The LAST warp to leave a stage (shared-memory counter) re-arms it: claims the next item, resets the sub-item counter and
  // starts the TMA copies; everybody else finds the stage ready through its mbarrier phase.  When the queue is exhausted the
  // stage gets a sentinel item and a plain arrive, so that the waiting warps wake up and leave.  (A __syncthreads per item
  // instead, with thread 0 refilling the other stage, measured 2 % slower.)
  __shared__ int s_done[2];
  constexpr int kWarps = kPoseThreads / 32;
  auto arm_stage = [&](int s) {   // one thread
    s_sub[s] = 0;
    s_done[s] = 0;
    const unsigned int item = atomicAdd(args.queue, 1u);
    s_item[s] = item;
    if (item < n_items) issue_tile(item, s);
    else MbarArrive(&full_bar[s]);
  };
  if (tid == 0) {
    MbarInit(&full_bar[0], 1);
    MbarInit(&full_bar[1], 1);
    FenceBarrierInit();
    arm_stage(0);
    arm_stage(1);
  }
  __syncthreads();

  for (uint32_t it = 0;; ++it) {
    const int s = it & 1;
    MbarWait(&full_bar[s], (it >> 1) & 1);
    const unsigned int item = *reinterpret_cast<volatile unsigned int*>(&s_item[s]);
    if (item >= n_items) break;

    // staged rows: x y z normal radius^2 d1 d2, or (PRE) x y z d1 d2 + 9 frame rows
    const float* sx = stage_base + (s * kRows + 0) * TILE;
    const float* sy = sx + TILE;
    const float* sz = sy + TILE;
    const float* sn = sz + TILE;                 // !PRE: packed normal
    const float* sr = sn + TILE;                 // !PRE: radius^2
    const float* sd1 = PRE ? sz + TILE : sr + TILE;
    const float* sd2 = sd1 + TILE;
    const float* sf = sd2 + TILE;                // PRE: nx ny nz q1x q1y q1z q2x q2y q2z
    const uint32_t group = item / n_tiles;
    const uint32_t tile = item - group * n_tiles;
    const uint32_t base = tile * TILE;
    const uint32_t cnt = min(static_cast<uint32_t>(TILE), args.n - base);
    const int kfs_in_group = min(kPoseGroup, n_work - static_cast<int>(group) * kPoseGroup);
    // 256-surfel chunks (one warp-level reduction per 8 steps); 128 for a work list of fewer than 4 keyframes, so that every
    // warp of the CTA still finds a sub-item.  Choosing the size per item, from the keyframes in its group, measured 0.5 %
    // slower at cfg3: the extra reductions of the smaller chunks cost more than the idle warps of the few short groups.
    const int wanted_shift = n_work >= 4 ? kPoseChunkShift : 7;
    const int chunk_shift = wanted_shift < kTileShift ? wanted_shift : kTileShift;
    const uint32_t chunk_len = 1u << chunk_shift;
    const int chunks_per_tile = TILE >> chunk_shift;
    const int n_sub = kfs_in_group * chunks_per_tile;

    for (;;) {
      int sub = 0;
      if (lane == 0) sub = atomicAdd(&s_sub[s], 1);
      sub = __shfl_sync(0xffffffffu, sub, 0);
      if (sub >= n_sub) break;
      const int kf_local = sub / chunks_per_tile;
      const uint32_t j0 = static_cast<uint32_t>(sub - kf_local * chunks_per_tile) << chunk_shift;
      if (j0 >= cnt) continue;
      const uint32_t j1 = min(cnt, j0 + chunk_len);
      KfRegs K;
      const int kf = LoadKfShared(&s_kf[s][kf_local], &K);
      K.tex = UniformTexture(K.tex);

      float acc[kPoseAccSize];
#pragma unroll
      for (int i = 0; i < kPoseAccSize; ++i) acc[i] = 0.f;
      unsigned touched = 0;
      unsigned n_inimg = 0, n_depthok = 0;

#pragma unroll kPoseUnroll
      for (uint32_t j = j0 + lane; j < j0 + (j1 - j0 + 31u) / 32u * 32u; j += 32) {
        int st = 0;
        Assoc r;
        Vec3 gp, nrm;
        DescEval e;
        bool photo = false;
        if (j < j1) {
          gp = V3(sx[j], sy[j], sz[j]);
          if (ProjectIntoImage(cam, K.T, gp, &r)) {
            // Put every gather of the pair in flight before the first dependent use: the pixel's depth / normal /
            // cfactor, and -- speculatively, ~99 % of in-image pairs end up associated -- the six texture fetches of
            // the descriptor residual.  The association tests below then wait for the slowest load once.
            const PixelLoads l = LoadPixel(cam, K.depth, K.depth_pitch, K.normals, K.normals_pitch, r);
            nrm = PRE ? V3(sf[j], sf[TILE + j], sf[2 * TILE + j]) : UnpackNormal(__float_as_uint(sn[j]));
            if (cam.use_desc) {
              // Scalar on purpose.  A 2-wide (fp32x2) form of the post-association maths was no faster (3.7145 vs 3.7148 ms per
              // launch: the kernel waits on dependent-issue latency, not on the FMA pipe), and it rounds the sample coordinates
              // differently from the reference: the texture unit quantises the filter fraction to 1/256 pixel, so a last-bit
              // change flips the filter weights of ~1 % of the samples.
              float ccx, ccy;
              photo = DepthToColor(cam, r.pxf, r.pyf, &ccx, &ccy);
              float t1x, t1y, t2x, t2y;
              if (PRE) {
                ProjectTangentPoints(cam, K.T, V3(sf[3 * TILE + j], sf[4 * TILE + j], sf[5 * TILE + j]),
                                     V3(sf[6 * TILE + j], sf[7 * TILE + j], sf[8 * TILE + j]), &t1x, &t1y, &t2x, &t2y);
              } else {
                TangentProjections(cam, K.T, gp, nrm, sr[j], &t1x, &t1y, &t2x, &t2y);
              }
              EvalDescriptor(K.tex, ccx, ccy, t1x, t1y, t2x, t2y, sd1[j], sd2[j], &e);
            }
            st = Associate(cam, K.T, nrm, l, &r);
          }
        }
        if (STATS) {
          // per-lane counts (one predicated add each), summed over the warp once per chunk below
          n_inimg += st >= 1;
          n_depthok += st >= 2;
        }
        const unsigned assoc_mask = __ballot_sync(0xffffffffu, st == 3);
        if (assoc_mask == 0) continue;
        touched |= assoc_mask;
        if (st == 3) {
          acc[27] += 1.f;
          if (cam.use_depth) {
            float inv_stddev;
            Vec3 up;
            const float raw = DepthResidual(cam, r, &inv_stddev, &up);
            // kernel_opt_pose.cu:88-93
            float J[6];
            J[0] = inv_stddev * r.ln.x;
            J[1] = inv_stddev * r.ln.y;
            J[2] = inv_stddev * r.ln.z;
            J[3] = inv_stddev * (-r.ln.y * up.z + r.ln.z * up.y);
            J[4] = inv_stddev * (r.ln.x * up.z - r.ln.z * up.x);
            J[5] = inv_stddev * (-r.ln.x * up.y + r.ln.y * up.x);
            AccumulateHb(acc, J, raw, DepthWeight(raw));
            if (STATS) acc[29] += DepthCost(raw);
          }
          if (cam.use_desc && photo) {
            acc[28] += 1.f;
            float J[6];
            DescPoseJacobian(cam, r.lp, e.gx1, e.gy1, J);
            AccumulateHb(acc, J, e.r1, DescWeight(e.r1));
            DescPoseJacobian(cam, r.lp, e.gx2, e.gy2, J);
            AccumulateHb(acc, J, e.r2, DescWeight(e.r2));
            if (STATS) {
              acc[30] += DescCost(e.r1);
              acc[31] += DescCost(e.r2);
            }
          }
        }
      }

      if (touched) {
        const float total = WarpTransposeReduce(acc, lane);
        atomicAdd(args.acc + static_cast<size_t>(kf) * kPoseAccSize + AccSlot(lane), static_cast<double>(total));
      }
      if (STATS) {
        n_inimg = __reduce_add_sync(0xffffffffu, n_inimg);
        n_depthok = __reduce_add_sync(0xffffffffu, n_depthok);
      }
      if (STATS && lane == 0 && n_inimg) {
        atomicAdd(args.stage_counts + 2 * kf, static_cast<unsigned long long>(n_inimg));
        if (n_depthok) atomicAdd(args.stage_counts + 2 * kf + 1, static_cast<unsigned long long>(n_depthok));
      }
    }
    __syncwarp();
    if (lane == 0) {
      __threadfence_block();   // this warp's reads of stage s are complete before the stage can be handed back
      if (atomicAdd(&s_done[s], 1) == kWarps - 1) {
        __threadfence_block();
        arm_stage(s);
      }
    }
  }
}

// work_records[i] = kfs[work_list[i]] with pad = the keyframe id: makes the records of a work group contiguous.
__global__ void __launch_bounds__(128) PackWorkRecordsKernel(const KfDevice* __restrict__ kfs, const int* __restrict__ work_list,
                                                             const int* __restrict__ work_count, KfDevice* __restrict__ records) {
  const int n = __ldg(work_count);
  constexpr int kWords = sizeof(KfDevice) / 16;   // 6 x 16 bytes per record
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n * kWords; i += gridDim.x * blockDim.x) {
    const int rec = i / kWords, w = i - rec * kWords;
    const int kf = __ldg(work_list + rec);
    uint4 v = __ldg(reinterpret_cast<const uint4*>(kfs + kf) + w);
    if (w == kWords - 1) v.y = static_cast<unsigned int>(kf);   // KfDevice::pad
    reinterpret_cast<uint4*>(records + rec)[w] = v;
  }
}

template <int TILE, bool STATS, bool PRE>
static void LaunchPoseAccumulateT(const PoseAccumulateArgs& args, int sm_count, cudaStream_t stream) {
  const size_t smem = static_cast<size_t>(2) * (PRE ? kPoseStagedRowsPre : kPoseStagedRows) * TILE * sizeof(float);
  static bool configured = false;
  if (!configured) {
    cudaFuncSetAttribute(PoseAccumulateKernel<TILE, STATS, PRE>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    configured = true;
  }
  PoseAccumulateKernel<TILE, STATS, PRE><<<kPoseMinCtas * sm_count, kPoseThreads, smem, stream>>>(args);   // persistent
}

template <bool STATS>
static void LaunchPoseAccumulateS(const PoseAccumulateArgs& args, int sm_count, cudaStream_t stream) {
  // Tile size: as large as possible (one group of TMA transactions per item), but small enough that a keyframe group still
  // yields several items per resident CTA.  With the precomputed frames 14 rows are staged: 512 surfels x 2 stages = 56 KB per
  // CTA (two CTAs per SM), the same footprint as 1024 surfels of the 7-row variant.
  const uint64_t slots = static_cast<uint64_t>(kPoseMinCtas * sm_count) * 4;
  if (args.frames != nullptr) {
    if (args.n >= slots * 512) LaunchPoseAccumulateT<512, STATS, true>(args, sm_count, stream);
    else LaunchPoseAccumulateT<256, STATS, true>(args, sm_count, stream);
    return;
  }
  if (args.n >= slots * 1024) LaunchPoseAccumulateT<1024, STATS, false>(args, sm_count, stream);
  else if (args.n >= slots * 512) LaunchPoseAccumulateT<512, STATS, false>(args, sm_count, stream);
  else LaunchPoseAccumulateT<256, STATS, false>(args, sm_count, stream);
}

void LaunchPoseAccumulate(const PoseAccumulateArgs& args, int sm_count, bool with_stats, int max_work, cudaStream_t stream) {
  if (args.n == 0) return;
  PackWorkRecordsKernel<<<(max_work * 6 + 127) / 128, 128, 0, stream>>>(args.kfs, args.work_list, args.work_count, args.work_records);
  if (with_stats) LaunchPoseAccumulateS<true>(args, sm_count, stream);
  else LaunchPoseAccumulateS<false>(args, sm_count, stream);
}

__global__ void __launch_bounds__(256) SurfelFramesKernel(const float* __restrict__ surfels, uint32_t pitch, uint32_t n,
                                                          float* __restrict__ frames, uint32_t fp) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const size_t P = pitch;
  const Vec3 gp = V3(surfels[kRowX * P + i], surfels[kRowY * P + i], surfels[kRowZ * P + i]);
  const Vec3 nrm = UnpackNormal(__float_as_uint(surfels[kRowNormal * P + i]));
  Vec3 q1, q2;
  TangentPoints(gp, nrm, surfels[kRowRadiusSq * P + i], &q1, &q2);
  const size_t F = fp;
  frames[0 * F + i] = nrm.x; frames[1 * F + i] = nrm.y; frames[2 * F + i] = nrm.z;
  frames[3 * F + i] = q1.x;  frames[4 * F + i] = q1.y;  frames[5 * F + i] = q1.z;
  frames[6 * F + i] = q2.x;  frames[7 * F + i] = q2.y;  frames[8 * F + i] = q2.z;
}

void LaunchSurfelFrames(const float* surfels, uint32_t pitch, uint32_t n, float* frames, uint32_t frames_pitch, cudaStream_t stream) {
  if (n == 0) return;
  SurfelFramesKernel<<<(n + 255) / 256, 256, 0, stream>>>(surfels, pitch, n, frames, frames_pitch);
}

// ------------------------------------------------------------------------------------------------
// Geometry step.  One thread owns one surfel and keeps its accumulators in registers while it walks over a GROUP of
// keyframes; work items (keyframe group, 256-surfel tile) are handed out group-major through a global counter so that
// all resident CTAs gather from the same <= 16 keyframes' images at a time (L2-resident) -- the surfel-major variant
// that looped over all K keyframes per thread re-read the images from HBM ~40 times (profiles/r1_notes.md).
// Between groups the partial sums of a surfel are parked in the scratch rows 8..16 of the surfel buffer (the rows the
// reference uses for exactly this purpose, kernels.cuh:78-86); a per-tile epoch word orders (group g, tile t) after
// (group g-1, tile t).  With K <= 16 there is a single group and no scratch traffic at all.

constexpr int kGeoThreads = 256;
// Keyframes per work item.  A group's images (1.5 MB per keyframe at 640x480) are what all resident warps gather from at one
// time; 16 keeps them in a fifth of the L2.  32 / 64 / 200 moved the two geometry kernels by -10 % ... +38 % on one rank's share
// of an 8-GPU cfg3 job, none better for both.
constexpr int kGeoGroup = 16;

__device__ __forceinline__ unsigned int LoadAcquire(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void StoreRelease(unsigned int* p, unsigned int v) {
  asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// Work items are owned by WARPS (no CTA-wide barrier anywhere in these kernels): a warp takes (group, 256-surfel tile),
// waits until the previous group of that tile has been retired, and walks the tile in 8 sub-steps of 32 surfels.
__device__ __forceinline__ bool NextGeoItem(const GeometryArgs& a, uint32_t n_tiles, uint32_t n_items, uint32_t* group, uint32_t* tile) {
  unsigned int item = 0;
  if ((threadIdx.x & 31) == 0) {
    item = atomicAdd(a.queue, 1u);
    if (item < n_items) {
      const uint32_t g = item / n_tiles, t = item - g * n_tiles;
      while (LoadAcquire(a.tile_epoch + t) < g) __nanosleep(64);
    }
  }
  item = __shfl_sync(0xffffffffu, item, 0);
  if (item >= n_items) return false;
  *group = item / n_tiles;
  *tile = item - *group * n_tiles;
  return true;
}

__device__ __forceinline__ void RetireGeoItem(const GeometryArgs& a, uint32_t group, uint32_t tile) {
  __syncwarp();
  if ((threadIdx.x & 31) == 0) {
    __threadfence();
    StoreRelease(a.tile_epoch + tile, group + 1);
  }
}

// Final stores of the geometry step: the local replica and, when peers are mapped, every other rank's replica (NVLink).
__device__ __forceinline__ void StoreSurfelRow(const GeometryArgs& a, int row, uint32_t i, float v) {
  const size_t o = static_cast<size_t>(row) * a.pitch + i;
  a.surfels[o] = v;
#pragma unroll
  for (int p = 0; p < kMaxPeers; ++p)
    if (p < a.peers.count) a.peers.surfels[p][o] = v;
}
__device__ __forceinline__ void StoreActiveFlag(const GeometryArgs& a, uint32_t i, uint8_t v) {
  a.active[i] = v;
#pragma unroll
  for (int p = 0; p < kMaxPeers; ++p)
    if (p < a.peers.count) a.peers.active[p][i] = v;
}

// The <= kGeoGroup keyframe records of a work item, copied once per item into the warp's own shared-memory slice (coalesced
// 16-byte loads; the per-keyframe reads in the pair loop are then conflict-free broadcasts with a fixed ~25-cycle latency
// instead of a chain of dependent L1 accesses: keyframe id -> record row 2 -> rows 0, 1 -> image pointers).  Staging all
// records of the launch once per CTA instead measured slower (position + descriptor 4.76 vs 4.58 ms at cfg3): the per-warp
// slices keep the records a warp reads next to each other.
__device__ __forceinline__ void StageGroupRecords(const KfDevice* __restrict__ kfs, const int* __restrict__ kf_list, int count,
                                                  KfDevice* dst, int lane) {
  constexpr int kWords = sizeof(KfDevice) / 16;
  __syncwarp();   // the previous item's readers are done
  const int my_kf = lane < count ? __ldg(kf_list + lane) : 0;
#pragma unroll
  for (int w = 0; w < (kGeoGroup * kWords + 31) / 32; ++w) {
    const int idx = w * 32 + lane, rec = idx / kWords, part = idx - rec * kWords;
    const int kf = __shfl_sync(0xffffffffu, my_kf, rec & 31);
    if (rec < count) {
      uint4 v = __ldg(reinterpret_cast<const uint4*>(kfs + kf) + part);
      reinterpret_cast<uint4*>(dst + rec)[part] = v;
    }
  }
  __syncwarp();
}

// One (surfel, keyframe) pair between "gathers issued" and "gathers consumed".
struct PendingPair {
  bool in_image;
  Assoc r;
  PixelLoads l;
};

template <bool DETERMINE, bool NORMALS>
__global__ void __launch_bounds__(kGeoThreads) ActivationNormalsKernel(const __grid_constant__ GeometryArgs a) {
  extern __shared__ __align__(16) unsigned char geo_smem[];   // one kGeoGroup-record slice per warp
  KfDevice* s_kfs = reinterpret_cast<KfDevice*>(geo_smem);
  const uint32_t tile_len = 1u << a.tile_shift;
  const uint32_t n_tiles = (a.end - a.begin + tile_len - 1) >> a.tile_shift;
  const uint32_t n_groups = (a.kf_count + kGeoGroup - 1) / kGeoGroup;
  const uint32_t n_items = n_groups * n_tiles;
  const size_t P = a.pitch;
  const int lane = threadIdx.x & 31;
  uint32_t group, tile;
  while (NextGeoItem(a, n_tiles, n_items, &group, &tile)) {
    const bool first = group == 0, last = group + 1 == n_groups;
    const int j_begin = group * kGeoGroup, j_end = min(a.kf_count, static_cast<int>(group + 1) * kGeoGroup);
    const int n_kf = j_end - j_begin;
    KfDevice* recs = s_kfs + (threadIdx.x >> 5) * kGeoGroup;
    StageGroupRecords(a.kfs, a.kf_list + j_begin, n_kf, recs, lane);
    for (uint32_t sub = 0; sub < tile_len / 32; ++sub) {
      const uint32_t li = a.begin + (tile << a.tile_shift) + sub * 32 + lane;
      const uint32_t i = SurfelShardToGlobal(li, a.shard_rank, a.shard_world);
      if (li >= a.end || i >= a.n) continue;
      const uint8_t flags = a.active[i];
      if (!DETERMINE && !(flags & kSurfelActiveFlag)) continue;   // normals are updated for active surfels only
      bool act = !DETERMINE;
      float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
      if (!first) {
        if (NORMALS) {
          s0 = __ldcg(a.surfels + (kRowAccum0 + 0) * P + i);
          s1 = __ldcg(a.surfels + (kRowAccum0 + 1) * P + i);
          s2 = __ldcg(a.surfels + (kRowAccum0 + 2) * P + i);
          s3 = __ldcg(a.surfels + (kRowAccum0 + 3) * P + i);
        }
        if (DETERMINE) act = __ldcg(a.surfels + (kRowAccum0 + 4) * P + i) != 0.f;
      }
      if (NORMALS || !act) {   // activation alone stops at the first association with an active keyframe
        const Vec3 gp = V3(a.surfels[kRowX * P + i], a.surfels[kRowY * P + i], a.surfels[kRowZ * P + i]);
        const Vec3 nrm = UnpackNormal(__float_as_uint(a.surfels[kRowNormal * P + i]));
        // The sums in keyframe order: the summation order -- and with it the result -- is the reference's (one thread,
        // ascending keyframes).  Two pairs in flight per thread measured slower at cfg3: 78 instead of 64 registers, 24
        // instead of 32 warps / SM, 2.54 instead of 2.26 ms.
        auto issue = [&](const KfRegs& K, PendingPair* p) {
          p->in_image = (NORMALS || K.activation == 0) && ProjectIntoImage(a.cam, K.T, gp, &p->r);   // activation only looks at kActive keyframes
          if (p->in_image) p->l = LoadPixel(a.cam, K.depth, K.depth_pitch, K.normals, K.normals_pitch, p->r);
        };
        auto consume = [&](const KfRegs& K, PendingPair* p) {
          if (!p->in_image || Associate(a.cam, K.T, nrm, p->l, &p->r) != 3) return;
          if (K.activation == 0) act = true;
          if (NORMALS) {
            // kernel_opt_geometry.cu:545-553: global_R_frame * local normal, global_R_frame = R(frame_T_global)^T
            const Vec3 ln = U16ToImageSpaceNormal(p->r.kf_normal);
            s0 += K.T[0] * ln.x + K.T[4] * ln.y + K.T[8] * ln.z;
            s1 += K.T[1] * ln.x + K.T[5] * ln.y + K.T[9] * ln.z;
            s2 += K.T[2] * ln.x + K.T[6] * ln.y + K.T[10] * ln.z;
            s3 += 1.f;
          }
        };
        for (int j = 0; j < n_kf; ++j) {
          KfRegs K0;
          PendingPair p0;
          LoadKfShared(recs + j, &K0);
          issue(K0, &p0);
          consume(K0, &p0);
          if (!NORMALS && act) break;
        }
      }
      if (!last) {
        if (NORMALS) {
          __stcg(a.surfels + (kRowAccum0 + 0) * P + i, s0);
          __stcg(a.surfels + (kRowAccum0 + 1) * P + i, s1);
          __stcg(a.surfels + (kRowAccum0 + 2) * P + i, s2);
          __stcg(a.surfels + (kRowAccum0 + 3) * P + i, s3);
        }
        if (DETERMINE) __stcg(a.surfels + (kRowAccum0 + 4) * P + i, act ? 1.f : 0.f);
      } else {
        // SetSurfelInactive + DetermineActiveSurfels (kernel_surfel_activation.cu:38-79)
        if (DETERMINE) StoreActiveFlag(a, i, act ? kSurfelActiveFlag : static_cast<uint8_t>(flags & ~kSurfelActiveFlag));
        if (NORMALS && act && s3 >= 1.f) {
          // kernel_opt_geometry.cu:577-597: the mean is packed without re-normalisation
          const float inv = 1.f / s3;
          StoreSurfelRow(a, kRowNormal, i, __uint_as_float(PackNormal(V3(inv * s0, inv * s1, inv * s2))));
        }
      }
    }
    RetireGeoItem(a, group, tile);
  }
}

template <bool USE_DEPTH, bool USE_DESC>
__global__ void __launch_bounds__(kGeoThreads, 3) PositionDescriptorKernel(const __grid_constant__ GeometryArgs a) {
  extern __shared__ __align__(16) unsigned char geo_smem[];   // one kGeoGroup-record slice per warp
  KfDevice* s_kfs = reinterpret_cast<KfDevice*>(geo_smem);
  const uint32_t tile_len = 1u << a.tile_shift;
  const uint32_t n_tiles = (a.end - a.begin + tile_len - 1) >> a.tile_shift;
  const uint32_t n_groups = (a.kf_count + kGeoGroup - 1) / kGeoGroup;
  const uint32_t n_items = n_groups * n_tiles;
  const size_t P = a.pitch;
  const int lane = threadIdx.x & 31;
  uint32_t group, tile;
  while (NextGeoItem(a, n_tiles, n_items, &group, &tile)) {
    const bool first = group == 0, last = group + 1 == n_groups;
    const int j_begin = group * kGeoGroup, j_end = min(a.kf_count, static_cast<int>(group + 1) * kGeoGroup);
    KfDevice* recs = s_kfs + (threadIdx.x >> 5) * kGeoGroup;
    StageGroupRecords(a.kfs, a.kf_list + j_begin, j_end - j_begin, recs, lane);
    for (uint32_t sub = 0; sub < tile_len / 32; ++sub) {
      const uint32_t li = a.begin + (tile << a.tile_shift) + sub * 32 + lane;
      const uint32_t i = SurfelShardToGlobal(li, a.shard_rank, a.shard_world);
      // The keyframe loop below is executed by the whole warp (a lane without a live surfel just skips every pair): the
      // per-keyframe record -- in particular the texture handle -- is then provably warp-uniform, see UniformTexture().
      const bool live = li < a.end && i < a.n && (a.active[i] & kSurfelActiveFlag);
      if (__ballot_sync(0xffffffffu, live) == 0) continue;
      Vec3 gp = V3(0.f, 0.f, 0.f), nrm = V3(0.f, 0.f, 1.f);
      float radius_sq = 0.f, d1 = 0.f, d2 = 0.f;
      if (live) {
        gp = V3(a.surfels[kRowX * P + i], a.surfels[kRowY * P + i], a.surfels[kRowZ * P + i]);
        nrm = UnpackNormal(__float_as_uint(a.surfels[kRowNormal * P + i]));
        if (USE_DESC) {
          radius_sq = a.surfels[kRowRadiusSq * P + i];
          d1 = a.surfels[kRowD1 * P + i];
          d2 = a.surfels[kRowD2 * P + i];
        }
      }
      // 3x3 normal equations over (t along normal, d1, d2): H00 H01 H02 H11 H12 H22 | b0 b1 b2
      float H00 = 0.f, H01 = 0.f, H02 = 0.f, H11 = 0.f, H22 = 0.f, b0 = 0.f, b1 = 0.f, b2 = 0.f;
      const float H12 = 0.f;   // never accumulated by the reference either (kernel_opt_geometry.cu:216-227)
      if (!first && live) {
        // same row assignment as the reference's accumulators (kernel_opt_geometry.cu:216-227)
        H00 = __ldcg(a.surfels + (kRowAccum0 + 0) * P + i);
        b0 = __ldcg(a.surfels + (kRowAccum0 + 6) * P + i);
        if (USE_DESC) {
          H01 = __ldcg(a.surfels + (kRowAccum0 + 1) * P + i);
          H02 = __ldcg(a.surfels + (kRowAccum0 + 2) * P + i);
          H11 = __ldcg(a.surfels + (kRowAccum0 + 3) * P + i);
          H22 = __ldcg(a.surfels + (kRowAccum0 + 5) * P + i);
          b1 = __ldcg(a.surfels + (kRowAccum0 + 7) * P + i);
          b2 = __ldcg(a.surfels + (kRowAccum0 + 8) * P + i);
        }
      }
      for (int j = 0; j < j_end - j_begin; ++j) {
        KfRegs K;
        LoadKfShared(recs + j, &K);
        K.tex = UniformTexture(K.tex);
        Assoc r;
        if (!live || !ProjectIntoImage(a.cam, K.T, gp, &r)) continue;
        // all gathers of the pair in flight before the first dependent use (see PoseAccumulateKernel)
        const PixelLoads l = LoadPixel(a.cam, K.depth, K.depth_pitch, K.normals, K.normals_pitch, r);
        DescEval e;
        bool photo = false;
        if (USE_DESC) {
          // Scalar on purpose (see PoseAccumulateKernel): a 2-wide form of this maths lost the bit-exact agreement of the
          // surfel positions with the reference (errors up to 9e-5 m on 0.07 % of the surfels).
          float ccx, ccy;
          photo = DepthToColor(a.cam, r.pxf, r.pyf, &ccx, &ccy);
          float t1x, t1y, t2x, t2y;
          TangentProjections(a.cam, K.T, gp, nrm, radius_sq, &t1x, &t1y, &t2x, &t2y);
          EvalDescriptor(K.tex, ccx, ccy, t1x, t1y, t2x, t2y, d1, d2, &e);
        }
        if (Associate(a.cam, K.T, nrm, l, &r) != 3) continue;
        if (USE_DEPTH) {
          float inv_stddev;
          Vec3 up;
          const float raw = DepthResidual(a.cam, r, &inv_stddev, &up);
          const float jac = -inv_stddev;   // kernel_opt_geometry.cu:138
          const float w = DepthWeight(raw);
          if (USE_DESC) {
            H00 += w * jac * jac;
            b0 += w * raw * jac;
          } else {
            // kernel_opt_geometry.cu:452-456
            const float wj = w * jac;
            H00 += wj * jac;
            b0 += wj * raw;
          }
        }
        if (USE_DESC && photo) {
          // kernel_opt_geometry.cu:176-181
          const float term1 = -a.cam.cfx * (r.ln.x * r.lp.z - r.ln.z * r.lp.x);
          const float term2 = -a.cam.cfy * (r.ln.y * r.lp.z - r.ln.z * r.lp.y);
          const float term3 = 1.f / (r.lp.z * r.lp.z);
          const float j1 = -(e.gx1 * term1 + e.gy1 * term2) * term3;
          const float j2 = -(e.gx2 * term1 + e.gy2 * term2) * term3;
          constexpr float jd = -1.f;
          const float w1 = DescWeight(e.r1), wr1 = w1 * e.r1;
          const float w2 = DescWeight(e.r2), wr2 = w2 * e.r2;
          H00 += w1 * j1 * j1 + w2 * j2 * j2;
          H01 += w1 * j1 * jd;
          H11 += w1 * jd * jd;
          b0 += wr1 * j1 + wr2 * j2;
          b1 += wr1 * jd;
          H02 += w2 * j2 * jd;
          H22 += w2 * jd * jd;
          b2 += wr2 * jd;
        }
      }

      if (!live) continue;
      if (!last) {
        __stcg(a.surfels + (kRowAccum0 + 0) * P + i, H00);
        __stcg(a.surfels + (kRowAccum0 + 6) * P + i, b0);
        if (USE_DESC) {
          __stcg(a.surfels + (kRowAccum0 + 1) * P + i, H01);
          __stcg(a.surfels + (kRowAccum0 + 2) * P + i, H02);
          __stcg(a.surfels + (kRowAccum0 + 3) * P + i, H11);
          __stcg(a.surfels + (kRowAccum0 + 5) * P + i, H22);
          __stcg(a.surfels + (kRowAccum0 + 7) * P + i, b1);
          __stcg(a.surfels + (kRowAccum0 + 8) * P + i, b2);
        }
      } else if (!USE_DESC) {
        // UpdateSurfelPositionCUDAKernel, kernel_opt_geometry.cu:487-507
        if (H00 > 1e-6f) {
          const float t = -1.f * b0 / H00;
          StoreSurfelRow(a, kRowX, i, gp.x + t * nrm.x);
          StoreSurfelRow(a, kRowY, i, gp.y + t * nrm.y);
          StoreSurfelRow(a, kRowZ, i, gp.z + t * nrm.z);
        }
      } else {
        // UpdateSurfelPositionAndDescriptorCUDAKernel, kernel_opt_geometry.cu:273-361 (in-place Cholesky)
        constexpr float kEpsilon = 1e-6f;
        const float L00 = sqrtf(H00 + kEpsilon);
        const float L01 = H01 / L00;
        const float L11 = sqrtf((H11 + kEpsilon) - L01 * L01);
        const float L02 = H02 / L00;
        const float L12 = (H12 - L02 * L01) / L11;
        const float L22 = sqrtf((H22 + kEpsilon) - L02 * L02 - L12 * L12);
        const float y0 = b0 / L00;
        const float y1 = (b1 - L01 * y0) / L11;
        const float y2 = (b2 - L02 * y0 - L12 * y1) / L22;
        const float x2 = y2 / L22;
        const float x1 = (y1 - L12 * x2) / L11;
        const float x0 = (y0 - L02 * x2 - L01 * x1) / L00;
        if (x0 != 0) {
          StoreSurfelRow(a, kRowX, i, gp.x - x0 * nrm.x);
          StoreSurfelRow(a, kRowY, i, gp.y - x0 * nrm.y);
          StoreSurfelRow(a, kRowZ, i, gp.z - x0 * nrm.z);
        }
        if (x1 != 0) StoreSurfelRow(a, kRowD1, i, fmaxf(-180.f, fminf(180.f, d1 - x1)));
        if (x2 != 0) StoreSurfelRow(a, kRowD2, i, fmaxf(-180.f, fminf(180.f, d2 - x2)));
      }
    }
    RetireGeoItem(a, group, tile);
  }
}

constexpr size_t kGeoSmemBytes = sizeof(KfDevice) * (kGeoThreads / 32) * kGeoGroup;   // one record slice per warp

// Persistent grid: as many CTAs as can be co-resident (the epoch wait relies on every launched CTA being scheduled).
// The tile (the unit one warp walks through, 32..256 surfels) is chosen so that every keyframe group offers several
// items per resident warp: with too few tiles the per-tile epoch chain serialises the groups (seen at 2+ ranks).
template <typename Kernel>
static uint32_t GeoGrid(Kernel kernel, GeometryArgs* a, int sm_count) {
  int per_sm = 0;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kGeoThreads, kGeoSmemBytes);
  if (per_sm < 1) per_sm = 1;
  const uint64_t resident_warps = static_cast<uint64_t>(per_sm) * sm_count * (kGeoThreads / 32);
  const uint32_t n = a->end - a->begin;
  int shift = 8;
  while (shift > 5 && 2 * static_cast<uint64_t>((n + (1u << shift) - 1) >> shift) < 3 * resident_warps) --shift;
  a->tile_shift = shift;
  const uint32_t n_tiles = (n + (1u << shift) - 1) >> shift;
  const uint32_t n_groups = (a->kf_count + kGeoGroup - 1) / kGeoGroup;
  const uint64_t n_items = static_cast<uint64_t>(n_tiles) * (n_groups ? n_groups : 1);
  const uint64_t ctas_needed = (n_items + kGeoThreads / 32 - 1) / (kGeoThreads / 32);   // one item per warp
  return static_cast<uint32_t>(std::min<uint64_t>(ctas_needed, static_cast<uint64_t>(per_sm) * sm_count));
}

static void PrepareGeo(const GeometryArgs& a, cudaStream_t stream) {
  const uint32_t n_tiles = (a.end - a.begin + (1u << a.tile_shift) - 1) >> a.tile_shift;
  cudaMemsetAsync(a.queue, 0, sizeof(unsigned int), stream);
  cudaMemsetAsync(a.tile_epoch, 0, sizeof(unsigned int) * n_tiles, stream);
}

template <typename Kernel>
static void LaunchGeo(Kernel kernel, GeometryArgs a, int sm_count, cudaStream_t stream) {
  const uint32_t grid = GeoGrid(kernel, &a, sm_count);
  PrepareGeo(a, stream);
  kernel<<<grid, kGeoThreads, kGeoSmemBytes, stream>>>(a);
}

void LaunchActivationAndNormals(const GeometryArgs& a, int sm_count, bool determine_activation, bool update_normals, cudaStream_t stream) {
  if (a.end <= a.begin || (!determine_activation && !update_normals)) return;
  if (a.kf_count <= 0) {
    // no keyframe to look at: activation clears every flag, normals keep their value
    if (determine_activation) cudaMemsetAsync(a.active, 0, a.n, stream);   // (every rank clears its whole replica)
    return;
  }
  if (determine_activation && update_normals) LaunchGeo(ActivationNormalsKernel<true, true>, a, sm_count, stream);
  else if (determine_activation) LaunchGeo(ActivationNormalsKernel<true, false>, a, sm_count, stream);
  else LaunchGeo(ActivationNormalsKernel<false, true>, a, sm_count, stream);
}

void LaunchPositionAndDescriptor(const GeometryArgs& a, int sm_count, cudaStream_t stream) {
  if (a.end <= a.begin || a.kf_count <= 0) return;
  if (a.cam.use_desc) {
    if (a.cam.use_depth) LaunchGeo(PositionDescriptorKernel<true, true>, a, sm_count, stream);
    else LaunchGeo(PositionDescriptorKernel<false, true>, a, sm_count, stream);
  } else {
    LaunchGeo(PositionDescriptorKernel<true, false>, a, sm_count, stream);
  }
}

// ------------------------------------------------------------------------------------------------
// Multi-GPU exchange helpers (the collectives themselves run in the host's NCCL communicator).

__constant__ int kShardRowIds[kShardRows - 1] = {kRowX, kRowY, kRowZ, kRowNormal, kRowD1, kRowD2};

__global__ void __launch_bounds__(256) PackShardKernel(const float* __restrict__ surfels, uint32_t pitch,
                                                       const uint8_t* __restrict__ active, uint32_t n, uint32_t rank, uint32_t world,
                                                       uint32_t shard_len, float* __restrict__ slice) {
  const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;   // local index
  if (c >= shard_len) return;
  const uint32_t i = SurfelShardToGlobal(c, rank, world);
  const bool in = i < n;
#pragma unroll
  for (int r = 0; r < kShardRows - 1; ++r)
    slice[static_cast<size_t>(r) * shard_len + c] = in ? surfels[static_cast<size_t>(kShardRowIds[r]) * pitch + i] : 0.f;
  slice[static_cast<size_t>(kShardRows - 1) * shard_len + c] = in ? static_cast<float>(active[i]) : 0.f;
}

__global__ void __launch_bounds__(256) UnpackShardsKernel(float* __restrict__ surfels, uint32_t pitch, uint8_t* __restrict__ active,
                                                          uint32_t n, uint32_t shard_len, uint32_t world, int skip_rank,
                                                          const float* __restrict__ buffer) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;   // global index
  if (i >= n) return;
  const uint32_t granule = i >> kShardGranuleShift;
  const uint32_t rank = granule % world;
  if (static_cast<int>(rank) == skip_rank) return;
  const uint32_t c = ((granule / world) << kShardGranuleShift) | (i & ((1u << kShardGranuleShift) - 1u));
  const float* slice = buffer + static_cast<size_t>(rank) * kShardRows * shard_len;
#pragma unroll
  for (int r = 0; r < kShardRows - 1; ++r)
    surfels[static_cast<size_t>(kShardRowIds[r]) * pitch + i] = slice[static_cast<size_t>(r) * shard_len + c];
  active[i] = static_cast<uint8_t>(slice[static_cast<size_t>(kShardRows - 1) * shard_len + c]);
}

void LaunchPackShard(const float* surfels, uint32_t pitch, const uint8_t* active, uint32_t n, uint32_t rank, uint32_t world,
                     uint32_t shard_len, float* slice, cudaStream_t stream) {
  if (shard_len == 0) return;
  PackShardKernel<<<(shard_len + 255) / 256, 256, 0, stream>>>(surfels, pitch, active, n, rank, world, shard_len, slice);
}

void LaunchUnpackShards(float* surfels, uint32_t pitch, uint8_t* active, uint32_t n, uint32_t shard_len, int world, int skip_rank,
                        const float* buffer, cudaStream_t stream) {
  if (n == 0) return;
  UnpackShardsKernel<<<(n + 255) / 256, 256, 0, stream>>>(surfels, pitch, active, n, shard_len, static_cast<uint32_t>(world), skip_rank, buffer);
}

__global__ void PackPoseResultsKernel(const int* __restrict__ ids, int n, const float* __restrict__ pose_est,
                                      const int* __restrict__ iterations, const int* __restrict__ converged,
                                      const double* __restrict__ first_stats, float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int kf = ids[i];
  float* o = out + static_cast<size_t>(kf) * kPoseSlot;
  for (int j = 0; j < 7; ++j) o[j] = pose_est[kf * 7 + j];
  o[7] = static_cast<float>(iterations[kf]);
  o[8] = static_cast<float>(converged[kf]);
  for (int j = 0; j < 8; ++j) o[9 + j] = static_cast<float>(first_stats[kf * 8 + j]);
}

void LaunchPackPoseResults(const int* ids, int n, const float* pose_est, const int* iterations, const int* converged,
                           const double* first_stats, float* out, cudaStream_t stream) {
  if (n <= 0) return;
  PackPoseResultsKernel<<<(n + 127) / 128, 128, 0, stream>>>(ids, n, pose_est, iterations, converged, first_stats, out);
}

// ------------------------------------------------------------------------------------------------
// uchar4 (.w = luma, cuda_image_processing.cu:165-176) -> dense u8 luma plane.  128-bit loads: 4 pixels per thread.

__global__ void __launch_bounds__(256) ExtractLumaKernel(const uint8_t* __restrict__ rgba, size_t rgba_pitch,
                                                         uint8_t* __restrict__ luma, size_t luma_pitch, int w, int h) {
  const int x4 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
  const int y = blockIdx.y;
  if (x4 >= w || y >= h) return;
  const uint8_t* src = rgba + static_cast<size_t>(y) * rgba_pitch + static_cast<size_t>(x4) * 4;
  uint8_t* dst = luma + static_cast<size_t>(y) * luma_pitch + x4;
  if (x4 + 3 < w && (reinterpret_cast<uintptr_t>(src) & 15) == 0 && (reinterpret_cast<uintptr_t>(dst) & 3) == 0) {
    const uint4 v = __ldg(reinterpret_cast<const uint4*>(src));
    const uint32_t packed = (v.x >> 24) | ((v.y >> 24) << 8) | ((v.z >> 24) << 16) | ((v.w >> 24) << 24);
    *reinterpret_cast<uint32_t*>(dst) = packed;
  } else {
    for (int k = 0; k < 4 && x4 + k < w; ++k) dst[k] = src[4 * k + 3];
  }
}

void LaunchExtractLuma(const uint8_t* rgba, size_t rgba_pitch, uint8_t* luma, size_t luma_pitch, int w, int h, cudaStream_t stream) {
  dim3 block(256);
  dim3 grid((w / 4 + 255) / 256 + 1, h);
  ExtractLumaKernel<<<grid, block, 0, stream>>>(rgba, rgba_pitch, luma, luma_pitch, w, h);
}

}  // namespace bba
