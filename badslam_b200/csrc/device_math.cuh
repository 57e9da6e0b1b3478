// device_math.cuh -- device-side surfel/keyframe maths of libbadba_b200 (sm_100a).
//
// What is computed follows the reference's device headers (cited per function, paths relative to
// /root/reference/applications/badslam/src/badslam/); how it is computed is our own: keyframe
// parameters live in one 96-byte record, images are addressed through raw pitched pointers with
// read-only (ld.global.nc) gathers, the luma plane is a single-channel u8 texture, and all
// association stages are expressed as early-outs that report which stage was reached (for the
// algorithmic-bytes counters of SURVEY.md 8d).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace bba {

// cost_function.cuh:44-52,105-109,126 ; kernels.cuh:38-58
constexpr float kDepthTukey = 10.f;
constexpr float kDepthUncertaintyFactor = 0.1f;
constexpr float kDescWeight = 1e-2f;
constexpr float kDescHuber = 10.f;
constexpr float kTangentScaling = 2.0f;
constexpr uint16_t kInvalidDepthBit = 0x8000u;
constexpr float kCosNormalCompat = 0.76604f;
constexpr uint8_t kSurfelActiveFlag = 1u;

// kernels.cuh:69-93
enum SurfelRow { kRowX = 0, kRowY, kRowZ, kRowNormal, kRowRadiusSq, kRowColor, kRowD1, kRowD2, kRowAccum0 };
constexpr int kSurfelRowCount = 17;

// Camera / depth model shared by all keyframes (surfel_projection.h:42-124 builders, DepthParameters
// surfel_projection.cuh:134-156).  Passed to kernels by value.
struct CameraParams {
  int w, h, cw, ch;
  float fx, fy, cx, cy;                  // depth PixelCornerProjector
  float fx_inv, fy_inv, cx_inv, cy_inv;  // depth PixelCenterUnprojector
  float d2c_fx, d2c_fy, d2c_cx, d2c_cy;  // DepthToColorPixelCorner
  float cfx, cfy, ccx, ccy;              // colour PixelCornerProjector (PixelCenterProjector shares fx, fy)
  float a, raw_to_float, baseline_fx;
  int cell, cf_w;
  unsigned int cell_magic;               // ceil(2^32 / cell): n / cell == __umulhi(n, cell_magic) for n, cell < 2^16 (cell > 1)
  const float* __restrict__ cfactor;     // dense [cf_h][cf_w]
  int use_depth, use_desc;
};

// One keyframe as the kernels see it (Keyframe members keyframe.h:160-237).
struct __align__(16) KfDevice {
  float T[12];                       // frame_T_global, row-major 3x4
  const uint16_t* depth;             // pitched u16
  const uint16_t* normals;           // pitched u16
  cudaTextureObject_t tex;           // u8 luma CUDA array (gather-enabled): linear filter, normalized float, clamp
  uint32_t depth_pitch, normals_pitch;   // bytes
  int activation;
  int pad;
};
static_assert(sizeof(KfDevice) == 96, "KfDevice layout");

struct Vec3 {
  float x, y, z;
};
__device__ __forceinline__ Vec3 V3(float x, float y, float z) { return Vec3{x, y, z}; }
__device__ __forceinline__ float Dot(const Vec3& a, const Vec3& b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
__device__ __forceinline__ Vec3 operator-(const Vec3& a, const Vec3& b) { return V3(a.x - b.x, a.y - b.y, a.z - b.z); }
__device__ __forceinline__ Vec3 operator+(const Vec3& a, const Vec3& b) { return V3(a.x + b.x, a.y + b.y, a.z + b.z); }
__device__ __forceinline__ Vec3 operator*(float s, const Vec3& a) { return V3(s * a.x, s * a.y, s * a.z); }
__device__ __forceinline__ Vec3 Cross(const Vec3& a, const Vec3& b) {   // cuda_util.cuh:76-80
  return V3(a.y * b.z - b.y * a.z, b.x * a.z - a.x * b.z, a.x * b.y - b.x * a.y);
}
__device__ __forceinline__ Vec3 Rotate(const float* __restrict__ T, const Vec3& p) {   // cuda_matrix.cuh:126-135
  return V3(T[0] * p.x + T[1] * p.y + T[2] * p.z, T[4] * p.x + T[5] * p.y + T[6] * p.z,
            T[8] * p.x + T[9] * p.y + T[10] * p.z);
}
__device__ __forceinline__ Vec3 Transform(const float* __restrict__ T, const Vec3& p) {   // cuda_matrix.cuh:104-112
  return V3(T[0] * p.x + T[1] * p.y + T[2] * p.z + T[3], T[4] * p.x + T[5] * p.y + T[6] * p.z + T[7],
            T[8] * p.x + T[9] * p.y + T[10] * p.z + T[11]);
}

// Sums acc[i] over the 32 lanes of the warp for all 32 i at once: after the call lane L holds the total of
// acc[L].  16+8+4+2+1 = 31 shuffles instead of 32 x 5.
__device__ __forceinline__ float WarpTransposeReduce(float (&v)[32], int lane) {
#pragma unroll
  for (int half = 16; half >= 1; half >>= 1) {
    const bool upper = (lane & half) != 0;
#pragma unroll
    for (int i = 0; i < half; ++i) {
      const float lo = v[i], hi = v[i + half];
      const float send = upper ? lo : hi;
      const float keep = upper ? hi : lo;
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, half);
    }
  }
  return v[0];
}

// robust_weighting.cuh:39-86
__device__ __forceinline__ float TukeyResidual(float r, float p) {
  if (fabsf(r) < p) {
    const float q = r / p, t = 1.f - q * q;
    return (1 / 6.f) * p * p * (1 - t * t * t);
  }
  return (1 / 6.f) * p * p;
}
__device__ __forceinline__ float TukeyWeight(float r, float p) {
  if (fabsf(r) < p) {
    const float q = r / p, t = 1.f - q * q;
    return t * t;
  }
  return 0.f;
}
__device__ __forceinline__ float HuberResidual(float r, float p) {
  const float a = fabsf(r);
  return (a < p) ? 0.5f * r * r : p * (a - 0.5f * p);
}
__device__ __forceinline__ float HuberWeight(float r, float p) {
  const float a = fabsf(r);
  return (a < p) ? 1.f : (p / a);
}
// cost_function.cuh:91-98,177-185 (kDepthResidualWeight = 1)
__device__ __forceinline__ float DepthWeight(float r) { return TukeyWeight(r, kDepthTukey); }
__device__ __forceinline__ float DepthCost(float r) { return TukeyResidual(r, kDepthTukey); }
__device__ __forceinline__ float DescWeight(float r) { return kDescWeight * HuberWeight(r, kDescHuber); }
__device__ __forceinline__ float DescCost(float r) { return kDescWeight * HuberResidual(r, kDescHuber); }

// util_nvcc_only.cuh:67-95 (10-bit signed pack / unpack, normal re-normalised after unpack)
__device__ __forceinline__ float S10ToFloat(uint32_t v) {
  // sign-extend the low 10 bits
  const int s = (static_cast<int>(v << 22)) >> 22;
  return s * (1.0f / 511);
}
__device__ __forceinline__ Vec3 UnpackNormal(uint32_t v) {
  Vec3 n = V3(S10ToFloat(v), S10ToFloat(v >> 10), S10ToFloat(v >> 20));
  const float f = 1.0f / sqrtf(Dot(n, n));
  return f * n;
}
__device__ __forceinline__ uint32_t FloatToS10(float v) {
  return 0x03ffu & static_cast<uint16_t>(static_cast<int16_t>(v * 511 + ((v > 0) ? 0.5f : -0.5f)));
}
__device__ __forceinline__ uint32_t PackNormal(const Vec3& n) {
  return FloatToS10(n.x) | (FloatToS10(n.y) << 10) | (FloatToS10(n.z) << 20);
}
// util.cuh:126-146
__device__ __forceinline__ Vec3 U16ToImageSpaceNormal(uint16_t v) {
  Vec3 r;
  r.x = static_cast<int8_t>(v & 0x00ff) * (1.0f / 127);
  r.y = static_cast<int8_t>(v >> 8) * (1.0f / 127);
  const float z = 1 - r.x * r.x - r.y * r.y;
  r.z = -sqrtf((z > 0.f) ? z : 0.f);
  return r;
}
// util.cuh:62-69
__device__ __forceinline__ float RawToCalibratedDepth(float a, float cfactor, float raw_to_float, uint16_t measured) {
  const float inv_depth = 1.0f / (raw_to_float * measured);
  return 1.f / (inv_depth + cfactor * expf(-a * inv_depth));
}

__device__ __forceinline__ uint16_t LoadPixelU16(const uint16_t* base, uint32_t pitch, int px, int py) {
  return __ldg(reinterpret_cast<const uint16_t*>(reinterpret_cast<const char*>(base) + static_cast<size_t>(py) * pitch) + px);
}
// The same read-only loads as `asm volatile`: the compiler must issue them where they are written.  Plain __ldg()s of the
// pixel's depth / normal / cfactor get SUNK below the association's early-outs (seen in the SASS of the geometry kernels: depth,
// then -- after the valid-depth branch -- cfactor, then -- after the depth tests -- the normal: three serial L2 round trips per
// pair instead of one).
__device__ __forceinline__ uint16_t LoadU16Now(const uint16_t* p) {
  uint16_t v;
  asm volatile("ld.global.nc.u16 %0, [%1];" : "=h"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ float LoadF32Now(const float* p) {
  float v;
  asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}

// Result of projecting one surfel into one keyframe.
struct Assoc {
  Vec3 lp;      // surfel position in the keyframe frame
  Vec3 ln;      // surfel normal rotated into the keyframe frame
  float d;      // calibrated depth of the pixel
  float nx, ny; // unprojector ray of the pixel
  int px, py;
  float pxf, pyf;
  uint16_t kf_normal;
};

// Projection + association, split into three steps so that callers can put ALL gathers of a (surfel, keyframe) pair in
// flight before the first dependent use (the association tests are cheap; the latency of the depth -> normal -> texture
// chain is what the reference's early-outs serialise).
// surfel_projection_nvcc_only.cuh:48-127,332-359 ; util.cuh:83-118 ; cuda_matrix.cuh:115-124 ; cost_function.cuh:81-83

// Step A: project into the depth image.  No memory access.  Returns false if behind the camera or outside the image.
__device__ __forceinline__ bool ProjectIntoImage(const CameraParams& cam, const float* __restrict__ T, const Vec3& gp, Assoc* r) {
  r->lp.z = T[8] * gp.x + T[9] * gp.y + T[10] * gp.z + T[11];
  if (r->lp.z <= 0.f) return false;
  r->lp.x = T[0] * gp.x + T[1] * gp.y + T[2] * gp.z + T[3];
  r->lp.y = T[4] * gp.x + T[5] * gp.y + T[6] * gp.z + T[7];
  const float inv_z = 1.0f / r->lp.z;
  r->pxf = cam.fx * (r->lp.x * inv_z) + cam.cx;
  r->pyf = cam.fy * (r->lp.y * inv_z) + cam.cy;
  // float -> int conversion saturates on the device, so the reference's bounds test is safe as is
  r->px = static_cast<int>(r->pxf);
  r->py = static_cast<int>(r->pyf);
  return (r->pxf >= 0.f) && (r->pyf >= 0.f) && r->px < cam.w && r->py < cam.h;
}

// Step B: the three independent gathers of the pixel the surfel projects to.  The keyframe normal is fetched together
// with the depth (the reference reads it only after the depth and facing tests passed; ~99 % of in-image pairs do).
struct PixelLoads {
  uint16_t measured;
  uint16_t kf_normal;
  float cf;
};
__device__ __forceinline__ PixelLoads LoadPixel(const CameraParams& cam, const uint16_t* __restrict__ depth, uint32_t depth_pitch,
                                                const uint16_t* __restrict__ normals, uint32_t normals_pitch, const Assoc& r) {
  PixelLoads l;
  l.measured = LoadU16Now(reinterpret_cast<const uint16_t*>(reinterpret_cast<const char*>(depth) + static_cast<size_t>(r.py) * depth_pitch) + r.px);
  l.kf_normal = LoadU16Now(reinterpret_cast<const uint16_t*>(reinterpret_cast<const char*>(normals) + static_cast<size_t>(r.py) * normals_pitch) + r.px);
  // sparse cell of the pixel: exact integer division by multiplication with a precomputed reciprocal
  const unsigned int cell_x = (cam.cell == 1) ? static_cast<unsigned int>(r.px) : __umulhi(static_cast<unsigned int>(r.px), cam.cell_magic);
  const unsigned int cell_y = (cam.cell == 1) ? static_cast<unsigned int>(r.py) : __umulhi(static_cast<unsigned int>(r.py), cam.cell_magic);
  l.cf = LoadF32Now(cam.cfactor + cell_y * cam.cf_w + cell_x);
  return l;
}

// Step C: the association tests.  Returns the stage reached: 1 in image only, 2 passed valid-depth + depth-threshold +
// facing tests, 3 associated.
__device__ __forceinline__ int Associate(const CameraParams& cam, const float* __restrict__ T, const Vec3& n, const PixelLoads& l,
                                         Assoc* r) {
  // Written without early returns: every test is evaluated and the stage selected at the end, so that all three loaded values
  // are consumed unconditionally.  With the reference's chain of early-outs the compiler sinks each load below the previous
  // test (three serial L2 round trips per pair); ~99 % of the in-image pairs pass every test anyway.  The predicates are the
  // reference's, including how they treat NaN (a comparison with NaN is false = "test passed", as in its `if (...) return`).
  const bool invalid = (l.measured & kInvalidDepthBit) != 0;
  r->d = RawToCalibratedDepth(cam.a, l.cf, cam.raw_to_float, l.measured);
  r->ln = Rotate(T, n);
  r->nx = cam.fx_inv * r->px + cam.cx_inv;
  r->ny = cam.fy_inv * r->py + cam.cy_inv;
  const float stddev =
      (kDepthUncertaintyFactor * fabsf(r->ln.x * r->nx + r->ln.y * r->ny + r->ln.z) * (r->d * r->d)) / cam.baseline_fx;
  const bool too_far = fabsf(r->lp.z - r->d) > kDepthTukey * stddev;
  // The reference tests (1 / |lp|) * dot(lp, ln) > 0 (surfel_projection_nvcc_only.cuh:104-108); for the finite,
  // positive |lp| of a point in front of the camera that is the sign of the dot product alone.
  const bool back_facing = Dot(r->lp, r->ln) > 0;
  r->kf_normal = l.kf_normal;
  const bool incompatible = Dot(r->ln, U16ToImageSpaceNormal(l.kf_normal)) < kCosNormalCompat;
  return (invalid | too_far | back_facing) ? 1 : (incompatible ? 2 : 3);
}

// All three steps.  Returns 0 culled / outside, else the stage of Associate().
__device__ __forceinline__ int ProjectAssociate(const CameraParams& cam, const float* __restrict__ T,
                                                const uint16_t* __restrict__ depth, uint32_t depth_pitch,
                                                const uint16_t* __restrict__ normals, uint32_t normals_pitch,
                                                const Vec3& gp, const Vec3& n, Assoc* r) {
  if (!ProjectIntoImage(cam, T, gp, r)) return 0;
  const PixelLoads l = LoadPixel(cam, depth, depth_pitch, normals, normals_pitch, *r);
  return Associate(cam, T, n, l, r);
}

// surfel_projection.cuh:196-207
__device__ __forceinline__ bool DepthToColor(const CameraParams& cam, float pxf, float pyf, float* cx, float* cy) {
  *cx = cam.d2c_fx * pxf + cam.d2c_cx;
  *cy = cam.d2c_fy * pyf + cam.d2c_cy;
  return *cx >= 0 && *cy >= 0 && static_cast<int>(*cx) < cam.cw && static_cast<int>(*cy) < cam.ch;
}

// cost_function.cuh:56-88 + kernel_opt_pose.cu:45-94 (inv_stddev, unprojected pixel point, raw residual)
__device__ __forceinline__ float DepthResidual(const CameraParams& cam, const Assoc& r, float* inv_stddev, Vec3* unproj) {
  *inv_stddev = cam.baseline_fx / (kDepthUncertaintyFactor * fabsf(r.ln.x * r.nx + r.ln.y * r.ny + r.ln.z) * (r.d * r.d));
  *unproj = V3(r.d * r.nx, r.d * r.ny, r.d);
  return *inv_stddev * Dot(r.ln, *unproj - r.lp);
}

// cost_function.cuh:115-136
__device__ __forceinline__ void TangentProjections(const CameraParams& cam, const float* __restrict__ T, const Vec3& gp,
                                                   const Vec3& n, float radius_sq, float* t1x, float* t1y, float* t2x,
                                                   float* t2y) {
  Vec3 t1 = Cross(n, (fabsf(n.x) > 0.9f) ? V3(0, 1, 0) : V3(1, 0, 0));
  t1 = (kTangentScaling * sqrtf(radius_sq / fmaxf(1e-12f, Dot(t1, t1)))) * t1;
  const Vec3 p1 = Transform(T, gp + t1);
  *t1x = cam.cfx * (p1.x / p1.z) + cam.ccx;
  *t1y = cam.cfy * (p1.y / p1.z) + cam.ccy;
  Vec3 t2 = Cross(n, t1);
  t2 = (kTangentScaling * sqrtf(radius_sq / fmaxf(1e-12f, Dot(t2, t2)))) * t2;
  const Vec3 p2 = Transform(T, gp + t2);
  *t2x = cam.cfx * (p2.x / p2.z) + cam.ccx;
  *t2y = cam.cfy * (p2.y / p2.z) + cam.ccy;
}


// The pose-independent half of ComputeTangentProjections (cost_function.cuh:115-133): the two tangent points gp + t1, gp + t2 of
// a surfel.  Same expressions as TangentProjections above (the pose kernel reads them precomputed per surfel, see
// SurfelFramesKernel; only Transform + projection depend on the keyframe).
__device__ __forceinline__ void TangentPoints(const Vec3& gp, const Vec3& n, float radius_sq, Vec3* q1, Vec3* q2) {
  Vec3 t1 = Cross(n, (fabsf(n.x) > 0.9f) ? V3(0, 1, 0) : V3(1, 0, 0));
  t1 = (kTangentScaling * sqrtf(radius_sq / fmaxf(1e-12f, Dot(t1, t1)))) * t1;
  *q1 = gp + t1;
  Vec3 t2 = Cross(n, t1);
  t2 = (kTangentScaling * sqrtf(radius_sq / fmaxf(1e-12f, Dot(t2, t2)))) * t2;
  *q2 = gp + t2;
}
__device__ __forceinline__ void ProjectTangentPoints(const CameraParams& cam, const float* __restrict__ T, const Vec3& q1, const Vec3& q2,
                                                     float* t1x, float* t1y, float* t2x, float* t2y) {
  const Vec3 p1 = Transform(T, q1);
  *t1x = cam.cfx * (p1.x / p1.z) + cam.ccx;
  *t1y = cam.cfy * (p1.y / p1.z) + cam.ccy;
  const Vec3 p2 = Transform(T, q2);
  *t2x = cam.cfx * (p2.x / p2.z) + cam.ccx;
  *t2y = cam.cfy * (p2.y / p2.z) + cam.ccy;
}

// One sample point of the descriptor residual: the bilinearly filtered intensity at (x, y)
// (ComputeRawDescriptorResidual, cost_function.cuh:140-156) and the finite-difference gradient built from the
// four texels around it (DescriptorJacobianWrtProjectedPosition, cost_function.cuh:191-254).
// The reference reads those four texels with four point fetches at (ix+0.5|1.5, iy+0.5|1.5); here ONE
// tex2Dgather centred on the 2x2 footprint returns exactly the same four (clamped) texels:
// .w = (ix, iy) top-left, .z = (ix+1, iy) top-right, .x = (ix, iy+1) bottom-left, .y = (ix+1, iy+1) bottom-right.
__device__ __forceinline__ void SamplePoint(cudaTextureObject_t tex, float x, float y, float* intensity, float* dx, float* dy) {
  // ix = int(max(0, x - 0.5)), tx = clamp(x - 0.5 - ix, 0, 1) of the reference, without leaving the float domain:
  // xm >= 0, fx = floor(xm) = float(ix), tx = xm - fx in [0, 1) (and 0 where the reference's clamp bites, x < 0.5).
  const float xm = fmaxf(0.f, x - 0.5f), ym = fmaxf(0.f, y - 0.5f);
  const float fx = floorf(xm), fy = floorf(ym);
  const float tx = xm - fx, ty = ym - fy;
  const float4 g = tex2Dgather<float4>(tex, fx + 1.0f, fy + 1.0f, 0);
  *intensity = tex2D<float>(tex, x, y);
  *dx = (g.y - g.x) * ty + (g.z - g.w) * (1 - ty);
  *dy = (g.y - g.z) * tx + (g.x - g.w) * (1 - tx);
}

struct DescEval {
  float r1, r2;              // raw residuals (cost_function.cuh:140-156)
  float gx1, gy1, gx2, gy2;  // gradients wrt the projected position (cost_function.cuh:250-253)
};

__device__ __forceinline__ void EvalDescriptor(cudaTextureObject_t tex, float cx, float cy, float t1x, float t1y, float t2x,
                                               float t2y, float d1, float d2, DescEval* e) {
  float intensity, t1i, t2i, cdx, cdy, t1dx, t1dy, t2dx, t2dy;
  SamplePoint(tex, cx, cy, &intensity, &cdx, &cdy);
  SamplePoint(tex, t1x, t1y, &t1i, &t1dx, &t1dy);
  SamplePoint(tex, t2x, t2y, &t2i, &t2dx, &t2dy);
  e->r1 = (180.f * (t1i - intensity)) - d1;
  e->r2 = (180.f * (t2i - intensity)) - d2;
  e->gx1 = 180.f * (t1dx - cdx);
  e->gy1 = 180.f * (t1dy - cdy);
  e->gx2 = 180.f * (t2dx - cdx);
  e->gy2 = 180.f * (t2dy - cdy);
}

// kernel_opt_pose.cu:96-142: Jacobian of a descriptor residual wrt the pose (global_T_frame * exp(hat(delta))).
__device__ __forceinline__ void DescPoseJacobian(const CameraParams& cam, const Vec3& ls, float gx, float gy, float (&J)[6]) {
  gx *= cam.cfx;
  gy *= cam.cfy;
  const float inv_z = 1.f / ls.z, z_sq = ls.z * ls.z, inv_z_sq = inv_z * inv_z, xy = ls.x * ls.y;
  J[0] = -gx * inv_z;
  J[1] = -gy * inv_z;
  J[2] = (ls.x * gx + ls.y * gy) * inv_z_sq;
  J[3] = ((ls.y * ls.y + z_sq) * gy + xy * gx) * inv_z_sq;
  J[4] = -((ls.x * ls.x + z_sq) * gx + xy * gy) * inv_z_sq;
  J[5] = -(ls.x * gy - ls.y * gx) * inv_z;
}

}  // namespace bba
