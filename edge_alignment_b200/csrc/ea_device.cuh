// Device-side data structures and the per-point evaluation shared by every kernel of the
// pose-solve path.  sm_100a only.
//
// Per-point math replaces, fused:
//   EAResidue::operator()<Jet<double,7>>      standalone/utils.h:48-80
//   ceres::BiCubicInterpolator::Evaluate      (Ceres, cubic_interpolation.h; see oracle/)
//   AutoDiff + QuaternionParameterization     standalone/utils.h:87, standalone_edge_align.cpp:277
//   LossFunction + Corrector                  standalone_edge_align.cpp:272
// Precision plan (DESIGN.md "Numerics"): pose transform + projection + fractional pixel offsets
// in fp64 (B200 keeps a 1:2 fp64 pipe), bicubic + analytic 1x6 Jacobian in fp32, normal
// equations reduced by warp butterflies in fp32 and accumulated in fp64.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <cstring>

#include "ea_cabi.h"

#define EA_WARP 32
#define EA_NSUM 32  // butterfly slots: 0..20 upper-tri J^T J, 21..26 J^T r, 27 #failed, 28..31 unused
#define EA_SUMS 29  // reduced totals: [0..20] H upper-tri, [21..26] b, [27] #failed, [28] cost

struct EaLevelDesc {   // one per (slot, level); lives in device memory
  const void* pts;     // point stream, see EaPtStream (EA_POINTS_PIXEL: 8 B packed {u | v << 16, raw depth}; EA_POINTS_XYZ: float4 {X,Y,Z,1})
  const int* n_pts;    // device-resident count (written by the compaction kernel)
  const float* dt;     // raw distance transform (pixels), f32: pixel (0,0) of a replicate-padded image, see EA_DT_PAD
  const float2* dt_affine;  // {scale, shift} of cv::normalize(MINMAX): sampled value = raw * scale + shift
  int w, h;
  int pts_mode, dt_pitch;   // dt_pitch = ea_dt_pitch(w), floats per padded row
  const int* truncated;     // device flag: the point list was cut at its capacity (written by the compaction kernel)
};

// Distance transforms live in HBM with a replicated border of EA_DT_PAD pixels on every side: rows -4 .. h+3 and
// columns -4 .. w+3 hold the value of the nearest image pixel, which IS ceres::Grid2D::GetValue's clamp-to-edge.  With
// floor(u'), floor(v') clamped to [-3, w+1] x [-3, h+1] the 4x4 footprint of BiCubicInterpolator::Evaluate always lies
// inside the padded image and reads exactly the values the clamped reference would read (a footprint further out sees
// one constant either way) -- no per-texel clamps, no border path in the gather.
#define EA_DT_PAD 4
__host__ __device__ __forceinline__ int ea_dt_pitch(int w) { return (w + 2 * EA_DT_PAD + 3) & ~3; }
__host__ __device__ __forceinline__ size_t ea_dt_slot_floats(int w, int h) { return size_t(ea_dt_pitch(w)) * size_t(h + 2 * EA_DT_PAD); }
__host__ __device__ __forceinline__ size_t ea_dt_origin_offset(int w) { return size_t(EA_DT_PAD) * ea_dt_pitch(w) + EA_DT_PAD; }

struct EaLevelGeom {   // per level, identical for every slot of a frameset (kernel parameter => constant bank)
  double fx, fy, cx, cy;
  double inv_fx, inv_fy;
  int w, h;
};

struct EaPose {  // per-evaluation uniform transform, fp64
  // q = s * (A * a) + tt with A = K_now * R * B, tt = K_now * t; (u', v') = (q0, q1) / q2, z' = q2.
  //   EA_POINTS_PIXEL: a = (u, v, 1), s = Z = raw depth / depth_scale, B = K_ref^-1 (back-projection utils.cpp:235-237)
  //   EA_POINTS_XYZ:   a = (X, Y, Z), s = 1, B = I
  double A[9];
  double tt[3];
  float m2t[3];      // -2 t, for 2 (R X) = 2 p' - 2 t in the Jacobian
  float fx, fy, inv_fx, inv_fy;   // now-level intrinsics in fp32 (Jacobian)
  float cx, cy;      // now-level principal point (only the Jacobian's lever arm u' - cx uses it: fp32)
};

// Eigen::Quaternion::toRotationMatrix(), as called at standalone/utils.h:51-53 (no normalisation), folded with the
// intrinsics of the reference level (back-projection) and of the now level (projection, utils.h:74-75).
template <bool XYZ>
__device__ __forceinline__ void ea_pose_setup(const double* x7, const EaLevelGeom& ref, const EaLevelGeom& now, EaPose& P) {
  const double qw = x7[0], qx = x7[1], qy = x7[2], qz = x7[3];
  const double tx = 2.0 * qx, ty = 2.0 * qy, tz = 2.0 * qz;
  const double twx = tx * qw, twy = ty * qw, twz = tz * qw;
  const double txx = tx * qx, txy = ty * qx, txz = tz * qx;
  const double tyy = ty * qy, tyz = tz * qy, tzz = tz * qz;
  double R[9];
  R[0] = 1.0 - (tyy + tzz); R[1] = txy - twz;         R[2] = txz + twy;
  R[3] = txy + twz;         R[4] = 1.0 - (txx + tzz); R[5] = tyz - twx;
  R[6] = txz - twy;         R[7] = tyz + twx;         R[8] = 1.0 - (txx + tyy);
  double M[9];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    if (XYZ) { M[3 * i] = R[3 * i]; M[3 * i + 1] = R[3 * i + 1]; M[3 * i + 2] = R[3 * i + 2]; }
    else {
      M[3 * i] = R[3 * i] * ref.inv_fx;
      M[3 * i + 1] = R[3 * i + 1] * ref.inv_fy;
      M[3 * i + 2] = R[3 * i + 2] - ref.cx * M[3 * i] - ref.cy * M[3 * i + 1];
    }
  }
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    P.A[j] = now.fx * M[j] + now.cx * M[6 + j];
    P.A[3 + j] = now.fy * M[3 + j] + now.cy * M[6 + j];
    P.A[6 + j] = M[6 + j];
  }
  P.tt[0] = now.fx * x7[4] + now.cx * x7[6];
  P.tt[1] = now.fy * x7[5] + now.cy * x7[6];
  P.tt[2] = x7[6];
  P.m2t[0] = -2.0f * float(x7[4]); P.m2t[1] = -2.0f * float(x7[5]); P.m2t[2] = -2.0f * float(x7[6]);
  P.fx = float(now.fx); P.fy = float(now.fy); P.inv_fx = float(now.inv_fx); P.inv_fy = float(now.inv_fy);
  P.cx = float(now.cx); P.cy = float(now.cy);
}

struct EaPointEval {
  float f, gu, gv;         // normalised bicubic value; gradient of the raw (pixel-unit) field (grid row == u, col == v: SEA:258)
  float ub, vb;            // u' - cx, v' - cy
  float pz, iz;            // z' and 1/z'
  bool fail;               // |z'| < 0.01  (utils.h:70-73)
};

// ceres CubicHermiteSpline<1> (Catmull-Rom), fp32, with the 1/2 factors pulled out of the coefficients:
//   a2 = -p0 + 3 p1 - 3 p2 + p3,  b2 = 2 p0 - 5 p1 + 4 p2 - p3,  c2 = p2 - p0
//   f = p1 + (x/2) (c2 + x (b2 + x a2)),   f' = c2/2 + x (b2 + (3x/2) a2)
// hx = x/2 and x15 = 3x/2 are shared by all splines evaluated at the same x.
__device__ __forceinline__ void ea_cubic(float p0, float p1, float p2, float p3, float x, float hx, float x15, float& f, float& dfdx) {
  const float a2 = fmaf(3.0f, p1 - p2, p3 - p0);
  const float b2 = fmaf(4.0f, p2, fmaf(-5.0f, p1, fmaf(2.0f, p0, -p3)));
  const float c2 = p2 - p0;
  f = fmaf(hx, fmaf(x, fmaf(x, a2, b2), c2), p1);
  dfdx = fmaf(x, fmaf(x15, a2, b2), 0.5f * c2);
}
__device__ __forceinline__ float ea_cubic_val(float p0, float p1, float p2, float p3, float x, float hx) {
  const float a2 = fmaf(3.0f, p1 - p2, p3 - p0);
  const float b2 = fmaf(4.0f, p2, fmaf(-5.0f, p1, fmaf(2.0f, p0, -p3)));
  const float c2 = p2 - p0;
  return fmaf(hx, fmaf(x, fmaf(x, a2, b2), c2), p1);
}

// floor(x) and x - floor(x), exact for |x| < 2^31, on the fp64 pipe alone: x + (2^52 + 2^51) rounded DOWN is that constant plus
// floor(x), whose low mantissa word is floor(x) in two's complement (DADD.RM, DADD, DADD and one narrowing -- the F2I / I2F pair
// it replaces runs on the quarter-rate conversion unit, four of them per point).  Wild values (only possible when the z-guard
// has already failed the evaluation) give unspecified indices, which the caller clamps.
__device__ __forceinline__ void ea_floor_frac(double x, int& i, float& frac) {
  const double magic = 6755399441055744.0;
  const double t = __dadd_rd(x, magic);
  i = __double2loint(t);
  frac = float(x - (t - magic));
}
// 1 / x to within an ulp or two: hardware seed (2^-23) and one cubically convergent correction, r (1 + e + e^2) with e = 1 - x r.
// No slow path: zero, infinite and denormal x give inf / NaN, which only a failed evaluation can meet.
__device__ __forceinline__ double ea_rcp64(double x) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  double e = fma(-x, r, 1.0);
  e = fma(e, e, e);
  return fma(r, e, r);
}

// Point stream element.  Pixel points are 8 bytes: integer pixel coordinates (images up to 65535 px a side) and the raw
// depth as f32 (exact for u16 and f32 depth maps) -- half the bytes of a float4 per evaluation, and no dead load
// component for the register allocator to recycle while the prefetch is still in flight.
template <bool XYZ> struct EaPtStream;
template <> struct EaPtStream<false> {
  typedef uint2 T;
  static __device__ __forceinline__ T load(const void* base, size_t i) { return __ldg(reinterpret_cast<const uint2*>(base) + i); }
  static __device__ __forceinline__ T pad() { return make_uint2(0u, 0x3f800000u); }
  static __device__ __forceinline__ void unpack(const T r, double& a0, double& a1, double& a2) {
    a0 = double(int(r.x & 0xffffu)); a1 = double(int(r.x >> 16)); a2 = double(__uint_as_float(r.y));
  }
  static __device__ __forceinline__ float4 as_float4(const T r) {
    return make_float4(float(r.x & 0xffffu), float(r.x >> 16), __uint_as_float(r.y), 1.0f);
  }
};
template <> struct EaPtStream<true> {
  typedef float4 T;
  static __device__ __forceinline__ T load(const void* base, size_t i) { return __ldg(reinterpret_cast<const float4*>(base) + i); }
  static __device__ __forceinline__ T pad() { return make_float4(0.f, 0.f, 1.f, 0.f); }
  static __device__ __forceinline__ void unpack(const T r, double& a0, double& a1, double& a2) {
    a0 = double(r.x); a1 = double(r.y); a2 = double(r.z);
  }
  static __device__ __forceinline__ float4 as_float4(const T r) { return r; }
};
__host__ __device__ __forceinline__ uint2 ea_pack_pixel_point(unsigned u, unsigned v, float depth) {
  uint2 r; r.x = (u & 0xffffu) | (v << 16);
#ifdef __CUDA_ARCH__
  r.y = __float_as_uint(depth);
#else
  memcpy(&r.y, &depth, 4);
#endif
  return r;
}

// ---- one edge point in three stages: project (fp64) -> gather (16 texels) -> interpolate (fp32) ----------------------
struct EaProj {
  int off;                 // element offset of texel (floor(v') - 1, floor(u') - 1) from texel (-1, -1) of the image: iv * pitch + iu
  float du, dv;            // fractional offsets (from fp64)
  float ub, vb, pz, iz;    // u' - cx, v' - cy, z', 1/z'
  int zm;                  // high word of |z'| - 0.01: negative <=> |z'| < 0.01, the evaluation fails (utils.h:70-73)
};
// (a0, a1, a2) = (u, v, raw depth) or (X, Y, Z)
template <bool XYZ>
__device__ __forceinline__ void ea_project(const double a0, const double a1, const double a2, const int W, const int H, const int pitch,
                                           double inv_depth_scale, const EaPose& P, EaProj& r) {
  double q0, q1, q2;
  if (XYZ) {
    q0 = fma(P.A[0], a0, fma(P.A[1], a1, fma(P.A[2], a2, P.tt[0])));
    q1 = fma(P.A[3], a0, fma(P.A[4], a1, fma(P.A[5], a2, P.tt[1])));
    q2 = fma(P.A[6], a0, fma(P.A[7], a1, fma(P.A[8], a2, P.tt[2])));
  } else {
    const double Z = a2 * inv_depth_scale;
    q0 = fma(Z, fma(P.A[0], a0, fma(P.A[1], a1, P.A[2])), P.tt[0]);
    q1 = fma(Z, fma(P.A[3], a0, fma(P.A[4], a1, P.A[5])), P.tt[1]);
    q2 = fma(Z, fma(P.A[6], a0, fma(P.A[7], a1, P.A[8])), P.tt[2]);
  }
  // the sign of an IEEE difference is exact, so this is q2 < 0.01 && q2 > -0.01 to the last bit; a running integer minimum of
  // it is all the evaluation loop keeps of the z-guard
  r.zm = __double2hiint(fabs(q2) - 0.01);
  const double iz = ea_rcp64(q2);
  const double u = q0 * iz, v = q1 * iz;
  int iu, iv;
  ea_floor_frac(u, iu, r.du);
  ea_floor_frac(v, iv, r.dv);
  // the clamp keeps the 4x4 footprint inside the padded image for any input
  iu = min(max(iu, 1 - EA_DT_PAD), W + 1);
  iv = min(max(iv, 1 - EA_DT_PAD), H + 1);
  r.off = iv * pitch + iu;
  r.ub = float(u) - P.cx; r.vb = float(v) - P.cy;
  r.pz = float(q2); r.iz = float(iz);
}
// The gather base of a padded distance transform whose FIRST element is dt_pad: texel (-1, -1) of the image.
__device__ __forceinline__ const float* ea_gather_base(const float* dt_pad, const int pitch) {
  return dt_pad + size_t(EA_DT_PAD - 1) * size_t(pitch) + (EA_DT_PAD - 1);
}
// t[4 * row + col] = dt(floor(v') - 1 + row, floor(u') - 1 + col) with Grid2D clamp-to-edge (through the padding).
// base = ea_gather_base(...), off = EaProj::off
__device__ __forceinline__ void ea_gather(const float* __restrict__ base, const int off, const int pitch, float (&t)[16]) {
  // one 32-bit element offset per footprint row, widened against the single 64-bit base (IMAD.WIDE), the four columns as
  // immediates: 7 integer instructions for the 16 addresses
  const int o1 = off + pitch, o2 = o1 + pitch, o3 = o2 + pitch;
  const float* p0 = base + off;
  const float* p1 = base + o1;
  const float* p2 = base + o2;
  const float* p3 = base + o3;
  t[0] = __ldg(p0); t[1] = __ldg(p0 + 1); t[2] = __ldg(p0 + 2); t[3] = __ldg(p0 + 3);
  t[4] = __ldg(p1); t[5] = __ldg(p1 + 1); t[6] = __ldg(p1 + 2); t[7] = __ldg(p1 + 3);
  t[8] = __ldg(p2); t[9] = __ldg(p2 + 1); t[10] = __ldg(p2 + 2); t[11] = __ldg(p2 + 3);
  t[12] = __ldg(p3); t[13] = __ldg(p3 + 1); t[14] = __ldg(p3 + 2); t[15] = __ldg(p3 + 3);
}
// BiCubicInterpolator::Evaluate: for each grid row (== image column x_k) spline along c (== image y), then spline the
// four results along r (== image x).  cv::normalize(NORM_MINMAX) is folded in: the interpolant is linear in the texels.
//
// Packed fp32x2 (sm_100 FFMA2 / FADD2 / FMUL2: two IEEE fp32 operations per issued instruction): the four column splines run
// as two pairs, and the two row splines (of the values and of the v-derivatives) as one pair -- the same operations, in the
// same order, with the same roundings as the scalar ea_cubic, in half the issue slots (the evaluation loop is issue-bound).
__device__ __forceinline__ float2 ea_f2(float a, float b) { return make_float2(a, b); }
__device__ __forceinline__ float2 ea_bc(float a) { return make_float2(a, a); }
__device__ __forceinline__ float2 ea_sub2(float2 a, float2 b) { return __fadd2_rn(a, make_float2(-b.x, -b.y)); }
// two ea_cubic at once: value f and derivative d of the Catmull-Rom splines through (p0.x .. p3.x) and (p0.y .. p3.y) at x
__device__ __forceinline__ void ea_cubic2(const float2 p0, const float2 p1, const float2 p2, const float2 p3, const float x, const float hx,
                                          const float x15, float2& f, float2& d) {
  const float2 a2 = __ffma2_rn(ea_bc(3.0f), ea_sub2(p1, p2), ea_sub2(p3, p0));
  const float2 b2 = __ffma2_rn(ea_bc(4.0f), p2, __ffma2_rn(ea_bc(-5.0f), p1, __ffma2_rn(ea_bc(2.0f), p0, make_float2(-p3.x, -p3.y))));
  const float2 c2 = ea_sub2(p2, p0);
  f = __ffma2_rn(ea_bc(hx), __ffma2_rn(ea_bc(x), __ffma2_rn(ea_bc(x), a2, b2), c2), p1);
  d = __ffma2_rn(ea_bc(x), __ffma2_rn(ea_bc(x15), a2, b2), __fmul2_rn(ea_bc(0.5f), c2));
}
// f = normalised value; gu, gv = derivatives of the RAW (pixel-unit) interpolant along u and v: the caller folds the
// normalisation scale and the focal lengths into one factor per axis (ea_jacobian).
__device__ __forceinline__ void ea_interp(const float (&t)[16], const float du, const float dv, const float2 affine, float& f, float& gu, float& gv) {
  const float hv = 0.5f * dv, v15 = 1.5f * dv, hu = 0.5f * du, u15 = 1.5f * du;
  float2 f01, d01, f23, d23;      // columns 0,1 and 2,3: value and derivative along v (the texel pairs arrive in adjacent registers)
  ea_cubic2(ea_f2(t[0], t[1]), ea_f2(t[4], t[5]), ea_f2(t[8], t[9]), ea_f2(t[12], t[13]), dv, hv, v15, f01, d01);
  ea_cubic2(ea_f2(t[2], t[3]), ea_f2(t[6], t[7]), ea_f2(t[10], t[11]), ea_f2(t[14], t[15]), dv, hv, v15, f23, d23);
  // along u: scalar (pairing {f_k, d_k} would cost a register move per element, more than the packed operations save)
  float val;
  ea_cubic(f01.x, f01.y, f23.x, f23.y, du, hu, u15, val, gu);
  gv = ea_cubic_val(d01.x, d01.y, d23.x, d23.y, du, hu);
  f = fmaf(val, affine.x, affine.y);
}

// Per-solve constants of the evaluation loop in the form it consumes them, derived once on the host (kernel arguments: the hot
// loop reads them as constant-bank operands instead of converting ea_solve_params' doubles in every iteration).
struct EaEvalConsts {
  int type; float a, b, two_a, inv_a, inv_b;   // loss: type, scale a, a^2, 2a, 1/a, 1/a^2 (fp32, IEEE-rounded as the loop used to)
  unsigned stride_bytes[2];                    // byte step of the point stream per residual: point_stride x 8 (pixel points), x 16 (XYZ)
};
__host__ __device__ inline EaEvalConsts ea_eval_consts(int type, double scale, int point_stride = 1) {
  EaEvalConsts L;
  L.type = type; L.a = float(scale); L.b = L.a * L.a; L.two_a = 2.0f * L.a; L.inv_a = 1.0f / L.a; L.inv_b = 1.0f / L.b;
  L.stride_bytes[0] = unsigned(point_stride) * 8u; L.stride_bytes[1] = unsigned(point_stride) * 16u;
  return L;
}

// Loss (ceres/loss_function.cc) + Corrector (rho'' <= 0 for all three => scale by sqrt(rho')) in fp32.
// Returns sqrt(rho'), writes rho(s).
__device__ __forceinline__ float ea_loss_eval(const EaEvalConsts& L, float r, float& rho0) {
  const float s = r * r;
  if (L.type == EA_LOSS_CAUCHY) {
    const float sum = fmaf(s, L.inv_b, 1.0f);
    rho0 = L.b * log1pf(s * L.inv_b);
    return rsqrtf(sum);
  } else if (L.type == EA_LOSS_HUBER) {
    if (s > L.b) {
      // rho = 2 a |r| - a^2, sqrt(rho') = sqrt(a / |r|) = rsqrt(|r| / a): MUFU.RSQ plus one Newton step (<= 1 ulp) instead of an
      // IEEE division and square root (25 instructions with their slow-path calls, paid by every warp that holds one outlier)
      const float ar = fabsf(r);
      rho0 = fmaf(L.two_a, ar, -L.b);
      const float x = ar * L.inv_a;
      float y = rsqrtf(x);
      y = y * fmaf(-0.5f * x, y * y, 1.5f);
      return y;
    }
    rho0 = s;
    return 1.0f;
  }
  rho0 = s;
  return 1.0f;
}

// Analytic local Jacobian (collapsed closed form of AutoDiff x QuaternionParameterization, SURVEY.md A.3):
// g = dr/dp', J = [ 2 (R X) x g | g ], then robust re-weighting.  Everything is rebuilt in fp32 from the projected
// coordinates: p' = z' (xn, yn, 1) with xn = (u' - cx) / fx, R X = p' - t.  gu, gv: raw interpolant derivatives (ea_interp);
// afx = scale * fx, afy = scale * fy (normalisation scale of the distance transform times the focal lengths).
__device__ __forceinline__ void ea_jacobian(const float gu, const float gv, const float ub, const float vb, const float pz, const float iz,
                                            const EaPose& P, const float afx, const float afy, const float w, float J[6]) {
  const float xn = ub * P.inv_fx, yn = vb * P.inv_fy;
  const float y2x = fmaf(2.0f, pz * xn, P.m2t[0]), y2y = fmaf(2.0f, pz * yn, P.m2t[1]), y2z = fmaf(2.0f, pz, P.m2t[2]);   // 2 (R X)
  const float wi = w * iz;
  const float g0 = (gu * afx) * wi;
  const float g1 = (gv * afy) * wi;
  const float g2 = fmaf(-g0, xn, -(g1 * yn));
  J[0] = fmaf(y2y, g2, -(y2z * g1));
  J[1] = fmaf(y2z, g0, -(y2x * g2));
  J[2] = fmaf(y2x, g1, -(y2y * g0));
  J[3] = g0; J[4] = g1; J[5] = g2;
}

// Warp, project, bicubic lookup for one edge point (per-point API of the parity tests and the EAResidue facade).
// dt = pixel (0,0) of the padded distance transform.
template <bool XYZ>
__device__ __forceinline__ void ea_point_eval(const double a0, const double a1, const double a2, const EaLevelGeom& now,
                                              double inv_depth_scale, const EaPose& P,
                                              const float* __restrict__ dt, const float2 affine, EaPointEval& o) {
  const int pitch = ea_dt_pitch(now.w);
  EaProj r;
  ea_project<XYZ>(a0, a1, a2, now.w, now.h, pitch, inv_depth_scale, P, r);
  float t[16];
  ea_gather(ea_gather_base(dt - ea_dt_origin_offset(now.w), pitch), r.off, pitch, t);
  ea_interp(t, r.du, r.dv, affine, o.f, o.gu, o.gv);
  o.ub = r.ub; o.vb = r.vb; o.pz = r.pz; o.iz = r.iz; o.fail = r.zm < 0;
}

// Transposing warp reduction: every lane holds 32 partial sums v[0..31]; afterwards lane L holds in v[0]
// the warp-wide sum of slot L.  31 shuffles instead of 32 x 5.
template <int N>
__device__ __forceinline__ void ea_bfly_stage(float (&v)[EA_NSUM], bool upper, int bit) {
#pragma unroll
  for (int k = 0; k < N / 2; ++k) {
    const float send = upper ? v[k] : v[k + N / 2];
    const float keep = upper ? v[k + N / 2] : v[k];
    v[k] = keep + __shfl_xor_sync(0xffffffffu, send, bit);
  }
}
__device__ __forceinline__ float ea_warp_transpose_reduce(float (&v)[EA_NSUM], int lane) {
  ea_bfly_stage<32>(v, lane & 16, 16);
  ea_bfly_stage<16>(v, lane & 8, 8);
  ea_bfly_stage<8>(v, lane & 4, 4);
  ea_bfly_stage<4>(v, lane & 2, 2);
  ea_bfly_stage<2>(v, lane & 1, 1);
  return v[0];
}
__device__ __forceinline__ double ea_warp_sum(double x) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  return x;
}

// accumulate one point's outer products into the 32 fp32 slots
__device__ __forceinline__ void ea_accumulate(float (&acc)[EA_NSUM], const float J[6], float rw) {
  int k = 0;
#pragma unroll
  for (int a = 0; a < 6; ++a)
#pragma unroll
    for (int c = a; c < 6; ++c) { acc[k] = fmaf(J[a], J[c], acc[k]); ++k; }
#pragma unroll
  for (int a = 0; a < 6; ++a) acc[21 + a] = fmaf(J[a], rw, acc[21 + a]);
}

// =================================================================================================================
// General per-point evaluation for the residual VARIANTS of the reference (standalone/utils.h:101-421):
//   EAResidueEx           radial-tangential distortion between normalisation and K            (utils.h:140-149)
//   EAResidueSecondCam    rigid rig: b_T_a_SecCam = T_1to2 * b_T_a * T_1to2_inv               (utils.h:244-256)
//   EAResidueSecondCamEx  both
// Same skeleton as ea_point_eval; not the batched hot path (used by ea_eval_views / ea_solve_views).
// =================================================================================================================
struct EaViewXf {            // kernel parameter
  double T21[12], T12[12];   // trans_1to2 / trans_1to2_inv, 3x4 row-major [R | t]
  double dist[5];            // k1, k2, p1, p2, k3
  int use_rig, use_dist;
};

struct EaPoseG {
  double A[9], tt[3];        // q = s * (A a) + tt ; camera coordinates when use_dist, else K-folded as in EaPose
  double k1, k2, p1, p2, k3, fx, fy, cx, cy;
  float Rt21[9];             // R21^T (identity without rig): pulls the gradient back into the first camera
  float t21[3], t[3];
  float fxf, fyf, inv_fx, inv_fy;
  int use_dist, use_rig;
};

template <bool XYZ>
__device__ __forceinline__ void ea_pose_setup_general(const double* x7, const EaLevelGeom& ref, const EaLevelGeom& now,
                                                      const EaViewXf& V, EaPoseG& P) {
  const double qw = x7[0], qx = x7[1], qy = x7[2], qz = x7[3];
  const double tx = 2.0 * qx, ty = 2.0 * qy, tz = 2.0 * qz;
  const double twx = tx * qw, twy = ty * qw, twz = tz * qw;
  const double txx = tx * qx, txy = ty * qx, txz = tz * qx;
  const double tyy = ty * qy, tyz = tz * qy, tzz = tz * qz;
  double R[9] = {1.0 - (tyy + tzz), txy - twz, txz + twy, txy + twz, 1.0 - (txx + tzz), tyz - twx, txz - twy, tyz + twx, 1.0 - (txx + tyy)};
  double t[3] = {x7[4], x7[5], x7[6]};
  double Rp[9], tp[3];
  if (V.use_rig) {   // R' = R21 R R12 ; t' = R21 (R t12 + t) + t21
    double RR[9], v[3];
    for (int i = 0; i < 3; ++i) {
      for (int j = 0; j < 3; ++j) RR[3 * i + j] = R[3 * i] * V.T12[j] + R[3 * i + 1] * V.T12[4 + j] + R[3 * i + 2] * V.T12[8 + j];
      v[i] = R[3 * i] * V.T12[3] + R[3 * i + 1] * V.T12[7] + R[3 * i + 2] * V.T12[11] + t[i];
    }
    for (int i = 0; i < 3; ++i) {
      for (int j = 0; j < 3; ++j) Rp[3 * i + j] = V.T21[4 * i] * RR[j] + V.T21[4 * i + 1] * RR[3 + j] + V.T21[4 * i + 2] * RR[6 + j];
      tp[i] = V.T21[4 * i] * v[0] + V.T21[4 * i + 1] * v[1] + V.T21[4 * i + 2] * v[2] + V.T21[4 * i + 3];
    }
    for (int i = 0; i < 3; ++i) { for (int j = 0; j < 3; ++j) P.Rt21[3 * i + j] = float(V.T21[4 * j + i]); P.t21[i] = float(V.T21[4 * i + 3]); }
  } else {
    for (int i = 0; i < 9; ++i) Rp[i] = R[i];
    for (int i = 0; i < 3; ++i) tp[i] = t[i];
    for (int i = 0; i < 9; ++i) P.Rt21[i] = (i % 4 == 0) ? 1.0f : 0.0f;
    P.t21[0] = P.t21[1] = P.t21[2] = 0.0f;
  }
  double M[9];
  for (int i = 0; i < 3; ++i) {
    if (XYZ) { M[3 * i] = Rp[3 * i]; M[3 * i + 1] = Rp[3 * i + 1]; M[3 * i + 2] = Rp[3 * i + 2]; }
    else {
      M[3 * i] = Rp[3 * i] * ref.inv_fx;
      M[3 * i + 1] = Rp[3 * i + 1] * ref.inv_fy;
      M[3 * i + 2] = Rp[3 * i + 2] - ref.cx * M[3 * i] - ref.cy * M[3 * i + 1];
    }
  }
  if (V.use_dist) {
    for (int i = 0; i < 9; ++i) P.A[i] = M[i];
    for (int i = 0; i < 3; ++i) P.tt[i] = tp[i];
  } else {
    for (int j = 0; j < 3; ++j) {
      P.A[j] = now.fx * M[j] + now.cx * M[6 + j];
      P.A[3 + j] = now.fy * M[3 + j] + now.cy * M[6 + j];
      P.A[6 + j] = M[6 + j];
    }
    P.tt[0] = now.fx * tp[0] + now.cx * tp[2]; P.tt[1] = now.fy * tp[1] + now.cy * tp[2]; P.tt[2] = tp[2];
  }
  P.k1 = V.dist[0]; P.k2 = V.dist[1]; P.p1 = V.dist[2]; P.p2 = V.dist[3]; P.k3 = V.dist[4];
  P.fx = now.fx; P.fy = now.fy; P.cx = now.cx; P.cy = now.cy;
  P.t[0] = float(t[0]); P.t[1] = float(t[1]); P.t[2] = float(t[2]);
  P.fxf = float(now.fx); P.fyf = float(now.fy); P.inv_fx = float(now.inv_fx); P.inv_fy = float(now.inv_fy);
  P.use_dist = V.use_dist; P.use_rig = V.use_rig;
}

// value f, robust weight and local Jacobian of one point for any variant; returns the failure flag
template <bool XYZ>
__device__ __forceinline__ bool ea_point_eval_general(const float4 p, const EaLevelGeom& now, double inv_depth_scale, const EaPoseG& P,
                                                      const float* __restrict__ dt, const float2 affine, int loss_type, float loss_a,
                                                      float& f_out, float& w_out, float& rho0, float J[6]) {
  const double a0 = double(p.x), a1 = double(p.y);
  double q0, q1, q2;
  if (XYZ) {
    const double a2 = double(p.z);
    q0 = fma(P.A[0], a0, fma(P.A[1], a1, fma(P.A[2], a2, P.tt[0])));
    q1 = fma(P.A[3], a0, fma(P.A[4], a1, fma(P.A[5], a2, P.tt[1])));
    q2 = fma(P.A[6], a0, fma(P.A[7], a1, fma(P.A[8], a2, P.tt[2])));
  } else {
    const double Z = double(p.z) * inv_depth_scale;
    q0 = fma(Z, fma(P.A[0], a0, fma(P.A[1], a1, P.A[2])), P.tt[0]);
    q1 = fma(Z, fma(P.A[3], a0, fma(P.A[4], a1, P.A[5])), P.tt[1]);
    q2 = fma(Z, fma(P.A[6], a0, fma(P.A[7], a1, P.A[8])), P.tt[2]);
  }
  const bool fail = (q2 < 0.01) && (q2 > -0.01);
  const double iz = 1.0 / q2;
  double u, v;
  float Dxx = 1.f, Dxy = 0.f, Dyx = 0.f, Dyy = 1.f, xn, yn;   // d(distorted)/d(normalised)
  if (P.use_dist) {
    const double x = q0 * iz, y = q1 * iz;
    const double r2 = x * x + y * y, r4 = r2 * r2, r6 = r4 * r2;
    const double radial = 1.0 + P.k1 * r2 + P.k2 * r4 + P.k3 * r6;
    const double dx = x * radial + 2.0 * P.p1 * x * y + P.p2 * (r2 + 2.0 * x * x);
    const double dy = y * radial + 2.0 * P.p2 * x * y + P.p1 * (r2 + 2.0 * y * y);
    u = P.fx * dx + P.cx; v = P.fy * dy + P.cy;
    const double rd = P.k1 + 2.0 * P.k2 * r2 + 3.0 * P.k3 * r4;
    Dxx = float(radial + 2.0 * x * x * rd + 2.0 * P.p1 * y + 6.0 * P.p2 * x);
    Dxy = float(2.0 * x * y * rd + 2.0 * P.p1 * x + 2.0 * P.p2 * y);
    Dyx = float(2.0 * x * y * rd + 2.0 * P.p2 * y + 2.0 * P.p1 * x);
    Dyy = float(radial + 2.0 * y * y * rd + 2.0 * P.p2 * x + 6.0 * P.p1 * y);
    xn = float(x); yn = float(y);
  } else {
    u = q0 * iz; v = q1 * iz;
    xn = float((u - P.cx)) * P.inv_fx; yn = float((v - P.cy)) * P.inv_fy;
  }
  const int W = now.w, H = now.h, pitch = ea_dt_pitch(W);
  int iu, iv;
  float du, dv;
  ea_floor_frac(u, iu, du);
  ea_floor_frac(v, iv, dv);
  iu = min(max(iu, 1 - EA_DT_PAD), W + 1); iv = min(max(iv, 1 - EA_DT_PAD), H + 1);
  float tex[16];
  ea_gather(ea_gather_base(dt - ea_dt_origin_offset(W), pitch), iv * pitch + iu, pitch, tex);
  float f0, f1, f2, f3, d0, d1, d2, d3, fr, fdu;
  const float hv = 0.5f * dv, v15 = 1.5f * dv, hu = 0.5f * du, u15 = 1.5f * du;
  ea_cubic(tex[0], tex[4], tex[8], tex[12], dv, hv, v15, f0, d0);
  ea_cubic(tex[1], tex[5], tex[9], tex[13], dv, hv, v15, f1, d1);
  ea_cubic(tex[2], tex[6], tex[10], tex[14], dv, hv, v15, f2, d2);
  ea_cubic(tex[3], tex[7], tex[11], tex[15], dv, hv, v15, f3, d3);
  ea_cubic(f0, f1, f2, f3, du, hu, u15, fr, fdu);
  const float f = fmaf(fr, affine.x, affine.y);
  const float gu = fdu * affine.x * P.fxf;                                          // dr/d(distorted x)
  const float gv = ea_cubic_val(d0, d1, d2, d3, du, hu) * affine.x * P.fyf;         // dr/d(distorted y)
  const float w = ea_loss_eval(ea_eval_consts(loss_type, double(loss_a)), f, rho0);
  // chain rule: distorted -> normalised -> p' (this camera) -> first camera
  const float gx = gu * Dxx + gv * Dyx, gy = gu * Dxy + gv * Dyy;
  const float pz = float(q2), izf = float(iz), wi = w * izf;
  const float g0 = gx * wi, g1 = gy * wi, g2 = -(gx * xn + gy * yn) * wi;
  const float h0 = P.Rt21[0] * g0 + P.Rt21[1] * g1 + P.Rt21[2] * g2;
  const float h1 = P.Rt21[3] * g0 + P.Rt21[4] * g1 + P.Rt21[5] * g2;
  const float h2 = P.Rt21[6] * g0 + P.Rt21[7] * g1 + P.Rt21[8] * g2;
  // y1 = R X1 = R21^T (p' - t21) - t
  const float px = xn * pz - P.t21[0], py = yn * pz - P.t21[1], pzz = pz - P.t21[2];
  const float yx = P.Rt21[0] * px + P.Rt21[1] * py + P.Rt21[2] * pzz - P.t[0];
  const float yy = P.Rt21[3] * px + P.Rt21[4] * py + P.Rt21[5] * pzz - P.t[1];
  const float yz = P.Rt21[6] * px + P.Rt21[7] * py + P.Rt21[8] * pzz - P.t[2];
  J[0] = 2.0f * (yy * h2 - yz * h1);
  J[1] = 2.0f * (yz * h0 - yx * h2);
  J[2] = 2.0f * (yx * h1 - yy * h0);
  J[3] = h0; J[4] = h1; J[5] = h2;
  f_out = f; w_out = w;
  return fail;
}
