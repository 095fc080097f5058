// Device-side Levenberg-Marquardt state machine (one thread) -- replaces ceres::Solve's
// TrustRegionMinimizer + LevenbergMarquardtStrategy + DenseQRSolver for the 6-DoF problem
// assembled at standalone_edge_align.cpp:265-286.  Works purely on the 27 normal-equation
// sums + cost (SURVEY.md A.4 "normal-equation form"): (S H S + diag/radius) y = S b by 6x6
// Cholesky in fp64 instead of Householder QR on the (n+6)x6 stacked Jacobian.
#pragma once
#include <cfloat>

#include "ea_device.cuh"

#ifndef EA_SOLVE_THREADS
#define EA_SOLVE_THREADS 512   // threads per CTA of every kernel built on ea_eval_slice (128 registers each: one CTA fills an SM)
#endif

#define EA_CMD_EVAL 0
#define EA_CMD_DONE 1


struct EaLmState {
  double x[7];        // accepted iterate
  double cand[7];     // candidate under evaluation
  double H[21], b[6]; // normal equations at x (corrected, unscaled, local)
  double scale[6], diag[6];
  double cost, initial_cost, radius, decrease_factor, model_cost_change;
  double dl_mu, dl_alpha, dl_step_norm, dl_grad[6], dl_gn[6];   // DoglegStrategy state (trust_region_strategy == 1)
  int phase, iter, accepted, rejected, invalid_run, reuse_diag, evals, term;
  int dl_reuse, pad;
#ifdef EA_LM_PROFILE
  long long prof[8];   // cycles per section of ea_lm_advance_warp's fast track (development aid)
#endif
};
#ifdef EA_LM_PROFILE
#define EA_LM_LAP(k) do { const long long t_ = clock64(); if (lane == 0) S.prof[k] += t_ - lm_t_; lm_t_ = t_; } while (0)
#else
#define EA_LM_LAP(k) do { } while (0)
#endif

__device__ inline void ea_quat_plus(const double* x, const double* d, double* out) {
  // ceres::QuaternionParameterization::Plus -- delta is a half-angle vector, left multiplication:
  //   q+ = (cos|d|, sin|d| / |d| * d) (x) q.   Both factors are even in |d|: for |d| < 0.1 (every LM step of a tracker) they
  // are taken from their Maclaurin series in |d|^2 (truncation < 1e-20, i.e. correct to the last bit or two) -- no sqrt, no
  // libm range reduction on the serial section between two evaluations.  Larger steps take the textbook form.
  const double n2 = d[0] * d[0] + d[1] * d[1] + d[2] * d[2];
  if (n2 > 0.0) {
    double s, c;
    if (n2 < 0.01) {
      c = fma(n2, fma(n2, fma(n2, fma(n2, fma(n2, fma(n2, 1.0 / 479001600.0, -1.0 / 3628800.0), 1.0 / 40320.0), -1.0 / 720.0), 1.0 / 24.0), -0.5), 1.0);
      s = fma(n2, fma(n2, fma(n2, fma(n2, fma(n2, fma(n2, 1.0 / 6227020800.0, -1.0 / 39916800.0), 1.0 / 362880.0), -1.0 / 5040.0), 1.0 / 120.0), -1.0 / 6.0), 1.0);
    } else {
      const double n = sqrt(n2);
      s = sin(n) / n; c = cos(n);
    }
    const double q0 = c, q1 = s * d[0], q2 = s * d[1], q3 = s * d[2];
    out[0] = q0 * x[0] - q1 * x[1] - q2 * x[2] - q3 * x[3];
    out[1] = q0 * x[1] + q1 * x[0] + q2 * x[3] - q3 * x[2];
    out[2] = q0 * x[2] - q1 * x[3] + q2 * x[0] + q3 * x[1];
    out[3] = q0 * x[3] + q1 * x[2] - q2 * x[1] + q3 * x[0];
  } else {
    out[0] = x[0]; out[1] = x[1]; out[2] = x[2]; out[3] = x[3];
  }
}
__device__ inline void ea_pose_plus(const double* x, const double* d, double* out) {
  ea_quat_plus(x, d, out);
  out[4] = x[4] + d[3]; out[5] = x[5] + d[4]; out[6] = x[6] + d[5];
}
__device__ inline int ea_tri(int a, int c) { return a * 6 - (a * (a - 1)) / 2 + (c - a); }  // a <= c

// true iff || x - Plus(x, -g) ||_inf <= tol  (trust_region_minimizer.cc, EvaluateGradientAndJacobian).
// The translation block of Plus is a plain addition, so the norm is at least max|g_t| (up to one rounding of
// x_t): unless that is already tiny the full quaternion update (sin/cos of |g|, possibly huge) is skipped.
__device__ inline bool ea_gradient_converged(const EaLmState& S, double tol) {
  double gt = fmax(fabs(S.b[3]), fmax(fabs(S.b[4]), fabs(S.b[5])));
  double xt = fmax(fabs(S.x[4]), fmax(fabs(S.x[5]), fabs(S.x[6])));
  if (gt > 2.0 * tol + 4.5e-16 * xt) return false;
  double ng[6], xp[7];
#pragma unroll
  for (int j = 0; j < 6; ++j) ng[j] = -S.b[j];
  ea_pose_plus(S.x, ng, xp);
  double m = 0.0;
#pragma unroll
  for (int i = 0; i < 7; ++i) m = fmax(m, fabs(S.x[i] - xp[i]));
  return m <= tol;
}

// (A + diag(add)) y = bs by 6x6 LDL^T in registers (fully unrolled; one reciprocal per pivot).  false on failure.
__device__ inline bool ea_ldlt_solve6(const double (&A)[6][6], const double* add, const double* bs, double* y) {
  double L[6][6], dinv[6], dval[6];
  bool ok = true;
#pragma unroll
  for (int j = 0; j < 6; ++j) {
    double d = A[j][j] + add[j];
    double v[6];
#pragma unroll
    for (int k = 0; k < j; ++k) { v[k] = L[j][k] * dval[k]; d = fma(-L[j][k], v[k], d); }
    ok = ok && (d > 0.0) && isfinite(d);
    dval[j] = d;
    dinv[j] = 1.0 / d;
#pragma unroll
    for (int i = j + 1; i < 6; ++i) {
      double s = A[i][j];
#pragma unroll
      for (int k = 0; k < j; ++k) s = fma(-L[i][k], v[k], s);
      L[i][j] = s * dinv[j];
    }
  }
  if (!ok) return false;
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    double s = bs[i];
#pragma unroll
    for (int k = 0; k < i; ++k) s = fma(-L[i][k], y[k], s);
    y[i] = s;
  }
#pragma unroll
  for (int i = 0; i < 6; ++i) y[i] *= dinv[i];
#pragma unroll
  for (int i = 5; i >= 0; --i) {
    double s = y[i];
#pragma unroll
    for (int k = i + 1; k < 6; ++k) s = fma(-L[k][i], y[k], s);
    y[i] = s;
    ok = ok && isfinite(s);
  }
  return ok;
}

// Trust-region step on the normal equations (H_s = S H S, b_s = S b).  Returns false on an invalid step.
//   strategy 0: LevenbergMarquardtStrategy::ComputeStep   (H_s + diag/radius) y = b_s, step = -y
//   strategy 1: DoglegStrategy::ComputeStep, TRADITIONAL_DOGLEG (src/SolveEA.cpp:192): Gauss-Newton / Cauchy interpolation
//               inside the elliptical region |D step| <= radius
__device__ inline bool ea_lm_compute_step(EaLmState& S, const ea_solve_params& sp, double* delta) {
  double A[6][6], bs[6], step[6];
#pragma unroll
  for (int a = 0; a < 6; ++a) {
    bs[a] = S.scale[a] * S.b[a];
#pragma unroll
    for (int c = a; c < 6; ++c) { A[a][c] = S.scale[a] * S.H[ea_tri(a, c)] * S.scale[c]; A[c][a] = A[a][c]; }
  }
  if (sp.trust_region_strategy == 0) {
    if (!S.reuse_diag) {
#pragma unroll
      for (int j = 0; j < 6; ++j) S.diag[j] = fmin(fmax(A[j][j], sp.min_lm_diagonal), sp.max_lm_diagonal);
    }
    S.reuse_diag = 1;
    const double inv_radius = 1.0 / S.radius;
    double add[6], y[6];
#pragma unroll
    for (int j = 0; j < 6; ++j) add[j] = S.diag[j] * inv_radius;
    if (!ea_ldlt_solve6(A, add, bs, y)) return false;
#pragma unroll
    for (int j = 0; j < 6; ++j) step[j] = -y[j];
  } else {
    if (!S.dl_reuse) {
      S.dl_reuse = 1;
      double g2 = 0.0, sg[6];
#pragma unroll
      for (int j = 0; j < 6; ++j) {
        S.diag[j] = sqrt(fmin(fmax(A[j][j], sp.min_lm_diagonal), sp.max_lm_diagonal));
        S.dl_grad[j] = bs[j] / S.diag[j];
        sg[j] = S.dl_grad[j] / S.diag[j];
        g2 = fma(S.dl_grad[j], S.dl_grad[j], g2);
      }
      double Jg2 = 0.0;
#pragma unroll
      for (int a = 0; a < 6; ++a) {
        double row = 0.0;
#pragma unroll
        for (int c = 0; c < 6; ++c) row = fma(A[a][c], sg[c], row);
        Jg2 = fma(sg[a], row, Jg2);
      }
      S.dl_alpha = g2 / Jg2;
      bool ok = false;
      double y[6];
      while (S.dl_mu < 1.0) {
        double add[6];
#pragma unroll
        for (int j = 0; j < 6; ++j) add[j] = S.diag[j] * S.diag[j] * S.dl_mu;
        if (ea_ldlt_solve6(A, add, bs, y)) { ok = true; break; }
        S.dl_mu *= 10.0;
      }
      if (!ok) return false;
#pragma unroll
      for (int j = 0; j < 6; ++j) S.dl_gn[j] = -y[j] * S.diag[j];
    }
    double gn2 = 0.0, g2 = 0.0, gdotgn = 0.0, ds[6];
#pragma unroll
    for (int j = 0; j < 6; ++j) { gn2 = fma(S.dl_gn[j], S.dl_gn[j], gn2); g2 = fma(S.dl_grad[j], S.dl_grad[j], g2); gdotgn = fma(S.dl_grad[j], S.dl_gn[j], gdotgn); }
    const double gn_norm = sqrt(gn2), g_norm = sqrt(g2);
    if (gn_norm <= S.radius) {
#pragma unroll
      for (int j = 0; j < 6; ++j) ds[j] = S.dl_gn[j];
      S.dl_step_norm = gn_norm;
    } else if (g_norm * S.dl_alpha >= S.radius) {
#pragma unroll
      for (int j = 0; j < 6; ++j) ds[j] = -(S.radius / g_norm) * S.dl_grad[j];
      S.dl_step_norm = S.radius;
    } else {
      const double b_dot_a = -S.dl_alpha * gdotgn;
      const double a2 = (S.dl_alpha * g_norm) * (S.dl_alpha * g_norm);
      const double bma2 = a2 - 2.0 * b_dot_a + gn2;
      const double c = b_dot_a - a2;
      const double d = sqrt(c * c + bma2 * (S.radius * S.radius - a2));
      const double beta = (c <= 0.0) ? (d - c) / bma2 : (S.radius * S.radius - a2) / (d + c);
      double nn = 0.0;
#pragma unroll
      for (int j = 0; j < 6; ++j) { ds[j] = (-S.dl_alpha * (1.0 - beta)) * S.dl_grad[j] + beta * S.dl_gn[j]; nn = fma(ds[j], ds[j], nn); }
      S.dl_step_norm = sqrt(nn);
    }
#pragma unroll
    for (int j = 0; j < 6; ++j) step[j] = ds[j] / S.diag[j];
  }
  // model_cost_change = -(step^T b_s + 1/2 step^T H_s step) = -(delta^T b + 1/2 delta^T H delta) with delta = S step: taken
  // from the unscaled sums in shared memory, so that the scaled matrix need not stay in registers across the factorisation
#pragma unroll
  for (int a = 0; a < 6; ++a) delta[a] = step[a] * S.scale[a];  // undo the Jacobi column scaling
  double lin = 0.0, quad = 0.0;
#pragma unroll
  for (int a = 0; a < 6; ++a) {
    lin = fma(delta[a], S.b[a], lin);
    double row = 0.0;
#pragma unroll
    for (int c = 0; c < 6; ++c) row = fma(S.H[a <= c ? ea_tri(a, c) : ea_tri(c, a)], delta[c], row);
    quad = fma(delta[a], row, quad);
  }
  S.model_cost_change = -(lin + 0.5 * quad);
  return S.model_cost_change > 0.0;
}

// Next candidate from the state at S.x (TrustRegionMinimizer's loop head + ComputeTrustRegionStep + HandleInvalidStep):
// EA_CMD_EVAL with S.cand set, or EA_CMD_DONE with S.term.
static __device__ __forceinline__ int ea_lm_propose(EaLmState& S, const ea_solve_params& sp) {
  for (;;) {
    if (S.iter >= sp.max_num_iterations) { S.term = EA_TERM_NO_CONVERGENCE; return EA_CMD_DONE; }
    if (S.radius < sp.min_trust_region_radius) { S.term = EA_TERM_CONVERGENCE_MIN_RADIUS; return EA_CMD_DONE; }
    S.iter++;
    double delta[6];
    if (!ea_lm_compute_step(S, sp, delta)) {  // HandleInvalidStep
      if (++S.invalid_run >= sp.max_consecutive_invalid_steps) { S.term = EA_TERM_FAILURE_INVALID_STEPS; return EA_CMD_DONE; }
      if (sp.trust_region_strategy == 0) { S.radius *= 0.5; S.reuse_diag = 0; }
      else { S.dl_mu *= 10.0; S.dl_reuse = 0; }   // DoglegStrategy::StepIsInvalid
      S.rejected++;
      continue;
    }
    S.invalid_run = 0;
    ea_pose_plus(S.x, delta, S.cand);
    return EA_CMD_EVAL;
  }
}

// Advance the minimiser after an evaluation of S.cand produced `sums`.  Returns EA_CMD_EVAL with a
// new S.cand, or EA_CMD_DONE with S.term set and S.x the final iterate.
static __device__ __forceinline__ int ea_lm_advance_impl(EaLmState& S, const double* sums, const ea_solve_params& sp) {
  const bool fail = sums[27] > 0.0;
  S.evals++;
  if (S.phase == 0) {  // IterationZero
    if (fail) { S.term = EA_TERM_FAILURE_EVAL_X0; S.cost = 0.0; S.initial_cost = 0.0; return EA_CMD_DONE; }
#pragma unroll 1
    for (int k = 0; k < 21; ++k) S.H[k] = sums[k];
#pragma unroll 1
    for (int k = 0; k < 6; ++k) S.b[k] = sums[21 + k];
    S.cost = S.initial_cost = sums[28];
#pragma unroll 1
    for (int j = 0; j < 6; ++j) S.scale[j] = sp.jacobi_scaling ? 1.0 / (1.0 + sqrt(S.H[ea_tri(j, j)])) : 1.0;
    if (ea_gradient_converged(S, sp.gradient_tolerance)) { S.term = EA_TERM_CONVERGENCE_GRADIENT; return EA_CMD_DONE; }
    S.radius = sp.initial_trust_region_radius; S.decrease_factor = 2.0; S.reuse_diag = 0;
    S.dl_mu = 1e-8; S.dl_reuse = 0; S.dl_step_norm = 0.0;
    S.iter = 0; S.phase = 1;
  } else {
    const double cand_cost = fail ? DBL_MAX : sums[28];
    double sn = 0.0, xn = 0.0;
#pragma unroll
    for (int i = 0; i < 7; ++i) { const double d = S.x[i] - S.cand[i]; sn += d * d; xn += S.x[i] * S.x[i]; }
    // |step| <= ptol (|x| + ptol).  (a + b)^2 <= 2 a^2 + 2 b^2, so a squared step above that bound cannot pass: the two square
    // roots are only taken when the step is within a factor sqrt(2) of the tolerance (same decisions either way)
    const double pt2 = sp.parameter_tolerance * sp.parameter_tolerance;
    if (sn <= 2.0 * pt2 * (xn + pt2)) {
      if (sqrt(sn) <= sp.parameter_tolerance * (sqrt(xn) + sp.parameter_tolerance)) { S.term = EA_TERM_CONVERGENCE_PARAMETER; return EA_CMD_DONE; }
    }
    const double cost_change = S.cost - cand_cost;
    if (fabs(cost_change) <= sp.function_tolerance * S.cost) { S.term = EA_TERM_CONVERGENCE_FUNCTION; return EA_CMD_DONE; }
    const double rel = fail ? -DBL_MAX : cost_change / S.model_cost_change;
    if (rel > sp.min_relative_decrease) {  // HandleSuccessfulStep (the fused pass already holds J at x_new)
#pragma unroll
      for (int i = 0; i < 7; ++i) S.x[i] = S.cand[i];
#pragma unroll
      for (int k = 0; k < 21; ++k) S.H[k] = sums[k];
#pragma unroll
      for (int k = 0; k < 6; ++k) S.b[k] = sums[21 + k];
      S.cost = cand_cost;
      if (sp.trust_region_strategy == 0) {
        const double t = 2.0 * rel - 1.0;
        S.radius = fmin(sp.max_trust_region_radius, S.radius / fmax(1.0 / 3.0, 1.0 - t * t * t));
        S.decrease_factor = 2.0; S.reuse_diag = 0;
      } else {   // DoglegStrategy::StepAccepted
        if (rel < 0.25) S.radius *= 0.5;
        if (rel > 0.75) S.radius = fmax(S.radius, 3.0 * S.dl_step_norm);
        S.dl_mu = fmax(1e-8, 2.0 * S.dl_mu / 10.0); S.dl_reuse = 0;
      }
      S.accepted++;
      if (ea_gradient_converged(S, sp.gradient_tolerance)) { S.term = EA_TERM_CONVERGENCE_GRADIENT; return EA_CMD_DONE; }
    } else {  // HandleUnsuccessfulStep
      if (sp.trust_region_strategy == 0) { S.radius = S.radius / S.decrease_factor; S.decrease_factor *= 2.0; S.reuse_diag = 1; }
      else { S.radius *= 0.5; S.dl_reuse = 1; }   // DoglegStrategy::StepRejected
      S.rejected++;
    }
  }
  return ea_lm_propose(S, sp);
}

// The serial state machine out of line: the slow paths of ea_lm_advance_warp call these, so that their register demand does not
// apply to its fast track.
static __device__ __noinline__ int ea_lm_advance(EaLmState& S, const double* sums, const ea_solve_params& sp) { return ea_lm_advance_impl(S, sums, sp); }
static __device__ __noinline__ int ea_lm_propose_slow(EaLmState& S, const ea_solve_params& sp) { return ea_lm_propose(S, sp); }

// ---- warp-cooperative advance: the common case on a fast track ------------------------------------------------------------
// Between two evaluations of a pair nothing else runs on its CTA, so the latency of this step is dead time (the serial version
// above measured 4.4 us per evaluation, 18 % of a persistent CTA's life).  All 32 lanes of one warp call this with the sums in
// shared memory.  The common case -- an accepted LM step that does not terminate the level -- runs here: every lane executes
// the same short, register-resident instruction stream (no divergence, no per-lane state), the state stores are spread over
// the lanes, and the heavy pieces are arranged for instruction-level parallelism (in-place 6x6 LDL^T on the 21 unique entries,
// six independent row chains for the model cost, series Plus).  Everything else (first evaluation of a level, rejected or
// invalid steps, any termination, the dogleg strategy) takes the serial state machine on lane 0, whose arithmetic for the
// shared parts is identical operation for operation.  On EA_CMD_EVAL the next candidate is in S.cand.
__device__ __forceinline__ bool ea_ldlt_solve6_packed(double (&U)[21], const double (&bs)[6], double (&y)[6]) {
  // U: upper triangle, row-major (ea_tri), damping already on the diagonal.  In place: U[tri(j,j)] <- d_j, U[tri(j,i)] <- L[i][j].
  double dinv[6];
  bool ok = true;
#pragma unroll
  for (int j = 0; j < 6; ++j) {
    double d = U[ea_tri(j, j)];
    double v[6];
#pragma unroll
    for (int k = 0; k < j; ++k) { v[k] = U[ea_tri(k, j)] * U[ea_tri(k, k)]; d = fma(-U[ea_tri(k, j)], v[k], d); }
    ok = ok && (d > 0.0) && isfinite(d);
    U[ea_tri(j, j)] = d;
    dinv[j] = 1.0 / d;
#pragma unroll
    for (int i = j + 1; i < 6; ++i) {
      double t = U[ea_tri(j, i)];
#pragma unroll
      for (int k = 0; k < j; ++k) t = fma(-U[ea_tri(k, i)], v[k], t);
      U[ea_tri(j, i)] = t * dinv[j];
    }
  }
  // (no early exit on a failed pivot: y is then meaningless but unused, and a branch here made ptxas spill y at the merge)
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    double t = bs[i];
#pragma unroll
    for (int k = 0; k < i; ++k) t = fma(-U[ea_tri(k, i)], y[k], t);
    y[i] = t;
  }
#pragma unroll
  for (int i = 0; i < 6; ++i) y[i] *= dinv[i];
#pragma unroll
  for (int i = 5; i >= 0; --i) {
    double t = y[i];
#pragma unroll
    for (int k = i + 1; k < 6; ++k) t = fma(-U[ea_tri(i, k)], y[k], t);
    y[i] = t;
    ok = ok && isfinite(t);
  }
  return ok;
}

static __device__ __noinline__ int ea_lm_advance_warp(EaLmState& __restrict__ S, const double* __restrict__ sums, const ea_solve_params& __restrict__ sp,
                                                      const int lane) {
  // (S, sums and the parameters never alias: without the qualifiers every store into S -- and there is one per state field --
  // orders the loads behind it, which serialises six clamp chains and most of the section boundaries)
  const unsigned full = 0xffffffffu;
#ifdef EA_LM_PROFILE
  long long lm_t_ = clock64();
#endif
  // the serial state machine serves: the dogleg strategy, failed evaluations, rejected steps, near-tolerance decisions
  bool fast = (sp.trust_region_strategy == 0) && !(sums[27] > 0.0);
  const int phase = S.phase;
  double rel = 0.0, radius = 0.0;
  const double cand_cost = sums[28];
  int iter = 0;
  if (fast && phase == 1) {
    double sn = 0.0, xn = 0.0;
#pragma unroll
    for (int i = 0; i < 7; ++i) { const double xo = S.x[i]; const double d = xo - S.cand[i]; sn += d * d; xn += xo * xo; }
    const double pt2 = sp.parameter_tolerance * sp.parameter_tolerance;
    if (sn <= 2.0 * pt2 * (xn + pt2)) fast = false;                    // near the parameter tolerance: the exact test decides
    const double cost_change = S.cost - cand_cost;
    if (fabs(cost_change) <= sp.function_tolerance * S.cost) {
      // CONVERGENCE_FUNCTION (what nearly every level ends with): decided here, the iterate stays where it is
      if (fast) {
        __syncwarp();
        if (lane == 0) { S.evals++; S.term = EA_TERM_CONVERGENCE_FUNCTION; }
        __syncwarp();
        return EA_CMD_DONE;
      }
    } else { rel = cost_change / S.model_cost_change; if (!(rel > sp.min_relative_decrease)) fast = false; }
  }
  if (!fast) {
    int cmd = 0;
    if (lane == 0) cmd = ea_lm_advance(S, sums, sp);
    cmd = __shfl_sync(full, cmd, 0);
    __syncwarp();
    return cmd;
  }
  EA_LM_LAP(0);
  if (phase == 0) {
    // ---- IterationZero: the state at x0, Jacobi scaling from the first Jacobian (one sqrt + one division per lane) ----
    double mine = 1.0;
    if (lane < 6 && sp.jacobi_scaling) mine = 1.0 / (1.0 + sqrt(sums[ea_tri(lane, lane)]));
    radius = sp.initial_trust_region_radius;
    iter = 0;
    __syncwarp();
    if (lane < 6) S.scale[lane] = mine;
    if (lane < 21) S.H[lane] = sums[lane]; else if (lane < 27) S.b[lane - 21] = sums[lane];
    if (lane == 27) {
      S.cost = cand_cost; S.initial_cost = cand_cost; S.radius = radius; S.decrease_factor = 2.0; S.evals++;
      S.dl_mu = 1e-8; S.dl_reuse = 0; S.dl_step_norm = 0.0; S.phase = 1; S.invalid_run = 0;
    }
  } else {
    // ---- HandleSuccessfulStep ----
    const double t = 2.0 * rel - 1.0;
    radius = fmin(sp.max_trust_region_radius, S.radius / fmax(1.0 / 3.0, 1.0 - t * t * t));
    iter = S.iter;
    __syncwarp();                                  // every lane has read the old state
    if (lane < 7) S.x[lane] = S.cand[lane];
    if (lane < 21) S.H[lane] = sums[lane]; else if (lane < 27) S.b[lane - 21] = sums[lane];
    if (lane == 27) { S.cost = cand_cost; S.radius = radius; S.decrease_factor = 2.0; S.accepted++; S.evals++; S.invalid_run = 0; }
  }
  // From here on the iterate and the scaling are read from the state where they are used (S.x, S.scale): held in registers
  // across the factorisation they pushed the fast track past the register budget of the solve kernels and into local memory.
  __syncwarp();
  // gradient tolerance (same shortcut as ea_gradient_converged: the translation block of Plus is a plain addition)
  {
    const double gt = fmax(fabs(sums[24]), fmax(fabs(sums[25]), fabs(sums[26])));
    const double xt = fmax(fabs(S.x[4]), fmax(fabs(S.x[5]), fabs(S.x[6])));
    if (!(gt > 2.0 * sp.gradient_tolerance + 4.5e-16 * xt)) {
      int conv = 0;
      if (lane == 0) { conv = ea_gradient_converged(S, sp.gradient_tolerance) ? 1 : 0; if (conv) S.term = EA_TERM_CONVERGENCE_GRADIENT; }
      if (__shfl_sync(full, conv, 0)) { if (lane == 0) { S.iter = iter; S.reuse_diag = 0; } __syncwarp(); return EA_CMD_DONE; }
    }
  }
  // ---- loop head of the next iteration ----
  if (iter >= sp.max_num_iterations) { if (lane == 0) { S.term = EA_TERM_NO_CONVERGENCE; S.iter = iter; S.reuse_diag = 0; } __syncwarp(); return EA_CMD_DONE; }
  if (radius < sp.min_trust_region_radius) { if (lane == 0) { S.term = EA_TERM_CONVERGENCE_MIN_RADIUS; S.iter = iter; S.reuse_diag = 0; } __syncwarp(); return EA_CMD_DONE; }
  EA_LM_LAP(1);
  // ---- LevenbergMarquardtStrategy::ComputeStep on (S H S + diag / radius) y = S b ----
  double U[21], bs[6], y[6], delta[6];
  const double inv_radius = 1.0 / radius;
#pragma unroll
  for (int a = 0; a < 6; ++a) {
    bs[a] = S.scale[a] * sums[21 + a];
#pragma unroll
    for (int c = a; c < 6; ++c) U[ea_tri(a, c)] = S.scale[a] * sums[ea_tri(a, c)] * S.scale[c];
  }
  const double dg_lo = sp.min_lm_diagonal, dg_hi = sp.max_lm_diagonal;
#pragma unroll
  for (int j = 0; j < 6; ++j) U[ea_tri(j, j)] += fmin(fmax(U[ea_tri(j, j)], dg_lo), dg_hi) * inv_radius;
  // lane j stores diag[j], recomputed from shared memory with the same operations (picking element `lane` of a register
  // array would put the array in local memory)
  if (lane < 6) S.diag[lane] = fmin(fmax(S.scale[lane] * sums[ea_tri(lane, lane)] * S.scale[lane], dg_lo), dg_hi);
  EA_LM_LAP(2);
  bool ok = ea_ldlt_solve6_packed(U, bs, y);
#pragma unroll
  for (int a = 0; a < 6; ++a) delta[a] = -y[a] * S.scale[a];
  EA_LM_LAP(3);
  // model_cost_change = -(delta^T b + 1/2 delta^T H delta): the serial code's order, as six independent row chains.  The sums
  // are read from their copies in the state (S.H, S.b, as the serial code does): reading `sums` again let the compiler keep
  // the 27 values loaded for U in registers across the factorisation.
  double lin = 0.0, quad = 0.0;
#pragma unroll
  for (int a = 0; a < 6; ++a) {
    lin = fma(delta[a], S.b[a], lin);
    double row = 0.0;
#pragma unroll
    for (int c = 0; c < 6; ++c) row = fma(S.H[a <= c ? ea_tri(a, c) : ea_tri(c, a)], delta[c], row);
    quad = fma(delta[a], row, quad);
  }
  const double model = -(lin + 0.5 * quad);
  ok = ok && (model > 0.0);
  EA_LM_LAP(4);
  if (!ok) {     // HandleInvalidStep: rare; the serial loop recomputes this step, finds it invalid and carries on from there
    __syncwarp();
    int cmd = 0;
    if (lane == 0) { S.iter = iter; S.reuse_diag = 0; cmd = ea_lm_propose_slow(S, sp); }
    cmd = __shfl_sync(full, cmd, 0);
    __syncwarp();
    return cmd;
  }
  double cand[7];
  ea_pose_plus(S.x, delta, cand);
  __syncwarp();
  if (lane == 28) { S.model_cost_change = model; S.iter = iter + 1; S.reuse_diag = 1; }
  if (lane == 29) {
#pragma unroll
    for (int i = 0; i < 7; ++i) S.cand[i] = cand[i];
  }
  __syncwarp();
  EA_LM_LAP(5);
  return EA_CMD_EVAL;
}

// ---- asynchronous point staging (cp.async: global -> shared without a register in between) -----------------------------
__device__ __forceinline__ void ea_cp_async8(const unsigned saddr, const void* g) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(saddr), "l"(g) : "memory");
}
__device__ __forceinline__ void ea_cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void ea_cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ uint2 ea_lds_u2(const unsigned saddr) {
  uint2 v;
  asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(saddr) : "memory");
  return v;
}

#ifndef EA_STAGE_SLOT
#define EA_STAGE_SLOT 512   // points per staging slot (uint2 stage[2][EA_STAGE_SLOT], 8 KB, aligned to 8 KB); a power of two >= the CTA size
#endif
// ---- slice evaluation shared by every solve kernel ----------------------------------------------------------
#ifndef EA_FLUSH_EVERY
#define EA_FLUSH_EVERY 16  // points per thread between fp32 -> fp64 flushes of the normal-equation slots (measured: 8 -> 16 = -1.7 %)
#endif
#ifndef EA_ALTERNATE_SWEEP
#define EA_ALTERNATE_SWEEP 1
#endif

// Per-thread accumulators of the evaluation loop between two flushes.
struct EaEvalAcc {
  float acc[EA_NSUM];    // fp32 normal-equation slots (ea_accumulate)
  float cost;            // fp32 sum of rho / 2 over the (at most EA_FLUSH_EVERY) points since the last flush
  int zmin;              // running minimum of EaProj::zm: negative <=> one of those points failed the z-guard
};

// One point of the evaluation loop: project -> gather -> interpolate -> loss -> Jacobian -> accumulate.  RAGGED: the iteration
// may hold lanes beyond the range (`valid` false: they carry the pad point and contribute nothing); full iterations skip the
// masking altogether.
template <bool XYZ, bool RAGGED>
__device__ __forceinline__ void ea_eval_point(const typename EaPtStream<XYZ>::T p, const bool valid, const int W, const int H, const int pitch,
                                              const double inv_depth_scale, const EaPose& P, const float* __restrict__ dt_base,
                                              const float2 affine, const float afx, const float afy, const EaEvalConsts& loss, EaEvalAcc& A) {
  EaProj r;
  {
    double a0, a1, a2;
    EaPtStream<XYZ>::unpack(p, a0, a1, a2);
    ea_project<XYZ>(a0, a1, a2, W, H, pitch, inv_depth_scale, P, r);
  }
  float t[16];
  ea_gather(dt_base, r.off, pitch, t);
  float f, gu, gv;
  ea_interp(t, r.du, r.dv, affine, f, gu, gv);
  float rho0;
  float w = ea_loss_eval(loss, f, rho0);
  if (RAGGED && !valid) { w = 0.0f; rho0 = 0.0f; f = 0.0f; r.zm = 0x7fffffff; }
  float J[6];
  ea_jacobian(gu, gv, r.ub, r.vb, r.pz, r.iz, P, afx, afy, w, J);
  if (RAGGED && !valid) {   // the pad point may project to inf / NaN
#pragma unroll
    for (int k = 0; k < 6; ++k) J[k] = 0.0f;
  }
  ea_accumulate(A.acc, J, f * w);
  A.zmin = min(A.zmin, r.zm);
  A.cost = fmaf(0.5f, rho0, A.cost);
}

// Evaluate residual indices [j0, j1) (point index = j * stride) with the CTA's threads and leave per-warp partial sums in
// part / cpart (caller synchronises).  dt_pad = FIRST element of the padded distance transform (pixel (-PAD,-PAD)).
//
// One CTA iteration covers THREADS consecutive residuals (a warp load covers 32 consecutive points; the CTA walks the list --
// and the DT rows under it -- front to back, or back to front when `reverse`: successive evaluations of a pair alternate the
// direction, so each sweep starts on the data the previous one touched last, still in L1 / L2, instead of on the data it
// evicted first).  Keeping more than one point per thread in flight was measured and lost (the evaluation phase is issue-
// bound at 16 warps, profiles/r2_kernels.md).
//
// Chunks (chunk_iters > 0, EA_FLUSH_EVERY times a power of two): [j0, j1) starts on a chunk boundary and is cut every
// chunk_iters * THREADS residuals; chunk k of the range leaves its partials in part[k * part_stride ...] / cpart[k * ...]
// (k counted from the range's LOW end in both directions).  A chunk's partials depend only on the chunk, not on the range it
// was evaluated in: iterations are aligned to the chunk grid from the low end (forward) or from the virtual high end `vend`
// (reverse; vend = j0 + n_chunks * chunk, the ragged part of the last chunk sits in the first iterations).  Chunk ends
// coincide with the fp32 -> fp64 flushes, so the bookkeeping lives in the flush branch, not in the loop body.
//
// stage (optional, pixel points only): shared memory, uint2 [2][EA_STAGE_SLOT] (THREADS <= EA_STAGE_SLOT), ALIGNED TO ITS OWN SIZE
// (the loop flips between the two slots with one XOR).  The point of iteration i + 1 is requested at the top of iteration i with cp.async straight into the
// thread's staging slot and read back (LDS) at the top of iteration i + 1: it never occupies registers across the loop body.
// (As a register prefetch it did, the loop sits at the 128-register limit, and ptxas parked it in local memory right behind
// the load -- exposing the load latency in every iteration, +27 % evaluation time.)
// pre_valid: slot 0 already holds (or is about to receive) this call's first point, requested by the previous call;
// prefetch_next: request the first point of the NEXT evaluation of the same range (direction next_reverse) into slot 0 before
// returning, so that its latency hides behind the CTA barrier and the serial LM step.
template <bool XYZ, int THREADS>
__device__ __forceinline__ void ea_eval_slice(const void* __restrict__ pts, const float* __restrict__ dt_pad, const float2 affine,
                                              const EaLevelGeom& ng,
                                              double inv_depth_scale, const EaEvalConsts& loss, const int stride, const EaPose& P, const int j0,
                                              const int j1, double (*part)[EA_NSUM], double* cpart, const bool reverse = false,
                                              uint2* stage = nullptr, const bool pre_valid = false,
                                              const bool prefetch_next = false, const bool next_reverse = false,
                                              const int chunk_iters = 0, const int part_stride = 0) {
  static_assert(THREADS <= EA_STAGE_SLOT, "staging slot too small");
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int W = ng.w, H = ng.h, pitch = ea_dt_pitch(W);
  const float* dt_base = ea_gather_base(dt_pad, pitch);
  const float afx = affine.x * P.fx, afy = affine.x * P.fy;
  typedef EaPtStream<XYZ> PS;
  // virtual iteration space: residual of (iteration it, thread t) = j0 + it * THREADS + t   (forward)
  //                                                                 vend - 1 - (it * THREADS + t)   (reverse)
  const int n = j1 - j0;
  const int n_it = (n + THREADS - 1) / THREADS;
  const int cspan = chunk_iters > 0 ? chunk_iters * THREADS : 0;
  const int n_chunks = cspan > 0 ? (n + cspan - 1) / cspan : 1;
  const int vend = cspan > 0 ? j0 + n_chunks * cspan : j1;
  const int it_first_rev = (vend - j1) / THREADS;             // reverse: whole iterations of padding above j1 are skipped
  auto residual_of = [&](const int it, const bool rev) { return rev ? vend - 1 - (it * THREADS + tid) : j0 + it * THREADS + tid; };
  const int it0 = reverse ? it_first_rev : 0;
  const int it1 = reverse ? (vend - j0 + THREADS - 1) / THREADS : n_it;
  const int rstep = reverse ? -THREADS : THREADS;
  EaEvalAcc A;
#pragma unroll
  for (int k = 0; k < EA_NSUM; ++k) A.acc[k] = 0.0f;
  A.cost = 0.0f; A.zmin = 0x7fffffff;
  // The fp64 accumulators of the 32 slots live in shared memory (part itself): they are touched once per flush, and the
  // registers they would hold across the loop body are what keeps the prefetched point out of local memory.
  double cost64 = 0.0;
  for (int k = 0; k < n_chunks; ++k) part[size_t(k) * part_stride + warp][lane] = 0.0;
  typename PS::T p_next = PS::pad();
  int rj = residual_of(it0, reverse);                          // this thread's residual in the current iteration
  const bool staged = !XYZ && stage != nullptr;
  const unsigned st0 = staged ? unsigned(__cvta_generic_to_shared(stage + tid)) : 0u;   // this thread's slot 0; slot 1 is EA_STAGE_SLOT * 8 bytes further
  unsigned st_cur = st0;
  const char* const pts8 = reinterpret_cast<const char*>(pts);
  const unsigned stride8 = loss.stride_bytes[XYZ ? 1 : 0];
  if (staged) {
    if (!pre_valid) { if (unsigned(rj - j0) < unsigned(n)) ea_cp_async8(st0, pts8 + size_t(unsigned(rj)) * stride8); ea_cp_async_commit(); }
  } else {
    if (unsigned(rj - j0) < unsigned(n)) p_next = PS::load(pts, size_t(rj) * stride);
  }
  for (int it = it0; it < it1; ++it) {
    const bool valid = unsigned(rj - j0) < unsigned(n);
    typename PS::T p = p_next;
    rj += rstep;
    if (staged) {
      ea_cp_async_wait_all();
      if constexpr (!XYZ) { p = ea_lds_u2(st_cur); }
      st_cur ^= unsigned(EA_STAGE_SLOT * 8);                                   // the other slot
      if (unsigned(rj - j0) < unsigned(n)) ea_cp_async8(st_cur, pts8 + size_t(unsigned(rj)) * stride8);
      ea_cp_async_commit();
    } else {
      if (unsigned(rj - j0) < unsigned(n)) p_next = PS::load(pts, size_t(rj) * stride);   // register prefetch (XYZ points, callers without staging)
    }
    // only the first and the last iteration of a range can hold lanes beyond it
    if (it == it0 || it + 1 == it1) {
      if constexpr (!XYZ) { if (!valid) p = PS::pad(); }
      ea_eval_point<XYZ, true>(p, valid, W, H, pitch, inv_depth_scale, P, dt_base, affine, afx, afy, loss, A);
    } else {
      ea_eval_point<XYZ, false>(p, true, W, H, pitch, inv_depth_scale, P, dt_base, affine, afx, afy, loss, A);
    }
    if (((it + 1) & (EA_FLUSH_EVERY - 1)) == 0 || it + 1 == it1) {   // flush cadence on the virtual iteration grid, and at the end
      A.acc[27] = A.zmin < 0 ? 1.0f : 0.0f;
      A.zmin = 0x7fffffff;
      cost64 += double(A.cost);
      A.cost = 0.0f;
      const int csh = 31 - __clz(chunk_iters | 1);                                                             // chunk_iters is a power of two
      const int kc = chunk_iters > 0 ? (reverse ? n_chunks - 1 - (it >> csh) : (it >> csh)) : 0;              // chunk, from the range's low end
      double* slot = &part[size_t(kc) * part_stride + warp][lane];
      *slot += double(ea_warp_transpose_reduce(A.acc, lane));
#pragma unroll
      for (int k = 0; k < EA_NSUM; ++k) A.acc[k] = 0.0f;
      if (it + 1 == it1 || (chunk_iters > 0 && ((it + 1) & (chunk_iters - 1)) == 0)) {   // the chunk is complete: its cost
        const double c64 = ea_warp_sum(cost64);
        if (lane == 0) cpart[size_t(kc) * part_stride + warp] = c64;
        cost64 = 0.0;
      }
    }
  }
  if (it1 <= it0) { if (lane == 0) cpart[warp] = 0.0; }        // empty range
  if (staged && prefetch_next) {
    const int rn = residual_of(next_reverse ? it_first_rev : 0, next_reverse);
    ea_cp_async_wait_all();                                      // (nothing of this call is still reading or filling slot 0)
    if (rn >= j0 && rn < j1) ea_cp_async8(st0, pts8 + size_t(unsigned(rn)) * stride8);
    ea_cp_async_commit();
  }
}

// An evaluation of n_res residuals is cut into at most EA_MAX_CHUNKS chunks of `size` residuals (a multiple of
// THREADS * EA_FLUSH_EVERY, so chunk ends coincide with the fp32 -> fp64 flushes).  Every chunk is reduced on its own, in a
// fixed order, by whichever CTA evaluates it, and the chunk totals are added in chunk order: the sums do not depend on how
// many CTAs shared the evaluation (tail helpers, ea_solve.cu).
#ifndef EA_MAX_CHUNKS
#define EA_MAX_CHUNKS 4
#endif
__device__ __forceinline__ int ea_chunking(const int n_res, const int threads, int& size) {
  // size = unit << s with the smallest s that leaves at most EA_MAX_CHUNKS chunks (a power-of-two number of iterations per
  // chunk: the loop finds its chunk with a shift)
  const int unit = threads * EA_FLUSH_EVERY;
  const int nb = (n_res + unit - 1) / unit;
  int s = 0;
  while (((nb + (1 << s) - 1) >> s) > EA_MAX_CHUNKS) ++s;
  size = unit << s;
  return n_res > 0 ? (n_res + size - 1) / size : 1;
}

// CTA totals from the per-warp partials: lane k of the calling warp returns slot k (k < EA_SUMS), fixed order.
template <int WARPS>
__device__ __forceinline__ double ea_cta_total(const double (*part)[EA_NSUM], const double* cpart, int lane) {
  double s = 0.0;
  if (lane < 28) {
#pragma unroll
    for (int w2 = 0; w2 < WARPS; ++w2) s += part[w2][lane];
  } else if (lane == 28) {
#pragma unroll
    for (int w2 = 0; w2 < WARPS; ++w2) s += cpart[w2];
  }
  return s;
}

