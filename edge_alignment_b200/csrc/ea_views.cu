// Multi-camera problems at one level: every view adds its residual blocks to the same 6-DoF problem.
//
// A problem is the reference's rig / distortion flow (standalone_edge_align.cpp:791-803, 3204-3219): any number of views, each
// one AddResidualBlock loop over a camera's points (EAResidue / EAResidueEx / EAResidueSecondCam / EAResidueSecondCamEx,
// standalone/utils.h:38-421), all on one b_T_a.  ea_eval_views evaluates a problem at a pose (per-point arrays and sums);
// ea_solve_views solves it with the whole GPU in one persistent cooperative kernel (k_views_solve).  Many problems, each coarse
// to fine, are ea_views_batch.cu's: a translation unit of its own, because k_views_batch spills more when it shares the
// out-of-line LM step (ea_lm_advance_warp) with k_views_solve's register budget.
#include <algorithm>
#include <vector>

#include "ea_internal.h"
#include "ea_solve.cuh"

#define GV_THREADS 256

namespace {

// ---- one problem at one level ------------------------------------------------------------------------------------------
template <bool XYZ>
__global__ void __launch_bounds__(GV_THREADS) k_view_eval_sums(EaLevelDesc rd, EaLevelDesc nd, EaLevelGeom rg, EaLevelGeom ng, EaViewXf V,
                                                               double inv_depth_scale, ea_solve_params sp, const double* pose7,
                                                               const int* done, int j_begin, int j_end, double* sums /*[grid][EA_SUMS]*/) {
  if (done && *done) return;
  __shared__ double part[GV_THREADS / 32][EA_NSUM];
  __shared__ double cpart[GV_THREADS / 32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n = j_end - j_begin;
  const int j0 = j_begin + int((long long)n * blockIdx.x / gridDim.x), j1 = j_begin + int((long long)n * (blockIdx.x + 1) / gridDim.x);
  EaPoseG P;
  ea_pose_setup_general<XYZ>(pose7, rg, ng, V, P);
  const float2 affine = *nd.dt_affine;
  double acc64 = 0.0, cost64 = 0.0;
  ea_eval_view<1, GV_THREADS>(XYZ, rd.pts, nd.dt, affine, ng, inv_depth_scale, P, sp, j0, j1, tid, lane, acc64, cost64);
  cost64 = ea_warp_sum(cost64);
  part[warp][lane] = acc64;
  if (lane == 0) cpart[warp] = cost64;
  __syncthreads();
  if (tid < 32) {
    const double tot = ea_cta_total<GV_THREADS / 32>(part, cpart, tid);
    if (tid < EA_SUMS) sums[size_t(blockIdx.x) * EA_SUMS + tid] = tot;
  }
}

template <bool XYZ>
__global__ void __launch_bounds__(256) k_view_eval_points(EaLevelDesc rd, EaLevelDesc nd, EaLevelGeom rg, EaLevelGeom ng, EaViewXf V,
                                                          double inv_depth_scale, ea_solve_params sp, const double* pose7, int n_res,
                                                          double* raw, double* res, double* jac, int* failed) {
  EaPoseG P;
  ea_pose_setup_general<XYZ>(pose7, rg, ng, V, P);
  const float2 affine = *nd.dt_affine;
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < n_res; j += gridDim.x * blockDim.x) {
    const float4 p = EaPtStream<XYZ>::as_float4(EaPtStream<XYZ>::load(rd.pts, size_t(j) * sp.point_stride));
    float f, w, rho0, J[6];
    const bool fail = ea_point_eval_general<XYZ>(p, ng, inv_depth_scale, P, nd.dt, affine, sp.loss_type, float(sp.loss_scale), f, w, rho0, J);
    if (raw) raw[j] = double(f);
    if (res) res[j] = double(f * w);
    if (jac) for (int k = 0; k < 6; ++k) jac[size_t(j) * 6 + k] = double(J[k]);
    if (fail && failed) atomicAdd(failed, 1);
  }
}

// One cooperative kernel for the whole solve of one problem at one level (ea_solve_views): every CTA evaluates its slice of
// every view's point list, the CTA that draws the evaluation's last ticket adds the CTA totals in a fixed order, runs the
// warp-cooperative LM step and releases the next evaluation (EaGridCtl).
struct ViewDev {                  // one view, device-side (array in global memory)
  EaLevelDesc rd, nd;
  EaLevelGeom rg, ng;
  EaViewXf X;
  double inv_depth_scale;
  int n_res, xyz;
};
__global__ void __launch_bounds__(GV_THREADS, 1) k_views_solve(const ViewDev* __restrict__ views, int n_views, ea_solve_params sp, EaGridCtl* ctl,
                                                               double* partials /*[grid][32]*/) {
  constexpr int WARPS = GV_THREADS / 32;
  __shared__ double part[WARPS][EA_NSUM];
  __shared__ double cpart[WARPS];
  __shared__ double wsum[WARPS][32];
  __shared__ unsigned long long s_ticket;
  __shared__ int s_stop;
  __shared__ EaLmState s_lm;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (unsigned long long e = 1;; ++e) {
    if (ea_grid_wait(ctl, e, s_stop)) break;
    double cand[7];
#pragma unroll
    for (int i = 0; i < 7; ++i) cand[i] = __ldcg(&ctl->lm.cand[i]);      // written by the LM warp of the previous round (L2)
    double acc64 = 0.0, cost64 = 0.0;
    for (int v = 0; v < n_views; ++v) {
      const ViewDev& V = views[v];
      const int j0 = int((long long)V.n_res * blockIdx.x / gridDim.x), j1 = int((long long)V.n_res * (blockIdx.x + 1) / gridDim.x);
      if (j1 <= j0) continue;                                            // (uniform per CTA)
      EaPoseG P;
      if (V.xyz) ea_pose_setup_general<true>(cand, V.rg, V.ng, V.X, P); else ea_pose_setup_general<false>(cand, V.rg, V.ng, V.X, P);
      const float2 affine = *V.nd.dt_affine;
      ea_eval_view<1, GV_THREADS>(V.xyz, V.rd.pts, V.nd.dt, affine, V.ng, V.inv_depth_scale, P, sp, j0, j1, tid, lane, acc64, cost64);
    }
    cost64 = ea_warp_sum(cost64);
    part[warp][lane] = acc64;
    if (lane == 0) cpart[warp] = cost64;
    __syncthreads();
    if (warp == 0) {
      const double tot = ea_cta_total<WARPS>(part, cpart, lane);
      __stcg(&partials[size_t(blockIdx.x) * 32 + lane], lane < EA_SUMS ? tot : 0.0);
      __threadfence();
      __syncwarp();
      if (lane == 0) s_ticket = atomicAdd(&ctl->ticket, 1ull);
    }
    __syncthreads();
    if (s_ticket != e * gridDim.x - 1) continue;          // not the last CTA of this evaluation: wait for the next release
    // ---- last CTA: grid reduce, LM, release ----
    __threadfence();
    const double tot = ea_grid_total<WARPS>(partials, wsum, warp, lane);
    if (warp == 0) {
      wsum[0][lane] = tot;
      ea_lm_load_warp(s_lm, ctl->lm, lane);
      __syncwarp();
      const int cmd = ea_lm_advance_warp(s_lm, wsum[0], sp, lane);            // (the next candidate is left in s_lm.cand)
      __syncwarp();
      ea_lm_store_warp(ctl->lm, s_lm, lane);
      __threadfence();
      __syncwarp();
      if (lane == 0) {
        ctl->done = cmd == EA_CMD_EVAL ? 0 : 1;
        ctl->prof[4] += 1;
        __threadfence();
        ea_st_release(&ctl->go, e + 1);
      }
    }
  }
  if (s_stop == 2 && tid == 0) ctl->error = 2;   // the release never came (a CTA of this grid is gone)
}

int check_view(const ea_view& v, int level) {
  if (!v.ref || !v.now) return ea_fail(EA_ERR_INVALID_ARG, "view with a null frameset");
  if (v.ref->ctx->device != v.now->ctx->device) return ea_fail(EA_ERR_INVALID_ARG, "view framesets on different devices");
  if (level < 0 || level >= v.ref->p.n_levels || level >= v.now->p.n_levels) return ea_fail(EA_ERR_INVALID_ARG, "bad level");
  if (v.ref_slot < 0 || v.ref_slot >= v.ref->n_slots || v.now_slot < 0 || v.now_slot >= v.now->n_slots) return ea_fail(EA_ERR_INVALID_ARG, "bad slot");
  return EA_OK;
}

// Validates the views of a single-level call and counts their residuals at `level`.
int count_view_residuals(int n_views, const ea_view* views, int level, int stride, std::vector<int>& nres, int& total) {
  nres.assign(size_t(n_views), 0);
  total = 0;
  for (int i = 0; i < n_views; ++i) {
    int rc = check_view(views[i], level);
    if (rc) return rc;
    int n_pts = 0;
    rc = ea_frameset_get_num_points(views[i].ref, views[i].ref_slot, level, &n_pts);
    if (rc) return rc;
    nres[size_t(i)] = (n_pts + stride - 1) / stride;
    total += nres[size_t(i)];
  }
  return EA_OK;
}

}  // namespace

extern "C" {

int ea_eval_views(ea_context* c, int n_views, const ea_view* views, int level, const double* pose7, const ea_solve_params* sp,
                  int* n_residuals, double* raw, double* residuals, double* jac, double* sums28, int* failed) {
  if (!c || !views || n_views < 1 || !pose7 || !sp) return ea_fail(EA_ERR_INVALID_ARG, "null argument");
  { const int prc = ea_check_solve_params(sp); if (prc) return prc; }
  CU(cudaSetDevice(c->device));
  cudaStream_t st = c->stream;
  std::vector<int> nres;
  int total = 0;
  int rc = count_view_residuals(n_views, views, level, sp->point_stride, nres, total);
  if (rc) return rc;
  if (n_residuals) *n_residuals = total;
  CU(cudaMemcpyAsync(c->d_pose, pose7, 56, cudaMemcpyHostToDevice, st));
  CU(cudaMemsetAsync(c->d_failed, 0, sizeof(int), st));
  rc = ea_ensure_tmp(c, size_t(std::max(total, 1)) * 8 * sizeof(double) + size_t(n_views) * 64 * EA_SUMS * 8);
  if (rc) return rc;
  double* d_raw = (double*)c->d_tmp; double* d_res = d_raw + total; double* d_jac = d_res + total; double* d_part = d_jac + size_t(total) * 6;
  int off = 0, nb_total = 0;
  for (int i = 0; i < n_views; ++i) {
    const ea_view& v = views[i];
    const EaLevelDesc& rd = v.ref->h_desc[size_t(v.ref_slot) * EA_MAX_LEVELS + level];
    const EaLevelDesc& nd = v.now->h_desc[size_t(v.now_slot) * EA_MAX_LEVELS + level];
    EaViewXf X; ea_view_xf(v, X);
    const double ids = v.ref->inv_depth_unit;
    if (nres[i] > 0) {
      const int blocks = (nres[i] + 255) / 256;
      if (rd.pts_mode == EA_POINTS_XYZ)
        k_view_eval_points<true><<<blocks, 256, 0, st>>>(rd, nd, v.ref->geom[level], v.now->geom[level], X, ids, *sp, c->d_pose, nres[i], d_raw + off, d_res + off, d_jac + size_t(off) * 6, c->d_failed);
      else
        k_view_eval_points<false><<<blocks, 256, 0, st>>>(rd, nd, v.ref->geom[level], v.now->geom[level], X, ids, *sp, c->d_pose, nres[i], d_raw + off, d_res + off, d_jac + size_t(off) * 6, c->d_failed);
      const int nb = std::max(1, std::min(64, (nres[i] + 2047) / 2048));
      if (rd.pts_mode == EA_POINTS_XYZ)
        k_view_eval_sums<true><<<nb, GV_THREADS, 0, st>>>(rd, nd, v.ref->geom[level], v.now->geom[level], X, ids, *sp, c->d_pose, nullptr, 0, nres[i], d_part + size_t(nb_total) * EA_SUMS);
      else
        k_view_eval_sums<false><<<nb, GV_THREADS, 0, st>>>(rd, nd, v.ref->geom[level], v.now->geom[level], X, ids, *sp, c->d_pose, nullptr, 0, nres[i], d_part + size_t(nb_total) * EA_SUMS);
      c->launches += 2;
      nb_total += nb;
    }
    off += nres[i];
  }
  CU(cudaGetLastError());
  if (raw && total) CU(cudaMemcpyAsync(raw, d_raw, size_t(total) * 8, cudaMemcpyDeviceToHost, st));
  if (residuals && total) CU(cudaMemcpyAsync(residuals, d_res, size_t(total) * 8, cudaMemcpyDeviceToHost, st));
  if (jac && total) CU(cudaMemcpyAsync(jac, d_jac, size_t(total) * 48, cudaMemcpyDeviceToHost, st));
  if (failed) CU(cudaMemcpyAsync(failed, c->d_failed, sizeof(int), cudaMemcpyDeviceToHost, st));
  std::vector<double> h(size_t(std::max(nb_total, 1)) * EA_SUMS, 0.0);
  if (nb_total) CU(cudaMemcpyAsync(h.data(), d_part, size_t(nb_total) * EA_SUMS * 8, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  if (sums28) ea_fold_sums28(h.data(), nb_total, sums28);
  return EA_OK;
}

int ea_solve_views(ea_context* c, int n_views, const ea_view* views, int level, double* pose7, const ea_solve_params* sp,
                   ea_summary* summary) {
  if (!c || !views || n_views < 1 || !pose7 || !sp) return ea_fail(EA_ERR_INVALID_ARG, "null argument");
  { const int prc = ea_check_solve_params(sp); if (prc) return prc; }
  CU(cudaSetDevice(c->device));
  cudaStream_t st = c->stream;
  std::vector<int> nres;
  int total = 0;
  int rc = count_view_residuals(n_views, views, level, sp->point_stride, nres, total);
  if (rc) return rc;
  if (total == 0) {   // as ea_solve_batch: nothing to align, pose untouched, no launch
    if (summary) { *summary = ea_summary{}; summary->termination = EA_TERM_SKIPPED_NO_POINTS; }
    return EA_OK;
  }
  // One persistent cooperative kernel for the whole solve (k_views_solve).  View descriptors, control block and CTA totals live
  // in the context's scratch (allocated on first use, grown on demand): no allocation on the path of a solve.
  const int grid = std::max(1, std::min(c->sm_count, (total + 1023) / 1024));
  const size_t off_ctl = (size_t(n_views) * sizeof(ViewDev) + 255) & ~size_t(255);
  const size_t off_part = off_ctl + ((sizeof(EaGridCtl) + 255) & ~size_t(255));
  rc = ea_ensure_views(c, off_part + size_t(grid) * 32 * 8);
  if (rc) return rc;
  char* vb = static_cast<char*>(c->d_views);
  ViewDev* d_vd = reinterpret_cast<ViewDev*>(vb);
  EaGridCtl* d_ctl = reinterpret_cast<EaGridCtl*>(vb + off_ctl);
  double* d_partials = reinterpret_cast<double*>(vb + off_part);
  std::vector<ViewDev> hv(static_cast<size_t>(n_views));
  for (int i = 0; i < n_views; ++i) {
    const ea_view& v = views[i];
    ViewDev& D = hv[size_t(i)];
    D.rd = v.ref->h_desc[size_t(v.ref_slot) * EA_MAX_LEVELS + level];
    D.nd = v.now->h_desc[size_t(v.now_slot) * EA_MAX_LEVELS + level];
    D.rg = v.ref->geom[level]; D.ng = v.now->geom[level];
    ea_view_xf(v, D.X);
    D.inv_depth_scale = v.ref->inv_depth_unit;
    D.n_res = nres[i]; D.xyz = D.rd.pts_mode == EA_POINTS_XYZ ? 1 : 0;
  }
  CU(cudaMemcpyAsync(d_vd, hv.data(), hv.size() * sizeof(ViewDev), cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(c->d_pose, pose7, 56, cudaMemcpyHostToDevice, st));
  k_shard_ctl_init<<<1, 1, 0, st>>>(d_ctl, c->d_pose, hv[0].rg, hv[0].ng, hv[0].xyz);
  ea_solve_params spv = *sp;
  const ViewDev* vd_arg = d_vd; int nv = n_views;
  void* args[] = {&vd_arg, &nv, &spv, &d_ctl, &d_partials};
  cudaError_t le = cudaLaunchCooperativeKernel((const void*)k_views_solve, dim3(unsigned(grid)), dim3(GV_THREADS), args, 0, st);
  c->launches += 2;
  if (le != cudaSuccess) return ea_fail(EA_ERR_CUDA, "views solve launch: %s", cudaGetErrorString(le));
  EaGridCtl h;
  CU(cudaMemcpyAsync(&h, d_ctl, sizeof h, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));      // (hv must outlive the upload)
  if (h.error) return ea_fail(EA_ERR_CUDA, "views solve: the persistent kernel lost a CTA (bounded wait expired)");
  for (int i = 0; i < 7; ++i) pose7[i] = h.lm.x[i];
  if (summary) {
    *summary = ea_lm_summary(h.lm, total, 0);
    summary->termination = h.done ? h.lm.term : EA_TERM_NO_CONVERGENCE;
  }
  return EA_OK;
}

}  // extern "C"
