// Many multi-camera problems, each solved coarse to fine, in one persistent launch (ea_solve_views_batch).
//
// A problem is the reference's rig / distortion flow (standalone_edge_align.cpp:791-803, 3204-3219): any number of views, each
// one AddResidualBlock loop over a camera's points (EAResidue / EAResidueEx / EAResidueSecondCam / EAResidueSecondCamEx,
// standalone/utils.h:38-421), all on one b_T_a.  ea_solve_views solves one problem at one level with the whole GPU; this
// scheduler gives the multi-camera problems what ea_k_solve_batch gives single-camera pairs:
//
//   order     k_vb_order sorts the problems by their residuals at the finest solved level (device-resident point counts, no
//             host read-back), largest first, ties by index
//   queue     one persistent CTA per problem: a CTA takes the next problem from an atomic ticket and runs its whole pyramid
//   boss      warp 0 runs the warp-cooperative LM step (ea_lm_advance_warp) on the state in shared memory, folds the candidate
//             pose once per view (ea_pose_setup_general, one lane per view) and handles the level / problem transitions
//   evaluate  all warps walk the problem's views in order (ea_eval_view); a view's residuals are cut into tiles of THREADS x 16:
//             per lane 16 points in fp32, the transposing warp butterfly, fp64 per-warp slots, CTA totals in fixed warp order
//
// The sums of a problem depend only on its views and VB_THREADS: not on the CTA that ran it, the batch or the order.
#include <algorithm>
#include <cstring>
#include <vector>

#include "ea_internal.h"
#include "ea_solve.cuh"

#define VB_THREADS 256
#define VB_MIN_CTAS 2          // 2 x 256 threads at 128 registers fill an SM; one problem's LM step overlaps the other's sweep
#define VB_TILE_ITERS 16       // points per lane between two fp32 -> fp64 flushes (EA_FLUSH_EVERY of the production loop)
#define VB_CMD_EXIT 2
#define VB_SORT_SMEM 4096      // problems sorted in shared memory; larger batches sort in global scratch

namespace {

struct VbView {                       // one view, all levels (device array built by the host)
  EaLevelDesc rd[EA_MAX_LEVELS], nd[EA_MAX_LEVELS];
  EaLevelGeom rg[EA_MAX_LEVELS], ng[EA_MAX_LEVELS];
  int ref_cap[EA_MAX_LEVELS];         // point-list capacity of the reference level (guards a truncated list)
  EaViewXf X;
  double inv_depth_scale;
};

struct VbArgs {
  const VbView* views;                // [total views]
  const int32_t* offsets;             // [n + 1]: problem i is views[offsets[i] .. offsets[i + 1])
  const int32_t* order;               // [n]: queue order (k_vb_order)
  double* poses;                      // [n][7] in/out
  ea_summary* summaries;              // [n][n_levels], zeroed by the host
  int* work_counter;                  // zeroed by the host
  int n_problems, n_levels, coarsest, finest;
  ea_solve_params sp;
};

struct VbLive {                       // one view of the (problem, level) in flight
  const void* pts;
  const float* dt;
  float2 affine;
  int n_res, xyz;
  double inv_depth_scale;
  EaLevelGeom rg, ng;
  EaViewXf X;
};

struct VbSmem {
  EaPoseG P[EA_MAX_VIEWS_PER_PROBLEM];        // the candidate folded per view (boss warp, one lane per view)
  VbLive live[EA_MAX_VIEWS_PER_PROBLEM];
  double part[VB_THREADS / 32][EA_NSUM];      // per warp: lane-slot sums
  double cpart[VB_THREADS / 32];              // per warp: cost
  double sums[32];                            // evaluation totals
  EaLmState lm;
  // the kernel's arguments: a __grid_constant__ parameter whose address reaches a non-inlined function is first copied to local
  // memory (ea_solve.cu, EaSolveSmem::args); the boss functions read this copy
  VbArgs args;
  int problem, level, v0, nv, n_res, truncated, cmd;
};

// Boss warp: the candidate S.lm.cand folded with each view's rig transform and intrinsics, lane v for view v.  Out of line: its
// fp64 temporaries would otherwise share the kernel's register budget with the evaluation loop.
__device__ __noinline__ void vb_fold(VbSmem& S, const int lane) {
  if (lane < S.nv) {
    const VbLive& Lv = S.live[lane];
    if (Lv.xyz) ea_pose_setup_general<true>(S.lm.cand, Lv.rg, Lv.ng, Lv.X, S.P[lane]);
    else ea_pose_setup_general<false>(S.lm.cand, Lv.rg, Lv.ng, Lv.X, S.P[lane]);
  }
  __syncwarp();
}

// Boss warp: move to the next (problem, level) with residuals and set up its first evaluation, or VB_CMD_EXIT.
__device__ __noinline__ void vb_boss_next(const VbArgs& A, VbSmem& S, const int lane, bool new_problem) {
  const unsigned full = 0xffffffffu;
  for (;;) {
    if (new_problem) {
      int t = 0;
      if (lane == 0) t = atomicAdd(A.work_counter, 1);
      t = __shfl_sync(full, t, 0);
      if (t >= A.n_problems) { if (lane == 0) S.cmd = VB_CMD_EXIT; __syncwarp(); return; }
      const int p = A.order[t];
      if (lane < 7) S.lm.x[lane] = A.poses[size_t(p) * 7 + lane];
      if (lane == 0) { S.problem = p; S.level = A.coarsest; S.v0 = A.offsets[p]; S.nv = A.offsets[p + 1] - A.offsets[p]; }
      __syncwarp();
      new_problem = false;
    }
    const int p = S.problem, level = S.level, nv = S.nv;
    if (level < A.finest) {       // problem finished: write its pose back, fetch another
      if (lane < 7) A.poses[size_t(p) * 7 + lane] = S.lm.x[lane];
      __syncwarp();
      new_problem = true;
      continue;
    }
    int n_res = 0, trunc = 0;
    if (lane < nv) {              // lane v: view v's residual count (device-resident, as ea_boss_next) and level data
      const VbView& V = A.views[S.v0 + lane];
      const EaLevelDesc rd = V.rd[level];
      const int n_pts = min(*rd.n_pts, V.ref_cap[level]);
      n_res = (n_pts + A.sp.point_stride - 1) / A.sp.point_stride;
      trunc = *rd.truncated;
      VbLive& Lv = S.live[lane];
      Lv.pts = rd.pts; Lv.dt = V.nd[level].dt; Lv.affine = *V.nd[level].dt_affine; Lv.n_res = n_res;
      Lv.xyz = rd.pts_mode == EA_POINTS_XYZ ? 1 : 0; Lv.inv_depth_scale = V.inv_depth_scale;
      Lv.rg = V.rg[level]; Lv.ng = V.ng[level]; Lv.X = V.X;
    }
    const int total = __reduce_add_sync(full, n_res);
    trunc = __any_sync(full, trunc);
    if (total == 0) {             // nothing to align at this level: the pose passes through
      if (lane == 0) {
        ea_summary z = {};
        z.termination = EA_TERM_SKIPPED_NO_POINTS; z.truncated = trunc;
        A.summaries[size_t(p) * A.n_levels + level] = z;
        S.level = level - 1;
      }
      __syncwarp();
      continue;
    }
    if (lane == 0) {
      ea_lm_restart(S.lm);
      S.n_res = total; S.truncated = trunc; S.cmd = EA_CMD_EVAL;
    }
    if (lane < 7) S.lm.cand[lane] = S.lm.x[lane];
    __syncwarp();
    vb_fold(S, lane);
    return;
  }
}

template <int THREADS>
__global__ void __launch_bounds__(THREADS, VB_MIN_CTAS) k_views_batch(const __grid_constant__ VbArgs A) {
  constexpr int WARPS = THREADS / 32;
  __shared__ VbSmem S;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) S.args = A;
  __syncthreads();
  if (warp == 0) vb_boss_next(S.args, S, lane, true);
  __syncthreads();
  for (;;) {
    if (S.cmd == VB_CMD_EXIT) break;
    // ---- one evaluation of the problem at the candidate: every view in order ----
    double acc64 = 0.0, cost64 = 0.0;
    const int nv = S.nv;
    for (int v = 0; v < nv; ++v) {
      const VbLive& Lv = S.live[v];
      if (Lv.n_res == 0) continue;
      if (Lv.xyz) ea_eval_view<VB_TILE_ITERS, THREADS>(true, Lv.pts, Lv.dt, Lv.affine, Lv.ng, Lv.inv_depth_scale, S.P[v], A.sp, 0, Lv.n_res, tid, lane, acc64, cost64);
      else ea_eval_view<VB_TILE_ITERS, THREADS>(false, Lv.pts, Lv.dt, Lv.affine, Lv.ng, Lv.inv_depth_scale, S.P[v], A.sp, 0, Lv.n_res, tid, lane, acc64, cost64);
    }
    cost64 = ea_warp_sum(cost64);
    S.part[warp][lane] = acc64;
    if (lane == 0) S.cpart[warp] = cost64;
    __syncthreads();
    // ---- boss warp: CTA totals, LM step, next candidate or next (problem, level) ----
    if (warp == 0) {
      const double tot = ea_cta_total<WARPS>(S.part, S.cpart, lane);
      S.sums[lane] = lane < EA_SUMS ? tot : 0.0;
      __syncwarp();
      const int level = S.level;
      const int cmd = ea_lm_advance_warp(S.lm, S.sums, S.args.sp, lane);
      if (cmd == EA_CMD_EVAL) {
        vb_fold(S, lane);
      } else {
        if (lane == 0) {
          A.summaries[size_t(S.problem) * A.n_levels + level] = ea_lm_summary(S.lm, S.n_res, S.truncated);
          S.level = level - 1;
        }
        __syncwarp();
        vb_boss_next(S.args, S, lane, false);
      }
    }
    __syncthreads();
  }
}

// Queue order: problems by decreasing residuals at the finest solved level, ties by index.  One CTA, bitonic sort of
// (work << 32 | ~index) keys; shared memory up to VB_SORT_SMEM problems, the scratch `gkeys` [m] beyond.
__global__ void __launch_bounds__(1024) k_vb_order(const VbView* __restrict__ views, const int32_t* __restrict__ offsets, int n, int finest,
                                                   int stride, unsigned long long* gkeys, int32_t* __restrict__ order) {
  __shared__ unsigned long long skeys[VB_SORT_SMEM];
  int m = 1;
  while (m < n) m <<= 1;
  unsigned long long* key = m <= VB_SORT_SMEM ? skeys : gkeys;
  for (int i = threadIdx.x; i < m; i += blockDim.x) {
    unsigned long long k = 0;
    if (i < n) {
      unsigned long long work = 0;
      for (int v = offsets[i]; v < offsets[i + 1]; ++v) {
        const EaLevelDesc& rd = views[v].rd[finest];
        const int n_pts = min(*rd.n_pts, views[v].ref_cap[finest]);
        work += (unsigned long long)((n_pts + stride - 1) / stride);
      }
      k = (work << 32) | (unsigned long long)(0xFFFFFFFFu - unsigned(i));
    }
    key[i] = k;
  }
  __syncthreads();
  ea_cta_sort_desc(key, m);
  for (int i = threadIdx.x; i < n; i += blockDim.x) order[i] = int32_t(0xFFFFFFFFu - unsigned(key[i] & 0xFFFFFFFFull));
}

size_t vb_align(size_t x) { return (x + 255) & ~size_t(255); }

int vb_check_view(const ea_context* c, const ea_view& v, int p, int k) {
  if (!v.ref || !v.now) return ea_fail(EA_ERR_INVALID_ARG, "problem %d, view %d: null frameset", p, k);
  if (v.ref->ctx->device != c->device || v.now->ctx->device != c->device)
    return ea_fail(EA_ERR_INVALID_ARG, "problem %d, view %d: a frameset lives on another device", p, k);
  if (v.ref_slot < 0 || v.ref_slot >= v.ref->n_slots || v.now_slot < 0 || v.now_slot >= v.now->n_slots)
    return ea_fail(EA_ERR_INVALID_ARG, "problem %d, view %d: bad slot", p, k);
  return EA_OK;
}

}  // namespace

extern "C" int ea_solve_views_batch(ea_context* c, int n, const int32_t* view_offsets, const ea_view* views, double* poses7,
                                    const ea_solve_params* sp, ea_summary* summaries) {
  if (!c) return ea_fail(EA_ERR_INVALID_ARG, "null context");
  if (n == 0) return EA_OK;
  if (n < 0 || !view_offsets || !views || !poses7) return ea_fail(EA_ERR_INVALID_ARG, "null argument or negative problem count");
  int rc = ea_check_solve_params(sp);
  if (rc) return rc;
  // ---- validation: nothing is launched and no pose is touched unless the whole call is valid ----
  if (view_offsets[0] != 0) return ea_fail(EA_ERR_INVALID_ARG, "view_offsets[0] must be 0");
  for (int i = 0; i < n; ++i) {
    const int k = view_offsets[i + 1] - view_offsets[i];
    if (k < 1 || k > EA_MAX_VIEWS_PER_PROBLEM)
      return ea_fail(EA_ERR_INVALID_ARG, "problem %d has %d views (1..%d; view_offsets must increase)", i, k, EA_MAX_VIEWS_PER_PROBLEM);
  }
  const int n_views = view_offsets[n];
  const int L = views[0].ref ? views[0].ref->p.n_levels : 0;
  for (int i = 0; i < n; ++i)
    for (int v = view_offsets[i]; v < view_offsets[i + 1]; ++v) {
      rc = vb_check_view(c, views[v], i, v - view_offsets[i]);
      if (rc) return rc;
      if (views[v].ref->p.n_levels != L || views[v].now->p.n_levels != L)
        return ea_fail(EA_ERR_INVALID_ARG, "problem %d, view %d: framesets differ in n_levels", i, v - view_offsets[i]);
    }
  const int coarsest = sp->coarsest_level < 0 ? L - 1 : sp->coarsest_level, finest = sp->finest_level;
  if (coarsest >= L || finest < 0 || finest > coarsest) return ea_fail(EA_ERR_INVALID_ARG, "bad level range [%d..%d]", coarsest, finest);
  for (int i = 0; i < n; ++i) {
    double q2 = 0;
    for (int k = 0; k < 4; ++k) q2 += poses7[i * 7 + k] * poses7[i * 7 + k];
    if (!(q2 > 0.999999 && q2 < 1.000001)) return ea_fail(EA_ERR_INVALID_ARG, "problem %d: quaternion is not unit (|q|^2=%g)", i, q2);
  }
  CU(cudaSetDevice(c->device));
  cudaStream_t st = c->stream;
  // ---- scratch (the context's views buffer, grown on demand): descriptors, offsets, order, poses, summaries, counter, keys ----
  int m = 1;
  while (m < n) m <<= 1;
  const size_t off_off = vb_align(size_t(n_views) * sizeof(VbView));
  const size_t off_ord = off_off + vb_align(size_t(n + 1) * sizeof(int32_t));
  const size_t off_pose = off_ord + vb_align(size_t(n) * sizeof(int32_t));
  const size_t off_sum = off_pose + vb_align(size_t(n) * 7 * sizeof(double));
  const size_t off_work = off_sum + vb_align(size_t(n) * L * sizeof(ea_summary));
  const size_t off_keys = off_work + 256;
  const size_t need = off_keys + (m > VB_SORT_SMEM ? size_t(m) * sizeof(unsigned long long) : 0);
  rc = ea_ensure_views(c, need);
  if (rc) return rc;
  char* base = static_cast<char*>(c->d_views);
  VbArgs A;
  std::memset(&A, 0, sizeof A);
  VbView* d_vw = reinterpret_cast<VbView*>(base);
  int32_t* d_off = reinterpret_cast<int32_t*>(base + off_off);
  int32_t* d_ord = reinterpret_cast<int32_t*>(base + off_ord);
  A.views = d_vw; A.offsets = d_off; A.order = d_ord;
  A.poses = reinterpret_cast<double*>(base + off_pose);
  A.summaries = reinterpret_cast<ea_summary*>(base + off_sum);
  A.work_counter = reinterpret_cast<int*>(base + off_work);
  A.n_problems = n; A.n_levels = L; A.coarsest = coarsest; A.finest = finest; A.sp = *sp;
  unsigned long long* d_keys = reinterpret_cast<unsigned long long*>(base + off_keys);
  std::vector<VbView> hv(static_cast<size_t>(n_views));
  for (int v = 0; v < n_views; ++v) {
    const ea_view& w = views[v];
    VbView& D = hv[size_t(v)];
    std::memset(&D, 0, sizeof D);
    for (int l = 0; l < L; ++l) {
      D.rd[l] = w.ref->h_desc[size_t(w.ref_slot) * EA_MAX_LEVELS + l];
      D.nd[l] = w.now->h_desc[size_t(w.now_slot) * EA_MAX_LEVELS + l];
      D.rg[l] = w.ref->geom[l]; D.ng[l] = w.now->geom[l];
      D.ref_cap[l] = w.ref->lv[l].cap;
    }
    ea_view_xf(w, D.X);
    D.inv_depth_scale = w.ref->inv_depth_unit;
  }
  CU(cudaMemcpyAsync(d_vw, hv.data(), hv.size() * sizeof(VbView), cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(d_off, view_offsets, size_t(n + 1) * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(A.poses, poses7, size_t(n) * 7 * sizeof(double), cudaMemcpyHostToDevice, st));
  CU(cudaMemsetAsync(A.summaries, 0, size_t(n) * L * sizeof(ea_summary), st));
  CU(cudaMemsetAsync(A.work_counter, 0, sizeof(int), st));
  int per_sm = 0;
  CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_views_batch<VB_THREADS>, VB_THREADS, 0));
  const int grid = std::max(1, std::min(n, c->sm_count * std::max(per_sm, 1)));
  {
    EaProfileScope prof(c, 1);
    k_vb_order<<<1, 1024, 0, st>>>(d_vw, d_off, n, finest, sp->point_stride, d_keys, d_ord);
    k_views_batch<VB_THREADS><<<grid, VB_THREADS, 0, st>>>(A);
  }
  c->launches += 2;
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(poses7, A.poses, size_t(n) * 7 * sizeof(double), cudaMemcpyDeviceToHost, st));
  if (summaries) CU(cudaMemcpyAsync(summaries, A.summaries, size_t(n) * L * sizeof(ea_summary), cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));      // (hv must outlive the upload)
  // ---- truncated reference lists among the solved levels: results are written, the call reports the first one ----
  std::vector<const ea_frameset*> seen;
  std::vector<std::vector<int>> ovf;
  for (int i = 0; i < n; ++i)
    for (int v = view_offsets[i]; v < view_offsets[i + 1]; ++v) {
      const ea_frameset* fs = views[v].ref;
      size_t k = std::find(seen.begin(), seen.end(), fs) - seen.begin();
      if (k == seen.size()) {
        seen.push_back(fs);
        ovf.emplace_back(size_t(fs->n_slots) * EA_MAX_LEVELS);
        CU(cudaMemcpy(ovf.back().data(), fs->d_overflow, ovf.back().size() * sizeof(int), cudaMemcpyDeviceToHost));
      }
      for (int l = finest; l <= coarsest; ++l)
        if (ovf[k][size_t(views[v].ref_slot) * EA_MAX_LEVELS + l])
          return ea_fail(EA_ERR_CAPACITY, "problem %d, view %d: the reference point list (slot %d, level %d) was truncated at max_points; "
                         "result uses the truncated list", i, v - view_offsets[i], views[v].ref_slot, l);
    }
  return EA_OK;
}
