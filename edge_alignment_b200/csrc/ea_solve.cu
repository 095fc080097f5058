// Fused residual / analytic-Jacobian / normal-equation kernels and the persistent on-device
// Levenberg-Marquardt solve.  One thread-block cluster (1..8 CTAs, DSMEM reduction) owns one
// frame pair for its whole coarse-to-fine solve: no host round trip per iteration.
//
// Replaces, for n pairs at once: the residual-block loop + ceres::Solve of
// standalone_edge_align.cpp:265-291 (and src/SolveEA.cpp:163-198).
//
// Control flow: the "boss" (thread 0 of cluster rank 0) owns the LM state machine and the work queue.  Every loop
// iteration of every CTA is exactly one evaluation: read the boss's message {point list, DT, candidate pose}, reduce
// the CTA's slice of the points to 29 sums, hand them to the boss, who advances LM / the pyramid level / the pair
// and publishes the next message.  Messages are parity double-buffered, so two barriers per evaluation suffice.
// Several small CTAs share an SM, so one pair's serial LM step overlaps the other pairs' evaluations.
#include <cooperative_groups.h>

#include "ea_internal.h"
#include <cstdlib>

#include "ea_solve.cuh"

namespace cg = cooperative_groups;

#define EA_SOLVE_WARPS (EA_SOLVE_THREADS / 32)
#ifndef EA_SOLVE_MIN_CTAS
#define EA_SOLVE_MIN_CTAS 1
#endif
// points per thread between fp32->fp64 flushes of the normal-equation slots
#define EA_CMD_EXIT 2

struct EaMsg {  // boss -> all threads of the cluster
  // -- constant over the evaluations of one (pair, level): 5 eight-byte words
  const void* pts;
  const float* dt;     // first element of the padded distance transform (pixel (-PAD, -PAD)): offsets from it are unsigned
  float2 affine;
  int n_res, level, pts_mode, cmd;
  // -- per evaluation
  int rev;        // sweep direction of this evaluation: alternates per evaluation of the (pair, level), see ea_eval_slice
  int same;       // this evaluation continues the previous one's (pair, level) with the same chunk range: the points prefetched before the barrier are its first
  int nh, pad;    // tail helpers sharing this evaluation (0: the owner evaluates every chunk)
  EaPose P;       // the candidate pose folded with the level's intrinsics (ea_pose_setup): computed once, by the boss
};
#define EA_MSG_FIXED_WORDS 5
static_assert(sizeof(EaMsg) % 8 == 0, "EaMsg is copied as 8-byte words");

// ---- tail helpers -------------------------------------------------------------------------------------------------------
// One pair per persistent CTA leaves the SMs idle once the work queue is empty while the last, longest pairs finish (measured:
// 29 % of the launch; a single pair that runs to the iteration limit can outweigh a CTA's whole mean load).  A CTA that finds
// the queue empty therefore becomes a HELPER: it registers on the board of a CTA that still owns a pair and from then on
// evaluates a share of the chunks of every evaluation the owner publishes there, delivering chunk totals the owner adds in
// chunk order -- the sums are the same whoever computed them (ea_chunking).  Owner and helpers talk through global memory
// only: release / acquire on an epoch word, bounded spins.
#define EA_MAX_HELPERS (EA_MAX_CHUNKS - 1)
#define EA_BOARD_EXIT (~0ull)
#define EA_BOARD_SPIN_LIMIT (1ll << 22)
struct EaHelpBoard {                          // one per persistent CTA; zeroed by the host before every launch
  unsigned long long word;                    // (epoch << 8) | helpers sharing that evaluation; EA_BOARD_EXIT: the owner is done
  int n_helpers;                              // registered helpers (atomicAdd by the helpers)
  int busy;                                   // the CTA owns a pair
  unsigned long long done[EA_MAX_HELPERS];    // per helper: epoch of the evaluation it last delivered
  double chunk[EA_MAX_CHUNKS][32];            // chunk totals written by the helpers
  EaMsg msg;                                  // the evaluation being shared
};

struct alignas(2 * EA_STAGE_SLOT * 8) EaSolveSmem {
  uint2 stage[2][EA_STAGE_SLOT];            // cp.async staging of the point stream (ea_eval_slice: aligned to its own size, first member)
  // the kernel's arguments, for the boss functions: a __grid_constant__ parameter whose address is handed to a non-inlined
  // function is copied to LOCAL memory first, and every access from the serial LM section then misses the L1 that the
  // evaluation loop has just swept (measured: the LM step was ~4x slower than its dependency chains).  Shared memory is not
  // evicted.  The inlined hot path keeps reading A from the constant bank.
  EaSolveArgs args;
  EaMsg msg[2];
  double part[EA_MAX_CHUNKS][EA_SOLVE_WARPS][EA_NSUM];     // per chunk, per warp: lane-slot sums
  double cpart[EA_MAX_CHUNKS][EA_SOLVE_WARPS];             // per chunk, per warp: cost
  double sums[EA_SUMS + 3];                 // evaluation totals
  double cluster_sums[8][EA_SUMS + 3];      // rank 0 only: one row per cluster rank
  EaLmState lm;                             // boss only
  int pair, level, truncated;               // boss only
  unsigned long long help_epoch;            // owner: evaluations published on its board so far
  int help_owner, help_index, help_fail;    // helper: the board it serves and its slot there (1-based); owner: a helper went missing
  long long dbg[6], dbg_t, dbg_t0;          // EA_SOLVE_DEBUG cycle counters (thread 0)
};

// Boss: move to the next (pair, level) that has points and publish its first evaluation, or EXIT.
template <bool INL>
__device__ __forceinline__ void ea_boss_next_impl(const EaSolveArgs& A, EaSolveSmem& S, EaMsg& out, bool new_pair_needed) {
  for (;;) {
    if (new_pair_needed) {
      const int ticket = atomicAdd(A.work_counter, 1);
      if (ticket >= A.n_pairs) { out.cmd = EA_CMD_EXIT; S.pair = -1; return; }
      const int pair = A.order ? A.order[ticket] : ticket;   // longest-expected-first when the caller knows better
      S.pair = pair; S.level = A.coarsest;
      const int pi = A.pose_index ? A.pose_index[pair] : pair;
#pragma unroll 1
      for (int i = 0; i < 7; ++i) S.lm.x[i] = A.poses[size_t(pi) * 7 + i];
      new_pair_needed = false;
    }
    const int pair = S.pair, level = S.level;
    if (level < A.finest) {  // pair finished: write the pose back, fetch another
      const int pi = A.pose_index ? A.pose_index[pair] : pair;
#pragma unroll 1
      for (int i = 0; i < 7; ++i) A.poses[size_t(pi) * 7 + i] = S.lm.x[i];
      new_pair_needed = true;
      continue;
    }
    const EaLevelDesc rd = A.ref_desc[size_t(A.ref_slots[pair]) * EA_MAX_LEVELS + level];
    const EaLevelDesc nd = A.now_desc[size_t(A.now_slots[pair]) * EA_MAX_LEVELS + level];
    const int n_pts = min(*rd.n_pts, A.ref_cap[level]);
    const int n_res = (n_pts + A.sp.point_stride - 1) / A.sp.point_stride;
    S.truncated = *rd.truncated;
    if (n_res == 0) {
      if (A.summaries) { ea_summary z = {}; z.termination = EA_TERM_SKIPPED_NO_POINTS; A.summaries[size_t(pair) * A.n_levels + level] = z; }
      S.level = level - 1;
      continue;
    }
    EaLmState& L = S.lm;
    L.phase = 0; L.iter = 0; L.accepted = 0; L.rejected = 0; L.invalid_run = 0; L.evals = 0; L.term = EA_TERM_NONE;
#pragma unroll 1
    for (int i = 0; i < 7; ++i) L.cand[i] = L.x[i];
    if (rd.pts_mode == EA_POINTS_XYZ) ea_pose_setup<true>(L.cand, A.ref_geom[level], A.now_geom[level], out.P);
    else ea_pose_setup<false>(L.cand, A.ref_geom[level], A.now_geom[level], out.P);
    out.pts = rd.pts; out.dt = nd.dt - ea_dt_origin_offset(nd.w); out.affine = *nd.dt_affine; out.n_res = n_res; out.level = level; out.pts_mode = rd.pts_mode; out.cmd = EA_CMD_EVAL; out.rev = 0; out.same = 0; out.nh = 0; out.pad = 0;
    return;
  }
}

// Boss: consume the sums of one evaluation; fills `out` with the next message.
__device__ __noinline__ void ea_boss_next(const EaSolveArgs& A, EaSolveSmem& S, EaMsg& out, bool new_pair_needed) { ea_boss_next_impl<false>(A, S, out, new_pair_needed); }

// Boss warp (all 32 lanes): consume the sums of one evaluation (S.sums) and write the next message into `out` (shared
// memory).  The LM step itself is warp-cooperative (ea_lm_advance_warp); level / pair changes stay on lane 0.  Inlined into
// warp 0's branch of the kernel: as a call it received its arguments and the kernel's live values through the stack frame.
__device__ __forceinline__ void ea_boss_step_warp(const EaSolveArgs& A, EaSolveSmem& S, const EaMsg& cur, EaMsg& out, const int lane) {
  const int acc0 = S.lm.accepted, rej0 = S.lm.rejected;
#ifdef EA_LM_PROFILE
  const long long t_in = clock64();
#endif
  const int cmd = ea_lm_advance_warp(S.lm, S.sums, A.sp, lane);
#ifdef EA_LM_PROFILE
  __syncwarp();
  if (lane == 0) { S.lm.prof[6] += clock64() - t_in; S.lm.prof[7] += 1; }
  __syncwarp();
#endif
  if (A.trace && lane == 0) {   // iteration log of a single-pair solve (ea_solve_traced): what Ceres prints with minimizer_progress_to_stdout
    const int k = (*A.trace_count)++;
    if (k < A.trace_cap) {
      double* r = A.trace + size_t(k) * EA_TRACE_DOUBLES;
      r[0] = cur.level; r[1] = S.lm.accepted + S.lm.rejected; r[2] = S.lm.cost; r[3] = S.sums[28]; r[4] = S.lm.radius;
      r[5] = S.lm.accepted > acc0 ? 1.0 : (S.lm.rejected > rej0 ? 0.0 : -1.0);   // accepted / rejected / no decision (first evaluation, termination)
    }
  }
  if (cmd == EA_CMD_EVAL) {
    // the same (pair, level) again at the new candidate: the fixed words are copied by lanes 0..4, every lane folds the pose
    // (no divergence), lane 0 stores it
    EaPose P;
    if (cur.pts_mode == EA_POINTS_XYZ) ea_pose_setup<true>(S.lm.cand, A.ref_geom[cur.level], A.now_geom[cur.level], P);
    else ea_pose_setup<false>(S.lm.cand, A.ref_geom[cur.level], A.now_geom[cur.level], P);
    if (lane < EA_MSG_FIXED_WORDS) reinterpret_cast<unsigned long long*>(&out)[lane] = reinterpret_cast<const unsigned long long*>(&cur)[lane];
    if (lane == 5) { out.rev = S.lm.evals & 1; out.same = 1; out.nh = 0; out.pad = 0; }
    if (lane == 0) out.P = P;
    __syncwarp();
    return;
  }
  if (lane == 0) {
    if (A.summaries) {
      const EaLmState& L = S.lm;
      ea_summary z;
      z.termination = L.term; z.iterations = L.iter; z.accepted = L.accepted; z.rejected = L.rejected;
      z.n_residuals = cur.n_res; z.evaluations = L.evals; z.initial_cost = L.initial_cost; z.final_cost = L.cost;
      z.truncated = S.truncated; z.reserved = 0;
      A.summaries[size_t(S.pair) * A.n_levels + cur.level] = z;
    }
    S.level = cur.level - 1;
    ea_boss_next(A, S, out, false);
  }
  __syncwarp();
}


__device__ __forceinline__ unsigned long long ea_ld_acquire(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void ea_st_release(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// One worker's share of an evaluation: chunks [cb, ce) of M, walked in M's direction; per-chunk partials into S.part / S.cpart.
// chain_next_eval: the same CTA evaluates the same chunks of the next evaluation of this (pair, level): prefetch its first point.
template <int THREADS>
__device__ __forceinline__ void ea_eval_chunks(const EaSolveArgs& A, EaSolveSmem& S, const EaMsg& M, const EaPose& P, const int cb, const int ce,
                                               const int chunk, const bool pre_valid, const bool chain_next_eval) {
  const EaLevelGeom& ng = A.now_geom[M.level];
  const bool rev = EA_ALTERNATE_SWEEP && M.rev, nrev = EA_ALTERNATE_SWEEP ? !rev : rev;
  const int lo = cb * chunk, hi = min(ce * chunk, M.n_res);
  if (M.pts_mode == EA_POINTS_XYZ)
    ea_eval_slice<true, THREADS>(M.pts, M.dt, M.affine, ng, A.inv_depth_scale, A.loss, A.sp.point_stride, P, lo, hi, S.part[cb], S.cpart[cb], rev, nullptr, false, false, false,
                                 chunk / THREADS, THREADS / 32);
  else
    ea_eval_slice<false, THREADS>(M.pts, M.dt, M.affine, ng, A.inv_depth_scale, A.loss, A.sp.point_stride, P, lo, hi, S.part[cb], S.cpart[cb], rev, &S.stage[0][0], pre_valid, chain_next_eval, nrev,
                                  chunk / THREADS, THREADS / 32);
}

template <int THREADS, bool CLUSTER>
__global__ void __launch_bounds__(THREADS, EA_SOLVE_MIN_CTAS) ea_k_solve_batch(const __grid_constant__ EaSolveArgs A) {
  __shared__ EaSolveSmem S;
  cg::cluster_group cluster = cg::this_cluster();
  const unsigned crank = CLUSTER ? cluster.block_rank() : 0u;
  const unsigned csize = CLUSTER ? cluster.num_blocks() : 1u;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const bool boss = (crank == 0 && tid == 0);
  const bool helpers_on = !CLUSTER && A.boards != nullptr;
  EaHelpBoard* const my_board = helpers_on ? A.boards + blockIdx.x : nullptr;
  auto sync_all = [&]() { if (CLUSTER) cluster.sync(); else __syncthreads(); };
  auto publish = [&](const EaMsg& m, unsigned slot) {
    for (unsigned r = 0; r < csize; ++r) {
      EaSolveSmem* Sr = CLUSTER ? cluster.map_shared_rank(&S, r) : &S;
      Sr->msg[slot] = m;
    }
  };
  unsigned g = 0;
  if (tid == 0) S.args = A;
  __syncthreads();
  if (boss) {
    EaMsg m;
    S.help_epoch = 0; S.help_fail = 0;
    ea_boss_next(S.args, S, m, true);
    if (helpers_on && m.cmd != EA_CMD_EXIT) { *reinterpret_cast<volatile int*>(&my_board->busy) = 1; __threadfence(); }
    publish(m, 0);
  }
  sync_all();
  // EA_SOLVE_DEBUG=1: where the boss thread's cycles go {evaluation, wait + totals, LM step, second wait, evaluations, lifetime}
  // (counters live in shared memory: the evaluation loop has no registers to spare)
  const bool dbg_on = A.debug != nullptr && tid == 0;
  if (dbg_on) { for (int k = 0; k < 6; ++k) S.dbg[k] = 0; S.dbg_t0 = clock64(); S.dbg_t = S.dbg_t0; }
#ifdef EA_LM_PROFILE
  if (tid == 0) for (int k = 0; k < 8; ++k) S.lm.prof[k] = 0;
#endif
  auto lap = [&](int k) { if (dbg_on) { const long long t = clock64(); S.dbg[k] += t - S.dbg_t; S.dbg_t = t; } };
  // ================================================= owner loop =================================================
  for (;;) {
    const EaMsg& M = S.msg[g & 1];
    if (M.cmd == EA_CMD_EXIT) break;
    const EaPose P = M.P;
    int chunk = 0, K = 1, cb = 0;
    if (CLUSTER) {
      // a cluster shares the evaluation by rank: one slice, one partial per CTA
      const int j0 = int((long long)M.n_res * crank / csize), j1 = int((long long)M.n_res * (crank + 1) / csize);
      const EaLevelGeom& ng = A.now_geom[M.level];
      const bool rev = EA_ALTERNATE_SWEEP && M.rev, nrev = EA_ALTERNATE_SWEEP ? !rev : rev;
      if (M.pts_mode == EA_POINTS_XYZ) ea_eval_slice<true, THREADS>(M.pts, M.dt, M.affine, ng, A.inv_depth_scale, A.loss, A.sp.point_stride, P, j0, j1, S.part[0], S.cpart[0], rev);
      else ea_eval_slice<false, THREADS>(M.pts, M.dt, M.affine, ng, A.inv_depth_scale, A.loss, A.sp.point_stride, P, j0, j1, S.part[0], S.cpart[0], rev, &S.stage[0][0], M.same != 0, true, nrev);
    } else {
      K = ea_chunking(M.n_res, THREADS, chunk);
      cb = (K * M.nh) / (M.nh + 1);             // the owner is the last of nh + 1 workers: chunks [cb, K)
      ea_eval_chunks<THREADS>(A, S, M, P, cb, K, chunk, M.same != 0, true);
    }
    lap(0);
    __syncthreads();
    if (warp == 0) {
      if (CLUSTER) {
        const double tot = ea_cta_total<THREADS / 32>(S.part[0], S.cpart[0], lane);
        EaSolveSmem* S0 = cluster.map_shared_rank(&S, 0);
        if (lane < EA_SUMS) S0->cluster_sums[crank][lane] = tot;
      } else {
        // chunk totals in chunk order: the helpers' from the board (once each has delivered this epoch), the owner's from
        // shared memory
        double tot = 0.0;
        if (M.nh > 0) {
          int ok = 1;
          if (lane < M.nh) {
            long long spins = 0;
            while (ea_ld_acquire(&my_board->done[lane]) != S.help_epoch) {
              if (++spins > EA_BOARD_SPIN_LIMIT) { ok = 0; break; }
            }
          }
          ok = __all_sync(0xffffffffu, ok);
          __threadfence();
          if (!ok && lane == 0) S.help_fail = 1;
          for (int c = 0; c < cb; ++c) tot += __ldcg(&my_board->chunk[c][lane]);
        }
        {   // the owner's chunks: four independent 16-term chains (unrolled so that they overlap), added in chunk order
          double ct[EA_MAX_CHUNKS];
#pragma unroll
          for (int c = 0; c < EA_MAX_CHUNKS; ++c) ct[c] = (c >= cb && c < K) ? ea_cta_total<THREADS / 32>(S.part[c], S.cpart[c], lane) : 0.0;
#pragma unroll
          for (int c = 0; c < EA_MAX_CHUNKS; ++c) if (c >= cb && c < K) tot += ct[c];
        }
        if (lane < EA_SUMS) S.sums[lane] = tot;
        if (lane == 27 && S.help_fail) S.sums[27] = 1.0;      // a helper went missing: the evaluation counts as failed
        __syncwarp();
        lap(1);
        EaMsg& nm = S.msg[(g + 1) & 1];
        // (the number of registered helpers is read early: its latency hides behind the LM step)
        int reg = 0;
        if (helpers_on && lane == 31) reg = *reinterpret_cast<volatile int*>(&my_board->n_helpers);
        ea_boss_step_warp(S.args, S, M, nm, lane);
        reg = __shfl_sync(0xffffffffu, reg, 31);
        if (helpers_on) {
          // share the next evaluation with the registered helpers when it has chunks to give away
          int nh = 0;
          if (nm.cmd == EA_CMD_EVAL && reg > 0) {
            int ch2; const int K2 = ea_chunking(nm.n_res, THREADS, ch2);
            nh = min(min(reg, EA_MAX_HELPERS), K2 - 1);
          }
          if (lane == 0) { nm.nh = nh; if (nh != M.nh) nm.same = 0; }
          __syncwarp();
          if (nh > 0) {
            unsigned long long* dst = reinterpret_cast<unsigned long long*>(&my_board->msg);
            for (int i = lane; i < int(sizeof(EaMsg) / 8); i += 32) __stcg(dst + i, reinterpret_cast<const unsigned long long*>(&nm)[i]);
            __threadfence();
            __syncwarp();
            if (lane == 0) { S.help_epoch += 1; ea_st_release(&my_board->word, (S.help_epoch << 8) | (unsigned long long)nh); }
          }
          if (nm.cmd == EA_CMD_EXIT && lane == 0) {        // this CTA owns nothing any more: release its helpers
            *reinterpret_cast<volatile int*>(&my_board->busy) = 0;
            __threadfence();
            ea_st_release(&my_board->word, EA_BOARD_EXIT);
          }
        }
        lap(2);
      }
    }
    if (CLUSTER) {
      cluster.sync();
      if (crank == 0 && warp == 0) {
        double s = 0.0;
        if (lane < EA_SUMS) for (unsigned r = 0; r < csize; ++r) s += S.cluster_sums[r][lane];
        if (lane < EA_SUMS) S.sums[lane] = s;
        __syncwarp();
        EaMsg& nm = S.msg[(g + 1) & 1];
        ea_boss_step_warp(S.args, S, M, nm, lane);
        for (unsigned r = 1; r < csize; ++r) {      // the other ranks' copies, word by word over DSMEM
          unsigned long long* dst = reinterpret_cast<unsigned long long*>(&cluster.map_shared_rank(&S, r)->msg[(g + 1) & 1]);
          for (int i = lane; i < int(sizeof(EaMsg) / 8); i += 32) dst[i] = reinterpret_cast<const unsigned long long*>(&nm)[i];
        }
      }
    }
    sync_all();
    lap(3);
    if (dbg_on) S.dbg[4] += 1;
    g += 1;
  }
#ifdef EA_LM_PROFILE
  if (dbg_on && blockIdx.x == 0 && S.dbg[4] > 0)
    printf("[EA_LM_PROFILE] CTA 0, %lld evaluations; cycles per evaluation: tests %lld, update %lld, build %lld, LDLT %lld, model %lld, plus+stores %lld | advance_warp mean %lld\n",
           S.dbg[4], S.lm.prof[0] / S.dbg[4], S.lm.prof[1] / S.dbg[4], S.lm.prof[2] / S.dbg[4], S.lm.prof[3] / S.dbg[4], S.lm.prof[4] / S.dbg[4], S.lm.prof[5] / S.dbg[4], S.lm.prof[6] / S.dbg[4]);
#endif
  if (dbg_on) {
    S.dbg[5] = clock64() - S.dbg_t0;
    for (int k = 0; k < 6; ++k) A.debug[size_t(blockIdx.x) * 6 + k] = (unsigned long long)S.dbg[k];
  }
  if (CLUSTER) { cluster.sync(); return; }  // no CTA may exit while a peer can still touch its shared memory
  if (!helpers_on) return;
  // ================================================= helper loop ================================================
  // The queue is empty (tickets only grow, so no CTA will ever own a new pair): serve the CTAs that still own one.
  for (;;) {
    // ---- pick the busy owner with the fewest helpers and register there ----
    if (tid == 0) {
      int best = -1, best_n = EA_MAX_HELPERS, any_busy = 0;
      const int G = int(gridDim.x);
      for (int k = 1; k < G; ++k) {
        const int o = (int(blockIdx.x) + k) % G;
        if (!*reinterpret_cast<volatile int*>(&A.boards[o].busy)) continue;
        any_busy = 1;
        const int nreg = *reinterpret_cast<volatile int*>(&A.boards[o].n_helpers);
        if (nreg < best_n) { best_n = nreg; best = o; }
      }
      int idx = 0;
      if (best >= 0) {
        idx = atomicAdd(&A.boards[best].n_helpers, 1) + 1;
        if (idx > EA_MAX_HELPERS) { atomicSub(&A.boards[best].n_helpers, 1); best = -2; }      // lost the race for the last slot: look again
      }
      S.help_owner = best >= 0 ? best : (any_busy || best == -2 ? -2 : -1);
      S.help_index = idx;
    }
    __syncthreads();
    const int owner = S.help_owner, index = S.help_index;
    __syncthreads();
    if (owner == -1) break;                         // nobody owns a pair any more
    if (owner == -2) { __nanosleep(2000); continue; }  // every busy owner has its helpers: wait for one to finish
    EaHelpBoard* const B = A.boards + owner;
    unsigned long long seen = 0;
    for (;;) {
      // ---- wait for an evaluation that includes this helper, or for the owner to finish ----
      if (tid == 0) {
        unsigned long long w;
        long long spins = 0;
        for (;;) {
          w = ea_ld_acquire(&B->word);
          if (w == EA_BOARD_EXIT) break;
          if ((w >> 8) != seen && int(w & 0xff) >= index) break;
          if ((w >> 8) != seen) seen = w >> 8;      // an evaluation this helper is not part of yet
          if (++spins > EA_BOARD_SPIN_LIMIT) { w = EA_BOARD_EXIT; break; }
          __nanosleep(100);
        }
        S.help_epoch = w;
      }
      __syncthreads();
      const unsigned long long w = S.help_epoch;
      if (w == EA_BOARD_EXIT) { __syncthreads(); break; }
      seen = w >> 8;
      const int nh = int(w & 0xff);
      // ---- the shared evaluation's message, then this helper's chunks (worker index - 1 of nh + 1) ----
      if (warp == 0) {
        __threadfence();
        const unsigned long long* src = reinterpret_cast<const unsigned long long*>(&B->msg);
        for (int i = lane; i < int(sizeof(EaMsg) / 8); i += 32) reinterpret_cast<unsigned long long*>(&S.msg[0])[i] = __ldcg(src + i);
      }
      __syncthreads();
      const EaMsg& M = S.msg[0];
      const EaPose P = M.P;
      int chunk;
      const int K = ea_chunking(M.n_res, THREADS, chunk);
      const int cb = (K * (index - 1)) / (nh + 1), ce = (K * index) / (nh + 1);
      ea_eval_chunks<THREADS>(A, S, M, P, cb, ce, chunk, false, false);
      __syncthreads();
      if (warp == 0) {
        for (int c = cb; c < ce; ++c) {
          const double tot = ea_cta_total<THREADS / 32>(S.part[c], S.cpart[c], lane);
          __stcg(&B->chunk[c][lane], lane < EA_SUMS ? tot : 0.0);
        }
        __threadfence();
        __syncwarp();
        if (lane == 0) ea_st_release(&B->done[index - 1], seen);
      }
      __syncthreads();
    }
  }
}

// Per-point outputs for ea_eval (parity tests / EAResidue facade): same device functions as the solve.
template <bool XYZ>
__global__ void __launch_bounds__(256) ea_k_eval_points(EaLevelDesc rd, EaLevelDesc nd, EaLevelGeom rg, EaLevelGeom ng,
                                                        double inv_depth_scale, ea_solve_params sp, const double* pose7,
                                                        int n_res, double* raw, double* res, double* jac, int* failed) {
  EaPose P;
  ea_pose_setup<XYZ>(pose7, rg, ng, P);
  const float2 affine = *nd.dt_affine;
  const int n_round = (n_res + 31) & ~31;   // whole warps
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < n_round; j += gridDim.x * blockDim.x) {
    const bool valid = j < n_res;
    typedef EaPtStream<XYZ> PS;
    const typename PS::T p = valid ? PS::load(rd.pts, size_t(j) * sp.point_stride) : PS::pad();
    EaPointEval e;
    double a0, a1, a2;
    PS::unpack(p, a0, a1, a2);
    ea_point_eval<XYZ>(a0, a1, a2, ng, inv_depth_scale, P, nd.dt, affine, e);
    float rho0;
    const float w = ea_loss_eval(ea_eval_consts(sp.loss_type, sp.loss_scale, sp.point_stride), e.f, rho0);
    float J[6];
    ea_jacobian(e.gu, e.gv, e.ub, e.vb, e.pz, e.iz, P, affine.x * P.fx, affine.x * P.fy, w, J);
    if (!valid) continue;
    if (raw) raw[j] = double(e.f);
    if (res) res[j] = double(e.f * w);
    if (jac) {
#pragma unroll
      for (int k = 0; k < 6; ++k) jac[size_t(j) * 6 + k] = double(J[k]);
    }
    if (e.fail && failed) atomicAdd(failed, 1);
  }
}

// Normal-equation sums through the production reduction path (one CTA per slice of the points).
template <int THREADS>
__global__ void __launch_bounds__(THREADS) ea_k_eval_sums(EaLevelDesc rd, EaLevelDesc nd, EaLevelGeom rg, EaLevelGeom ng,
                                                          double inv_depth_scale, ea_solve_params sp, EaEvalConsts loss, const double* pose7,
                                                          const int* done, int j_begin, int j_end, double* sums /*[grid][EA_SUMS]*/) {
  if (done && *done) return;
  __shared__ double part[THREADS / 32][EA_NSUM];
  __shared__ double cpart[THREADS / 32];
  const int n = j_end - j_begin;
  const int j0 = j_begin + int((long long)n * blockIdx.x / gridDim.x), j1 = j_begin + int((long long)n * (blockIdx.x + 1) / gridDim.x);
  EaPose P;
  if (rd.pts_mode == EA_POINTS_XYZ) {
    ea_pose_setup<true>(pose7, rg, ng, P);
    ea_eval_slice<true, THREADS>(rd.pts, nd.dt - ea_dt_origin_offset(nd.w), *nd.dt_affine, ng, inv_depth_scale, loss, sp.point_stride, P, j0, j1, part, cpart);
  } else {
    ea_pose_setup<false>(pose7, rg, ng, P);
    ea_eval_slice<false, THREADS>(rd.pts, nd.dt - ea_dt_origin_offset(nd.w), *nd.dt_affine, ng, inv_depth_scale, loss, sp.point_stride, P, j0, j1, part, cpart);
  }
  __syncthreads();
  if (threadIdx.x < 32) {
    const double tot = ea_cta_total<THREADS / 32>(part, cpart, threadIdx.x);
    if (threadIdx.x < EA_SUMS) sums[size_t(blockIdx.x) * EA_SUMS + threadIdx.x] = tot;
  }
}

// ---- memory-side roof of the fused evaluation (measurement only) -----------------------------------------------------
// The same point stream, the same fp64 projection (it generates the addresses) and the same 16-texel clamp-to-edge gather
// as ea_eval_slice, and nothing else: no interpolation, no Jacobian, no reduction, no LM, few registers, full occupancy.
// Its rate is the L1/L2-gather roofline of the access pattern for the frames and poses at hand (SURVEY.md 8d).
__global__ void __launch_bounds__(256) ea_k_gather_probe(const __grid_constant__ EaSolveArgs A, int level, int slices, int repeats,
                                                         float* __restrict__ sink) {
  const int pair = blockIdx.x / slices, slice = blockIdx.x % slices;
  if (pair >= A.n_pairs) return;
  const EaLevelDesc rd = A.ref_desc[size_t(A.ref_slots[pair]) * EA_MAX_LEVELS + level];
  const EaLevelDesc nd = A.now_desc[size_t(A.now_slots[pair]) * EA_MAX_LEVELS + level];
  const EaLevelGeom& rg = A.ref_geom[level];
  const EaLevelGeom& ng = A.now_geom[level];
  const int n = min(*rd.n_pts, A.ref_cap[level]);
  const int j0 = int((long long)n * slice / slices), j1 = int((long long)n * (slice + 1) / slices);
  if (rd.pts_mode != EA_POINTS_PIXEL) return;
  EaPose P;
  ea_pose_setup<false>(A.poses + size_t(pair) * 7, rg, ng, P);
  float s = 0.0f;
  const int pitch = ea_dt_pitch(ng.w);
  const float* dt_base = ea_gather_base(nd.dt - ea_dt_origin_offset(ng.w), pitch);
  for (int r = 0; r < repeats; ++r)
    for (int j = j0 + int(threadIdx.x); j < j1; j += 256) {
      typedef EaPtStream<false> PS;
      const PS::T p = PS::load(rd.pts, size_t(j));
      double a0, a1, a2;
      PS::unpack(p, a0, a1, a2);
      EaProj pr;
      ea_project<false>(a0, a1, a2, ng.w, ng.h, pitch, A.inv_depth_scale, P, pr);
      float t[16];
      ea_gather(dt_base, pr.off, pitch, t);
      float ts = pr.du + pr.dv;
#pragma unroll
      for (int k = 0; k < 16; ++k) ts += t[k];
      s += ts;
    }
  sink[size_t(blockIdx.x) * 256 + threadIdx.x] = s;
}

cudaError_t ea_launch_gather_probe(const EaSolveArgs& A, int level, int slices, int repeats, float* d_sink, cudaStream_t stream) {
  // EA_PROBE_SMEM_KB: occupancy experiment (dynamic shared memory only limits the number of resident CTAs)
  static const int smem_kb = getenv("EA_PROBE_SMEM_KB") ? atoi(getenv("EA_PROBE_SMEM_KB")) : 0;
  if (smem_kb > 48) cudaFuncSetAttribute(ea_k_gather_probe, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_kb * 1024);
  ea_k_gather_probe<<<unsigned(A.n_pairs * slices), 256, size_t(smem_kb) * 1024, stream>>>(A, level, slices, repeats, d_sink);
  return cudaGetLastError();
}

// ---- host launchers -----------------------------------------------------------------------------------
size_t ea_help_boards_bytes(int sm_count) { return size_t(sm_count) * EA_SOLVE_MIN_CTAS * sizeof(EaHelpBoard); }

cudaError_t ea_launch_solve_batch(const EaSolveArgs& A, int cluster_size, int sm_count, cudaStream_t stream) {
  if (A.n_pairs <= 0) return cudaSuccess;
  cudaError_t e = cudaMemsetAsync(A.work_counter, 0, sizeof(int), stream);
  if (e != cudaSuccess) return e;
  if (A.boards && cluster_size <= 1) {
    e = cudaMemsetAsync(A.boards, 0, ea_help_boards_bytes(sm_count), stream);
    if (e != cudaSuccess) return e;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.blockDim = dim3(EA_SOLVE_THREADS);
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  if (cluster_size <= 1) {
    // persistent CTAs (EA_SOLVE_MIN_CTAS per SM) pulling pairs from the work queue
    int max_ctas = sm_count * EA_SOLVE_MIN_CTAS;
    static const int env_ctas = getenv("EA_SOLVE_MAX_CTAS") ? atoi(getenv("EA_SOLVE_MAX_CTAS")) : 0;   // experiment knob (DESIGN.md 8)
    if (env_ctas > 0 && env_ctas < max_ctas) max_ctas = env_ctas;
    cfg.gridDim = dim3(unsigned(A.n_pairs < max_ctas ? A.n_pairs : max_ctas));
    cfg.numAttrs = 0;
    return cudaLaunchKernelEx(&cfg, ea_k_solve_batch<EA_SOLVE_THREADS, false>, A);
  }
  int n_clusters = A.n_pairs;
  const int max_clusters = (sm_count * EA_SOLVE_MIN_CTAS) / cluster_size;
  if (n_clusters > max_clusters) n_clusters = max_clusters;
  if (n_clusters < 1) n_clusters = 1;
  cfg.gridDim = dim3(unsigned(n_clusters * cluster_size));
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = unsigned(cluster_size);
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, ea_k_solve_batch<EA_SOLVE_THREADS, true>, A);
}

cudaError_t ea_launch_eval_points(const EaLevelDesc& rd, const EaLevelDesc& nd, const EaLevelGeom& rg,
                                  const EaLevelGeom& ng, double inv_depth_scale, const ea_solve_params& sp,
                                  const double* d_pose7, int n_res, double* d_raw, double* d_res, double* d_jac,
                                  int* d_failed, cudaStream_t stream) {
  if (n_res <= 0) return cudaSuccess;
  const int blocks = (n_res + 255) / 256;
  if (rd.pts_mode == EA_POINTS_XYZ)
    ea_k_eval_points<true><<<blocks, 256, 0, stream>>>(rd, nd, rg, ng, inv_depth_scale, sp, d_pose7, n_res, d_raw, d_res, d_jac, d_failed);
  else
    ea_k_eval_points<false><<<blocks, 256, 0, stream>>>(rd, nd, rg, ng, inv_depth_scale, sp, d_pose7, n_res, d_raw, d_res, d_jac, d_failed);
  return cudaGetLastError();
}

cudaError_t ea_launch_eval_sums(const EaLevelDesc& rd, const EaLevelDesc& nd, const EaLevelGeom& rg,
                                const EaLevelGeom& ng, double inv_depth_scale, const ea_solve_params& sp,
                                const double* d_pose7, const int* d_done, int j_begin, int j_end, int n_blocks, double* d_sums,
                                cudaStream_t stream) {
  if (n_blocks <= 0) return cudaSuccess;
  ea_k_eval_sums<EA_SOLVE_THREADS><<<n_blocks, EA_SOLVE_THREADS, 0, stream>>>(rd, nd, rg, ng, inv_depth_scale, sp, ea_eval_consts(sp.loss_type, sp.loss_scale, sp.point_stride),
                                                                              d_pose7, d_done, j_begin, j_end, d_sums);
  return cudaGetLastError();
}

#ifndef EA_ORDER_FIXED_COST
#define EA_ORDER_FIXED_COST 8000   // measured: 0 -> 6000 -> 12000 gives 7.41 -> 7.35 -> 7.34 ms per 1184-pair launch
#endif
// ---- longest-first ordering for the next launch: sort pairs by the work their last solve needed -----------------
// One CTA, bitonic sort of (work, index) in shared memory; n <= 4096.
__global__ void __launch_bounds__(1024) ea_k_order_by_work(const ea_summary* __restrict__ summaries, int n, int n_levels, int32_t* __restrict__ order) {
  __shared__ unsigned long long key[4096];
  int m = 1;
  while (m < n) m <<= 1;
  for (int i = threadIdx.x; i < m; i += blockDim.x) {
    unsigned long long k = 0;
    if (i < n) {
      unsigned long long work = 0;
      for (int l = 0; l < n_levels; ++l) {
        const ea_summary s = summaries[size_t(i) * n_levels + l];
        // evaluations x (points + the serial section between two evaluations in point-equivalents)
        work += (unsigned long long)((s.n_residuals > 0 ? s.n_residuals : 0) + EA_ORDER_FIXED_COST) * (unsigned long long)(s.evaluations > 0 ? s.evaluations : 0);
      }
      if (work > 0xFFFFFFFFFFFull) work = 0xFFFFFFFFFFFull;
      k = (work << 20) | (unsigned long long)(0xFFFFF - i);       // descending work, ascending index on ties
    }
    key[i] = k;
  }
  __syncthreads();
  for (int size = 2; size <= m; size <<= 1)
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int i = threadIdx.x; i < m; i += blockDim.x) {
        const int j = i ^ stride;
        if (j > i) {
          const bool desc = (i & size) == 0;
          const unsigned long long a = key[i], b = key[j];
          if (desc ? (a < b) : (a > b)) { key[i] = b; key[j] = a; }
        }
      }
      __syncthreads();
    }
  for (int i = threadIdx.x; i < n; i += blockDim.x) order[i] = int32_t(0xFFFFF - int(key[i] & 0xFFFFF));
}

cudaError_t ea_launch_order_by_work(const ea_summary* d_summaries, int n, int n_levels, int32_t* d_order, cudaStream_t stream) {
  if (n <= 0 || n > 4096) return cudaErrorInvalidValue;
  ea_k_order_by_work<<<1, 1024, 0, stream>>>(d_summaries, n, n_levels, d_order);
  return cudaGetLastError();
}
