// Point-sharded solve of ONE large frame pair across ranks (BASELINE config "4K, ~2M edge points"):
// every rank holds the full distance transform and a contiguous slice of the ordered point list, reduces its
// slice to the 29 normal-equation sums, and one ncclAllReduce(sum, 29 x fp64 = 232 B) per evaluation makes
// them global.  All ranks then run the identical 6x6 LM step on bit-identical sums, so they take identical
// accept/reject decisions with no broadcast.  Nothing in the reference corresponds to this (it is
// single-threaded); the math per point and the LM semantics are those of ea_solve.cu / ea_solve.cuh.
//
// NCCL is bound lazily with dlopen("libnccl.so.2") so the library has no hard NCCL dependency and, inside a
// torch process, resolves to the copy torch already loaded.
#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <cstring>
#include <new>
#include <vector>

#include "ea_internal.h"
#include "ea_solve.cuh"

namespace {

struct NcclApi {
  void* handle = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
};
NcclApi g_nccl;

int load_nccl() {
  if (g_nccl.handle) return EA_OK;
  void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
  if (!h) return ea_fail(EA_ERR_NCCL, "cannot dlopen libnccl.so.2: %s", dlerror());
  g_nccl.GetUniqueId = (decltype(g_nccl.GetUniqueId))dlsym(h, "ncclGetUniqueId");
  g_nccl.CommInitRank = (decltype(g_nccl.CommInitRank))dlsym(h, "ncclCommInitRank");
  g_nccl.AllReduce = (decltype(g_nccl.AllReduce))dlsym(h, "ncclAllReduce");
  g_nccl.AllGather = (decltype(g_nccl.AllGather))dlsym(h, "ncclAllGather");
  g_nccl.CommDestroy = (decltype(g_nccl.CommDestroy))dlsym(h, "ncclCommDestroy");
  g_nccl.GetErrorString = (decltype(g_nccl.GetErrorString))dlsym(h, "ncclGetErrorString");
  if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.AllReduce || !g_nccl.AllGather || !g_nccl.CommDestroy || !g_nccl.GetErrorString)
    return ea_fail(EA_ERR_NCCL, "libnccl.so.2 lacks a required symbol");
  g_nccl.handle = h;
  return EA_OK;
}
#define NC(call)                                                                                               \
  do {                                                                                                         \
    ncclResult_t r_ = (call);                                                                                  \
    if (r_ != ncclSuccess) return ea_fail(EA_ERR_NCCL, "%s -> %s", #call, g_nccl.GetErrorString(r_));          \
  } while (0)

struct ShardState {        // device-resident control block
  EaLmState lm;
  double cand[7];
  int done, started;
};

// ---- general (rig / distortion) evaluation kernels: residual variants of standalone/utils.h:101-421 ----------------
#define GV_THREADS 256
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
  float acc[EA_NSUM];
#pragma unroll
  for (int k = 0; k < EA_NSUM; ++k) acc[k] = 0.0f;
  double acc64 = 0.0, cost64 = 0.0;
  for (int base = j0 + warp * 32; base < j1; base += GV_THREADS) {
    const int j = base + lane;
    if (j < j1) {
      const float4 p = EaPtStream<XYZ>::as_float4(EaPtStream<XYZ>::load(rd.pts, size_t(j) * sp.point_stride));
      float f, w, rho0, J[6];
      const bool fail = ea_point_eval_general<XYZ>(p, ng, inv_depth_scale, P, nd.dt, affine, sp.loss_type, float(sp.loss_scale), f, w, rho0, J);
      ea_accumulate(acc, J, f * w);
      acc[27] += fail ? 1.0f : 0.0f;
      cost64 += double(0.5f * rho0);
    }
    acc64 += double(ea_warp_transpose_reduce(acc, lane));
#pragma unroll
    for (int k = 0; k < EA_NSUM; ++k) acc[k] = 0.0f;
  }
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

__global__ void k_shard_reduce(const ShardState* st, const double* partials, int n_blocks, double* sums) {
  if (st->done) return;
  const int k = threadIdx.x;
  if (k < EA_SUMS) {
    double s = 0.0;
    for (int b = 0; b < n_blocks; ++b) s += partials[size_t(b) * EA_SUMS + k];   // fixed order: deterministic
    sums[k] = s;
  }
}

__global__ void __launch_bounds__(32) k_shard_lm(ShardState* st, const double* sums, ea_solve_params sp) {   // one warp
  if (st->done) return;
  __shared__ double local[32];
  __shared__ EaLmState lm;
  const int lane = threadIdx.x;
  local[lane] = lane < EA_SUMS ? sums[lane] : 0.0;
  for (int i = lane; i < int(sizeof(EaLmState) / 8); i += 32) reinterpret_cast<unsigned long long*>(&lm)[i] = reinterpret_cast<const unsigned long long*>(&st->lm)[i];
  __syncwarp();
  const int cmd = ea_lm_advance_warp(lm, local, sp, lane);
  __syncwarp();
  for (int i = lane; i < int(sizeof(EaLmState) / 8); i += 32) reinterpret_cast<unsigned long long*>(&st->lm)[i] = reinterpret_cast<const unsigned long long*>(&lm)[i];
  if (lane == 0) {
    if (cmd == EA_CMD_EVAL) { for (int i = 0; i < 7; ++i) st->cand[i] = lm.cand[i]; }
    else st->done = 1;
  }
}

// =====================================================================================================================
// One persistent cooperative kernel per rank for the whole solve of one (pair, level): no host round trip, no kernel
// launch and no NCCL call per LM evaluation.
//
//   every CTA      evaluates its slice of this rank's point range (ea_eval_slice, the production loop) -> 29 CTA totals
//   grid reduce    totals to global memory, one atomic ticket per CTA; CTA 0 -- the reducer of every evaluation -- waits for the
//                  tickets and adds the per-CTA totals in a fixed order (bitwise reproducible)
//   all-reduce     CTA 0 stores the rank's sums straight into every peer's exchange buffer over NVLink (peer-mapped cudaIpc
//                  memory) as self-validating 8-byte packets {32 data bits, 32-bit epoch tag}, two per double: one store and
//                  one load per packet, no system-scope fence, no flag to order behind the data.  It then polls the world's
//                  packets in its own buffer and adds the contributions in rank order: every rank obtains bit-identical sums,
//                  so all ranks take identical LM decisions with no broadcast.  Slots are double-buffered by evaluation parity
//                  (a rank can be at most one evaluation ahead of a peer).
//   LM             CTA 0's first warp advances the Ceres-equivalent trust-region state machine on the state it keeps in shared
//                  memory (ea_lm_advance_warp), publishes the next candidate pose and releases the grid through an epoch word
//                  the other CTAs poll
// Every wait is bounded (EA_SHARD_SPIN_LIMIT polls): a lost peer ends the solve with EA_TERM_FAILURE_PEER instead of hanging
// the GPU.
#define EA_SHARD_MAX_WORLD 8
#define EA_SHARD_SPIN_LIMIT (1ll << 22)   // ~3 s of polling
struct ShardXchg {                                  // lives in cudaIpc-shared device memory, one per rank
  // Self-validating 8-byte packets {32 data bits, 32-bit epoch tag}, two per double (the "LL" idea of NCCL): a packet is one
  // store and one load, so there is no flag to order behind the data -- no system-scope fence, no second NVLink round trip.
  unsigned long long ll[2][EA_SHARD_MAX_WORLD][64]; // [evaluation parity][source rank][2 x 32 sums]
};
struct ShardPeers { ShardXchg* p[EA_SHARD_MAX_WORLD]; };
struct ShardCtl {                                   // per-rank control block (device memory)
  EaLmState lm;
  EaPose P;                                         // candidate pose folded with the intrinsics, for the evaluation in flight
  unsigned long long go;                            // evaluation epoch released to the grid
  unsigned long long ticket;                        // CTAs that have delivered their totals (monotonic over the solve)
  int done, error;
  long long prof[6];                                // cycles: {evaluation (CTA 0), grid reduce, all-reduce, LM} of the CTA that did them, evaluations
};

__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_gpu(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_gpu(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

template <int THREADS>
__global__ void __launch_bounds__(THREADS, 1) k_shard_solve(EaLevelDesc rd, EaLevelDesc nd, EaLevelGeom rg, EaLevelGeom ng,
                                                            double inv_depth_scale, ea_solve_params sp, EaEvalConsts loss, ShardCtl* ctl,
                                                            double* partials /*[grid][32]*/, ShardPeers peers, int rank, int world,
                                                            unsigned long long epoch0, int j_begin, int j_end) {
  __shared__ double part[THREADS / 32][EA_NSUM];
  __shared__ double cpart[THREADS / 32];
  __shared__ double wsum[THREADS / 32][32];
  __shared__ int s_stop, s_late;
  __shared__ EaLmState s_lm;      // CTA 0 only: the LM state stays in its shared memory for the whole solve
  __shared__ __align__(2 * EA_STAGE_SLOT * 8) uint2 stage[2][EA_STAGE_SLOT];   // cp.async staging of the point stream (ea_eval_slice: aligned to its size)
  static_assert(sizeof(EaLmState) % 8 == 0, "EaLmState is copied as 8-byte words");
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n = j_end - j_begin;
  const int j0 = j_begin + int((long long)n * blockIdx.x / gridDim.x), j1 = j_begin + int((long long)n * (blockIdx.x + 1) / gridDim.x);
  const float2 affine = *nd.dt_affine;
  const float* dt_pad = nd.dt - ea_dt_origin_offset(nd.w);
  const bool xyz = rd.pts_mode == EA_POINTS_XYZ;
  if (blockIdx.x == 0 && warp == 0) {   // the reducer CTA keeps the LM state (initialised by k_shard_ctl_init)
    const unsigned long long* src = reinterpret_cast<const unsigned long long*>(&ctl->lm);
    unsigned long long* dst = reinterpret_cast<unsigned long long*>(&s_lm);
    for (int i = lane; i < int(sizeof(EaLmState) / 8); i += 32) dst[i] = __ldcg(src + i);
  }
  for (unsigned long long e = 1;; ++e) {
    // ---- wait for the release of evaluation e (e == 1 is released by the host-side initialisation) ----
    if (tid == 0) {
      long long spins = 0;
      int stop = 0;
      while (ld_acquire_gpu(&ctl->go) < e) {
        if (++spins > EA_SHARD_SPIN_LIMIT) { stop = 2; break; }
        __nanosleep(20);
      }
      if (!stop) stop = *reinterpret_cast<volatile int*>(&ctl->done);
      s_stop = stop;
    }
    __syncthreads();
    if (s_stop) break;
    long long t0 = 0;
    if (blockIdx.x == 0 && tid == 0) t0 = clock64();
    EaPose P;
    {   // the candidate's folded pose, written by the LM thread of the previous round (L2: bypass the non-coherent L1)
      const double* src = reinterpret_cast<const double*>(&ctl->P);
      double* dst = reinterpret_cast<double*>(&P);
#pragma unroll
      for (int i = 0; i < int(sizeof(EaPose) / 8); ++i) dst[i] = __ldcg(src + i);
    }
    if (xyz) ea_eval_slice<true, THREADS>(rd.pts, dt_pad, affine, ng, inv_depth_scale, loss, sp.point_stride, P, j0, j1, part, cpart, EA_ALTERNATE_SWEEP && !(e & 1));
    else {
      const bool rev = EA_ALTERNATE_SWEEP && !(e & 1);
      ea_eval_slice<false, THREADS>(rd.pts, dt_pad, affine, ng, inv_depth_scale, loss, sp.point_stride, P, j0, j1, part, cpart, rev, &stage[0][0], e > 1, true, EA_ALTERNATE_SWEEP ? !rev : rev);
    }
    __syncthreads();
    if (warp == 0) {
      const double tot = ea_cta_total<THREADS / 32>(part, cpart, lane);
      __stcg(&partials[size_t(blockIdx.x) * 32 + lane], lane < EA_SUMS ? tot : 0.0);
      __threadfence();
      __syncwarp();
      if (lane == 0) {
        if (blockIdx.x != 0) atomicAdd(&ctl->ticket, 1ull);      // delivered; nothing to wait for: on to the next release
        else {
          ctl->prof[0] += clock64() - t0;
          // CTA 0 is the reducer of every evaluation: it waits for the other CTAs' tickets (monotonic over the solve)
          const unsigned long long want = e * (unsigned long long)(gridDim.x - 1);
          long long spins = 0;
          int late = 0;
          while (ld_acquire_gpu(&ctl->ticket) < want) { if (++spins > EA_SHARD_SPIN_LIMIT) { late = 1; break; } }
          s_late = late;
        }
      }
    }
    if (blockIdx.x != 0) continue;
    __syncthreads();
    // ---- CTA 0: grid reduce (fixed order: warp w adds CTAs w, w + W, ...; then the warps in order) ----
    __threadfence();
    long long t1 = clock64();
    {
      double s_ = 0.0;
      for (unsigned b = warp; b < gridDim.x; b += THREADS / 32) s_ += __ldcg(&partials[size_t(b) * 32 + lane]);
      wsum[warp][lane] = s_;
    }
    __syncthreads();
    if (warp == 0) {
      double tot = 0.0;
#pragma unroll
      for (int w2 = 0; w2 < THREADS / 32; ++w2) tot += wsum[w2][lane];
      long long t2 = clock64();
      int err = 0;
      // ---- all-reduce over NVLink peer memory ----
      if (world > 1) {
        const int par = int(e & 1);
        const unsigned long long epoch = epoch0 + e;
        // every lane ships its own sum to every rank (own one included) as two packets, then polls the world's packets for its slot
        const unsigned tag = unsigned(epoch);
        const unsigned long long bits = (unsigned long long)__double_as_longlong(tot);
        const unsigned long long p_lo = (bits & 0xffffffffull) | ((unsigned long long)tag << 32);
        const unsigned long long p_hi = (bits >> 32) | ((unsigned long long)tag << 32);
        for (int r = 0; r < world; ++r) {
          volatile unsigned long long* dst = &peers.p[r]->ll[par][rank][2 * lane];
          dst[0] = p_lo; dst[1] = p_hi;                   // 32 lanes x 16 B = one 512 B burst per peer
        }
        double g = 0.0;
        for (int r = 0; r < world; ++r) {                 // rank order: identical sums everywhere
          const volatile unsigned long long* src = &peers.p[rank]->ll[par][r][2 * lane];
          unsigned long long a = src[0], b = src[1];
          long long spins = 0;
          while (unsigned(a >> 32) != tag || unsigned(b >> 32) != tag) {
            if (++spins > EA_SHARD_SPIN_LIMIT) { err = 1; break; }
            a = src[0]; b = src[1];
          }
          g += __longlong_as_double((long long)((a & 0xffffffffull) | (b << 32)));
        }
        err = __any_sync(0xffffffffu, err);
        tot = g;
      }
      long long t3 = clock64();
      wsum[0][lane] = tot;
      __syncwarp();
      int done = 0;
      if (s_late) err = 1;            // a CTA of this grid never delivered
      if (err) { if (lane == 0) { s_lm.term = EA_TERM_FAILURE_PEER; ctl->error = 1; } done = 1; }
      else {
        const int cmd = ea_lm_advance_warp(s_lm, wsum[0], sp, lane);            // all 32 lanes: warp-cooperative LM step
        if (cmd == EA_CMD_EVAL) {
          EaPose Pn;
          if (xyz) ea_pose_setup<true>(s_lm.cand, rg, ng, Pn); else ea_pose_setup<false>(s_lm.cand, rg, ng, Pn);
          if (lane == 0) ctl->P = Pn;
        } else done = 1;
      }
      __syncwarp();
      if (done) {   // the host reads the final state from global memory
        const unsigned long long* src = reinterpret_cast<const unsigned long long*>(&s_lm);
        unsigned long long* dst = reinterpret_cast<unsigned long long*>(&ctl->lm);
        for (int i = lane; i < int(sizeof(EaLmState) / 8); i += 32) __stcg(dst + i, src[i]);
      }
      __threadfence();
      __syncwarp();
      if (lane == 0) {
        ctl->done = done;
        const long long t4 = clock64();
        ctl->prof[1] += t2 - t1; ctl->prof[2] += t3 - t2; ctl->prof[3] += t4 - t3; ctl->prof[4] += 1;
        __threadfence();
        st_release_gpu(&ctl->go, e + 1);
      }
    }
  }
  if (s_stop == 2 && tid == 0) ctl->error = 2;   // the release never came (a CTA of this grid or a peer rank is gone)
}

// ---- the same persistent scheme for the residual VARIANTS (ea_solve_views): any number of cameras constrain one pose ----------
// One cooperative kernel for the whole solve: every CTA evaluates its slice of every view's point list with the general
// per-point evaluation (rig transform and / or distortion per view), the CTA that draws the evaluation's last ticket adds the CTA
// totals in a fixed order, runs the warp-cooperative LM step on the state in shared memory and releases the next evaluation.
struct ViewDev {                  // one view, device-side (array in global memory)
  EaLevelDesc rd, nd;
  EaLevelGeom rg, ng;
  EaViewXf X;
  double inv_depth_scale;
  int n_res, xyz;
};
__global__ void __launch_bounds__(GV_THREADS, 1) k_views_solve(const ViewDev* __restrict__ views, int n_views, ea_solve_params sp, ShardCtl* ctl,
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
    if (tid == 0) {
      long long spins = 0;
      int stop = 0;
      while (ld_acquire_gpu(&ctl->go) < e) {
        if (++spins > EA_SHARD_SPIN_LIMIT) { stop = 2; break; }
        __nanosleep(20);
      }
      if (!stop) stop = *reinterpret_cast<volatile int*>(&ctl->done);
      s_stop = stop;
    }
    __syncthreads();
    if (s_stop) break;
    double cand[7];
#pragma unroll
    for (int i = 0; i < 7; ++i) cand[i] = __ldcg(&ctl->lm.cand[i]);      // written by the LM warp of the previous round (L2)
    float acc[EA_NSUM];
#pragma unroll
    for (int k = 0; k < EA_NSUM; ++k) acc[k] = 0.0f;
    double acc64 = 0.0, cost64 = 0.0;
    for (int v = 0; v < n_views; ++v) {
      const ViewDev& V = views[v];
      const int j0 = int((long long)V.n_res * blockIdx.x / gridDim.x), j1 = int((long long)V.n_res * (blockIdx.x + 1) / gridDim.x);
      if (j1 <= j0) continue;                                            // (uniform per CTA)
      EaPoseG P;
      if (V.xyz) ea_pose_setup_general<true>(cand, V.rg, V.ng, V.X, P); else ea_pose_setup_general<false>(cand, V.rg, V.ng, V.X, P);
      const float2 affine = *V.nd.dt_affine;
      for (int base = j0 + warp * 32; base < j1; base += GV_THREADS) {
        const int j = base + lane;
        if (j < j1) {
          float f, w, rho0, J[6];
          bool fail;
          if (V.xyz) {
            const float4 p = EaPtStream<true>::as_float4(EaPtStream<true>::load(V.rd.pts, size_t(j) * sp.point_stride));
            fail = ea_point_eval_general<true>(p, V.ng, V.inv_depth_scale, P, V.nd.dt, affine, sp.loss_type, float(sp.loss_scale), f, w, rho0, J);
          } else {
            const float4 p = EaPtStream<false>::as_float4(EaPtStream<false>::load(V.rd.pts, size_t(j) * sp.point_stride));
            fail = ea_point_eval_general<false>(p, V.ng, V.inv_depth_scale, P, V.nd.dt, affine, sp.loss_type, float(sp.loss_scale), f, w, rho0, J);
          }
          ea_accumulate(acc, J, f * w);
          acc[27] += fail ? 1.0f : 0.0f;
          cost64 += double(0.5f * rho0);
        }
        acc64 += double(ea_warp_transpose_reduce(acc, lane));
#pragma unroll
        for (int k = 0; k < EA_NSUM; ++k) acc[k] = 0.0f;
      }
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
    // ---- last CTA: grid reduce (fixed order: warp w adds CTAs w, w + W, ...; then the warps in order), LM, release ----
    __threadfence();
    {
      double s_ = 0.0;
      for (unsigned b = warp; b < gridDim.x; b += WARPS) s_ += __ldcg(&partials[size_t(b) * 32 + lane]);
      wsum[warp][lane] = s_;
    }
    __syncthreads();
    if (warp == 0) {
      double tot = 0.0;
#pragma unroll
      for (int w2 = 0; w2 < WARPS; ++w2) tot += wsum[w2][lane];
      wsum[0][lane] = tot;
      {
        const unsigned long long* src = reinterpret_cast<const unsigned long long*>(&ctl->lm);
        unsigned long long* dst = reinterpret_cast<unsigned long long*>(&s_lm);
        for (int i = lane; i < int(sizeof(EaLmState) / 8); i += 32) dst[i] = __ldcg(src + i);
      }
      __syncwarp();
      const int cmd = ea_lm_advance_warp(s_lm, wsum[0], sp, lane);            // (the next candidate is left in s_lm.cand)
      __syncwarp();
      {
        const unsigned long long* src = reinterpret_cast<const unsigned long long*>(&s_lm);
        unsigned long long* dst = reinterpret_cast<unsigned long long*>(&ctl->lm);
        for (int i = lane; i < int(sizeof(EaLmState) / 8); i += 32) __stcg(dst + i, src[i]);
      }
      __threadfence();
      __syncwarp();
      if (lane == 0) {
        ctl->done = cmd == EA_CMD_EVAL ? 0 : 1;
        ctl->prof[4] += 1;
        __threadfence();
        st_release_gpu(&ctl->go, e + 1);
      }
    }
  }
  if (s_stop == 2 && tid == 0) ctl->error = 2;   // the release never came (a CTA of this grid is gone)
}

// first evaluation's control block: LM state at the initial pose, its folded pose, evaluation 1 released
__global__ void k_shard_ctl_init(ShardCtl* ctl, const double* pose7, EaLevelGeom rg, EaLevelGeom ng, int xyz) {
  EaLmState& L = ctl->lm;
  L.phase = 0; L.iter = 0; L.accepted = 0; L.rejected = 0; L.invalid_run = 0; L.evals = 0; L.term = EA_TERM_NONE;
  L.cost = 0.0; L.initial_cost = 0.0;
  for (int i = 0; i < 7; ++i) { L.x[i] = pose7[i]; L.cand[i] = pose7[i]; }
  EaPose P;
  if (xyz) ea_pose_setup<true>(L.cand, rg, ng, P); else ea_pose_setup<false>(L.cand, rg, ng, P);
  ctl->P = P;
  ctl->ticket = 0; ctl->done = 0; ctl->error = 0;
  for (int k = 0; k < 6; ++k) ctl->prof[k] = 0;
  __threadfence();
  ctl->go = 1;
}

__global__ void k_shard_init(ShardState* st, const double* pose7) {
  EaLmState& L = st->lm;
  L.phase = 0; L.iter = 0; L.accepted = 0; L.rejected = 0; L.invalid_run = 0; L.evals = 0; L.term = EA_TERM_NONE;
  L.cost = 0.0; L.initial_cost = 0.0;
  for (int i = 0; i < 7; ++i) { L.x[i] = pose7[i]; L.cand[i] = pose7[i]; st->cand[i] = pose7[i]; }
  st->done = 0; st->started = 1;
}

}  // namespace

struct ea_shard {
  ea_context* ctx = nullptr;
  ncclComm_t comm = nullptr;
  int rank = 0, world = 1;
  // host-driven path (EA_SHARD_MODE=nccl, or no peer access): one launch triple + ncclAllReduce per evaluation
  ShardState* d_state = nullptr;
  double* d_partials = nullptr;
  double* d_sums = nullptr;
  double* d_pose = nullptr;
  int n_blocks = 0;
  int* h_done = nullptr;  // pinned
  // persistent path: one cooperative kernel per solve, all-reduce through peer-mapped exchange buffers
  bool in_kernel = false;
  ShardCtl* d_ctl = nullptr;
  double* d_cta_sums = nullptr;                 // [sm_count][32]
  ShardXchg* xchg = nullptr;                    // this rank's buffer (cudaMalloc; exported with cudaIpcGetMemHandle)
  ShardPeers peers{};                           // every rank's buffer as seen from this device
  bool peer_open[EA_SHARD_MAX_WORLD] = {};
  unsigned long long epoch = 1;                 // advances identically on every rank (same evaluation counts)
  bool poisoned = false;                        // a peer was lost: epochs may have diverged
  double clock_khz = 1.0;
  double prof[8] = {0, 0, 0, 0, 0, 0, 0, 0};    // last solve: see ea_shard_profile
};

extern "C" {

int ea_shard_unique_id(uint8_t id128[128]) {
  if (!id128) return ea_fail(EA_ERR_INVALID_ARG, "null id");
  int rc = load_nccl();
  if (rc) return rc;
  ncclUniqueId id;
  NC(g_nccl.GetUniqueId(&id));
  static_assert(sizeof(id) == 128, "ncclUniqueId size");
  std::memcpy(id128, &id, 128);
  return EA_OK;
}

int ea_shard_destroy(ea_shard* s) {
  if (!s) return EA_OK;
  cudaSetDevice(s->ctx->device);
  cudaStreamSynchronize(s->ctx->stream);
  for (int r = 0; r < EA_SHARD_MAX_WORLD; ++r)
    if (s->peer_open[r]) cudaIpcCloseMemHandle(s->peers.p[r]);
  if (s->comm) g_nccl.CommDestroy(s->comm);
  cudaFree(s->d_state); cudaFree(s->d_partials); cudaFree(s->d_sums); cudaFree(s->d_pose);
  cudaFree(s->d_ctl); cudaFree(s->d_cta_sums); cudaFree(s->xchg);
  if (s->h_done) cudaFreeHost(s->h_done);
  delete s;
  return EA_OK;
}

// Exchange buffers: every rank exports its own with cudaIpc, the 64-byte handles travel once through ncclAllGather (the
// only NCCL traffic of the persistent path), every rank maps its peers' buffers.  Returns EA_OK with in_kernel == false
// when the devices cannot reach each other (the host-driven NCCL path then serves).
static int shard_open_peers(ea_shard* s) {
  cudaStream_t st = s->ctx->stream;
  CU(cudaMalloc((void**)&s->xchg, sizeof(ShardXchg)));
  CU(cudaMemset(s->xchg, 0, sizeof(ShardXchg)));
  for (int r = 0; r < EA_SHARD_MAX_WORLD; ++r) s->peers.p[r] = s->xchg;
  if (s->world == 1) { s->in_kernel = true; return EA_OK; }
  if (s->world > EA_SHARD_MAX_WORLD) return EA_OK;
  cudaIpcMemHandle_t mine;
  if (cudaIpcGetMemHandle(&mine, s->xchg) != cudaSuccess) { cudaGetLastError(); return EA_OK; }
  unsigned char* d_all = nullptr;
  CU(cudaMalloc((void**)&d_all, size_t(s->world) * sizeof(mine)));
  CU(cudaMemcpyAsync(d_all + size_t(s->rank) * sizeof(mine), &mine, sizeof(mine), cudaMemcpyHostToDevice, st));
  ncclResult_t nr = g_nccl.AllGather(d_all + size_t(s->rank) * sizeof(mine), d_all, sizeof(mine), ncclChar, s->comm, st);
  if (nr != ncclSuccess) { cudaFree(d_all); return ea_fail(EA_ERR_NCCL, "ncclAllGather(ipc handles) -> %s", g_nccl.GetErrorString(nr)); }
  std::vector<cudaIpcMemHandle_t> all(static_cast<size_t>(s->world));
  cudaError_t ce = cudaMemcpyAsync(all.data(), d_all, size_t(s->world) * sizeof(mine), cudaMemcpyDeviceToHost, st);
  if (ce == cudaSuccess) ce = cudaStreamSynchronize(st);
  cudaFree(d_all);
  if (ce != cudaSuccess) return ea_fail(EA_ERR_CUDA, "ipc handle exchange: %s", cudaGetErrorString(ce));
  bool ok = true;
  for (int r = 0; r < s->world && ok; ++r) {
    if (r == s->rank) continue;
    void* p = nullptr;
    if (cudaIpcOpenMemHandle(&p, all[size_t(r)], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { cudaGetLastError(); ok = false; break; }
    s->peers.p[r] = static_cast<ShardXchg*>(p);
    s->peer_open[r] = true;
  }
  // all ranks must agree on the path: one that cannot map its peers sends everyone to the NCCL path
  int* d_ok = nullptr;
  CU(cudaMalloc((void**)&d_ok, sizeof(int)));
  const int mine_ok = ok ? 1 : 0;
  CU(cudaMemcpyAsync(d_ok, &mine_ok, sizeof(int), cudaMemcpyHostToDevice, st));
  nr = g_nccl.AllReduce(d_ok, d_ok, 1, ncclInt, ncclMin, s->comm, st);
  int all_ok = 0;
  if (nr == ncclSuccess) { cudaMemcpyAsync(&all_ok, d_ok, sizeof(int), cudaMemcpyDeviceToHost, st); cudaStreamSynchronize(st); }
  cudaFree(d_ok);
  if (nr != ncclSuccess) return ea_fail(EA_ERR_NCCL, "ncclAllReduce(path agreement) -> %s", g_nccl.GetErrorString(nr));
  s->in_kernel = all_ok == 1;
  return EA_OK;
}

int ea_shard_create(ea_context* ctx, const uint8_t id128[128], int rank, int world, ea_shard** out) {
  if (!ctx || !out) return ea_fail(EA_ERR_INVALID_ARG, "null argument");
  *out = nullptr;
  if (world < 1 || rank < 0 || rank >= world) return ea_fail(EA_ERR_INVALID_ARG, "bad rank/world %d/%d", rank, world);
  CU(cudaSetDevice(ctx->device));
  ea_shard* s = new (std::nothrow) ea_shard();
  if (!s) return ea_fail(EA_ERR_INVALID_ARG, "out of host memory");
  s->ctx = ctx; s->rank = rank; s->world = world;
  int rc = EA_OK;
  if (world > 1) {
    if (!id128) rc = ea_fail(EA_ERR_INVALID_ARG, "world > 1 needs the NCCL unique id");
    if (!rc) rc = load_nccl();
    if (!rc) {
      ncclUniqueId id;
      std::memcpy(&id, id128, 128);
      ncclResult_t r = g_nccl.CommInitRank(&s->comm, world, id, rank);
      if (r != ncclSuccess) rc = ea_fail(EA_ERR_NCCL, "ncclCommInitRank -> %s", g_nccl.GetErrorString(r));
    }
  }
  s->n_blocks = ctx->sm_count * 2;
  auto alloc = [&](void** p, size_t bytes) { if (!rc && cudaMalloc(p, bytes) != cudaSuccess) rc = ea_fail(EA_ERR_CUDA, "ea_shard_create: cudaMalloc(%zu) failed", bytes); };
  alloc((void**)&s->d_state, sizeof(ShardState));
  alloc((void**)&s->d_partials, size_t(s->n_blocks) * EA_SUMS * 8);
  alloc((void**)&s->d_sums, EA_SUMS * 8);
  alloc((void**)&s->d_pose, 7 * 8);
  alloc((void**)&s->d_ctl, sizeof(ShardCtl));
  alloc((void**)&s->d_cta_sums, size_t(ctx->sm_count) * 32 * 8);
  if (!rc && cudaHostAlloc((void**)&s->h_done, sizeof(int), cudaHostAllocDefault) != cudaSuccess) rc = ea_fail(EA_ERR_CUDA, "ea_shard_create: cudaHostAlloc failed");
  if (!rc) rc = shard_open_peers(s);
  if (!rc) {
    const char* mode = getenv("EA_SHARD_MODE");      // "nccl": force the host-driven path (A/B measurements)
    if (mode && !strcmp(mode, "nccl")) s->in_kernel = false;
    int khz = 0;
    cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, ctx->device);
    s->clock_khz = khz > 0 ? double(khz) : 1.0;
  }
  if (rc) { ea_shard_destroy(s); return rc; }     // nothing allocated above outlives a failed create
  *out = s;
  return EA_OK;
}

// Last solve of this shard: out[0] evaluations, out[1] device ms of the whole solve, out[2..5] microseconds per evaluation
// spent in {evaluation of the slice (CTA 0's view), grid reduce, cross-rank all-reduce, LM step}, out[6] 1 if the persistent
// in-kernel path ran (0: host-driven launches + ncclAllReduce), out[7] kernel launches of the solve.
int ea_shard_profile(ea_shard* s, double out[8]) {
  if (!s || !out) return ea_fail(EA_ERR_INVALID_ARG, "null argument");
  for (int i = 0; i < 8; ++i) out[i] = s->prof[i];
  return EA_OK;
}

static int shard_solve_persistent(ea_shard* s, ea_frameset* ref, int ref_slot, ea_frameset* now, int now_slot, int level, double* pose7,
                                  const ea_solve_params* sp, ea_summary* summary, int n_res, int j0, int j1) {
  ea_context* c = s->ctx;
  cudaStream_t st = c->stream;
  if (s->poisoned) return ea_fail(EA_ERR_STATE, "this shard lost a peer in an earlier solve; create a new one");
  EaLevelDesc rd = ref->h_desc[size_t(ref_slot) * EA_MAX_LEVELS + level];
  EaLevelDesc nd = now->h_desc[size_t(now_slot) * EA_MAX_LEVELS + level];
  EaLevelGeom rg = ref->geom[level], ng = now->geom[level];
  double ids = ref->inv_depth_unit;
  ea_solve_params spv = *sp;
  EaEvalConsts lossv = ea_eval_consts(sp->loss_type, sp->loss_scale, sp->point_stride);
  // one CTA per SM at most, at least ~2 iterations of the evaluation loop per CTA; every rank sizes its grid for its own slice
  int grid = std::max(1, std::min(c->sm_count, (j1 - j0 + 1023) / 1024));
  CU(cudaMemcpyAsync(s->d_pose, pose7, 56, cudaMemcpyHostToDevice, st));
  k_shard_ctl_init<<<1, 1, 0, st>>>(s->d_ctl, s->d_pose, rg, ng, rd.pts_mode == EA_POINTS_XYZ ? 1 : 0);
  cudaEvent_t e0, e1;
  CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
  CU(cudaEventRecord(e0, st));
  ShardCtl* ctl = s->d_ctl; double* cta = s->d_cta_sums; ShardPeers peers = s->peers; int rank = s->rank, world = s->world;
  unsigned long long epoch0 = s->epoch;
  void* args[] = {&rd, &nd, &rg, &ng, &ids, &spv, &lossv, &ctl, &cta, &peers, &rank, &world, &epoch0, &j0, &j1};
  cudaError_t le = cudaLaunchCooperativeKernel((const void*)k_shard_solve<EA_SOLVE_THREADS>, dim3(unsigned(grid)), dim3(EA_SOLVE_THREADS), args, 0, st);
  cudaEventRecord(e1, st);
  c->launches += 2;
  if (le != cudaSuccess) { cudaEventDestroy(e0); cudaEventDestroy(e1); return ea_fail(EA_ERR_CUDA, "shard solve launch: %s", cudaGetErrorString(le)); }
  ShardCtl h;
  cudaError_t ce = cudaMemcpyAsync(&h, s->d_ctl, sizeof h, cudaMemcpyDeviceToHost, st);
  if (ce == cudaSuccess) ce = cudaStreamSynchronize(st);
  float ms = 0.f;
  if (ce == cudaSuccess) cudaEventElapsedTime(&ms, e0, e1);
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  if (ce != cudaSuccess) return ea_fail(EA_ERR_CUDA, "shard solve: %s", cudaGetErrorString(ce));
  s->epoch += (unsigned long long)h.lm.evals + 1;
  const double ev = std::max(1, h.lm.evals), us = 1e3 / s->clock_khz;
  s->prof[0] = h.lm.evals; s->prof[1] = ms;
  s->prof[2] = double(h.prof[0]) * us / ev; s->prof[3] = double(h.prof[1]) * us / ev; s->prof[4] = double(h.prof[2]) * us / ev; s->prof[5] = double(h.prof[3]) * us / ev;
  s->prof[6] = 1.0; s->prof[7] = 2.0;
  for (int i = 0; i < 7; ++i) pose7[i] = h.lm.x[i];
  if (summary) {
    summary->termination = h.lm.term; summary->iterations = h.lm.iter; summary->accepted = h.lm.accepted; summary->rejected = h.lm.rejected;
    summary->n_residuals = n_res; summary->evaluations = h.lm.evals;
    summary->initial_cost = h.lm.initial_cost; summary->final_cost = h.lm.cost; summary->truncated = 0; summary->reserved = 0;
  }
  if (h.error) {
    s->poisoned = true;
    return ea_fail(EA_ERR_NCCL, "point-sharded solve: %s", h.error == 1 ? "a peer rank stopped answering the in-kernel all-reduce" : "the grid was never released (a CTA or peer is gone)");
  }
  return EA_OK;
}

int ea_shard_solve(ea_shard* s, ea_frameset* ref, int ref_slot, ea_frameset* now, int now_slot, int level, double* pose7,
                   const ea_solve_params* sp, ea_summary* summary) {
  if (!s || !ref || !now || !pose7 || !sp) return ea_fail(EA_ERR_INVALID_ARG, "null argument");
  if (level < 0 || level >= ref->p.n_levels || level >= now->p.n_levels) return ea_fail(EA_ERR_INVALID_ARG, "bad level");
  if (ref_slot < 0 || ref_slot >= ref->n_slots || now_slot < 0 || now_slot >= now->n_slots) return ea_fail(EA_ERR_INVALID_ARG, "bad slot");
  int rc = ea_check_solve_params(sp);
  if (rc) return rc;
  ea_context* c = s->ctx;
  CU(cudaSetDevice(c->device));
  cudaStream_t st = c->stream;
  int n_pts = 0;
  rc = ea_frameset_get_num_points(ref, ref_slot, level, &n_pts);
  if (rc) return rc;
  const int n_res = (n_pts + sp->point_stride - 1) / sp->point_stride;
  // this rank's contiguous slice of the ordered residual list
  const int j0 = int((long long)n_res * s->rank / s->world), j1 = int((long long)n_res * (s->rank + 1) / s->world);
  if (s->in_kernel) return shard_solve_persistent(s, ref, ref_slot, now, now_slot, level, pose7, sp, summary, n_res, j0, j1);
  cudaEvent_t pe0, pe1;
  CU(cudaEventCreate(&pe0)); CU(cudaEventCreate(&pe1));
  CU(cudaEventRecord(pe0, st));
  const int64_t launches0 = c->launches;
  const EaLevelDesc& rd = ref->h_desc[size_t(ref_slot) * EA_MAX_LEVELS + level];
  const EaLevelDesc& nd = now->h_desc[size_t(now_slot) * EA_MAX_LEVELS + level];
  const double ids = ref->inv_depth_unit;
  int nb = s->n_blocks;
  const int per_block = 2048;
  if ((j1 - j0 + per_block - 1) / per_block < nb) nb = std::max(1, (j1 - j0 + per_block - 1) / per_block);
  CU(cudaMemcpyAsync(s->d_pose, pose7, 56, cudaMemcpyHostToDevice, st));
  k_shard_init<<<1, 1, 0, st>>>(s->d_state, s->d_pose);
  c->launches++;
  const int max_evals = sp->max_num_iterations + 2;
  int evals = 0;
  *s->h_done = 0;
  while (evals < max_evals && !*s->h_done) {
    const int chunk = std::min(8, max_evals - evals);
    for (int i = 0; i < chunk; ++i) {
      cudaError_t le = ea_launch_eval_sums(rd, nd, ref->geom[level], now->geom[level], ids, *sp, s->d_state->cand, &s->d_state->done, j0, j1, nb, s->d_partials, st);
      if (le != cudaSuccess) return ea_fail(EA_ERR_CUDA, "shard eval launch: %s", cudaGetErrorString(le));
      k_shard_reduce<<<1, 32, 0, st>>>(s->d_state, s->d_partials, nb, s->d_sums);
      if (s->world > 1) NC(g_nccl.AllReduce(s->d_sums, s->d_sums, EA_SUMS, ncclDouble, ncclSum, s->comm, st));
      k_shard_lm<<<1, 32, 0, st>>>(s->d_state, s->d_sums, *sp);
      c->launches += 3;
    }
    evals += chunk;
    CU(cudaMemcpyAsync(s->h_done, &s->d_state->done, sizeof(int), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
  }
  cudaEventRecord(pe1, st);
  ShardState h;
  CU(cudaMemcpy(&h, s->d_state, sizeof h, cudaMemcpyDeviceToHost));
  float pms = 0.f;
  cudaEventSynchronize(pe1); cudaEventElapsedTime(&pms, pe0, pe1);
  cudaEventDestroy(pe0); cudaEventDestroy(pe1);
  for (int i = 0; i < 8; ++i) s->prof[i] = 0.0;
  s->prof[0] = h.lm.evals; s->prof[1] = pms; s->prof[7] = double(c->launches - launches0);
  for (int i = 0; i < 7; ++i) pose7[i] = h.lm.x[i];
  if (summary) {
    summary->termination = h.done ? h.lm.term : EA_TERM_NO_CONVERGENCE;
    summary->iterations = h.lm.iter; summary->accepted = h.lm.accepted; summary->rejected = h.lm.rejected;
    summary->n_residuals = n_res; summary->evaluations = h.lm.evals;
    summary->initial_cost = h.lm.initial_cost; summary->final_cost = h.lm.cost; summary->truncated = 0; summary->reserved = 0;
  }
  return EA_OK;
}


// ---- multi-camera problems: every view adds its residual blocks to the same 6-DoF problem ----------------------------
// (standalone_edge_align.cpp:791-803 / 3204-3219: one AddResidualBlock loop per camera with EAResidue /
//  EAResidueSecondCam / EAResidueEx / EAResidueSecondCamEx, all on the same b_quat_a, b_t_a)
static int view_xf(const ea_view& v, EaViewXf& X) {
  std::memset(&X, 0, sizeof X);
  X.use_rig = v.use_rig != 0; X.use_dist = v.use_distortion != 0;
  for (int i = 0; i < 12; ++i) { X.T21[i] = v.cam_T_first[i]; X.T12[i] = v.first_T_cam[i]; }
  if (!X.use_rig) { for (int i = 0; i < 12; ++i) X.T21[i] = X.T12[i] = (i % 5 == 0) ? 1.0 : 0.0; }
  for (int i = 0; i < 5; ++i) X.dist[i] = X.use_dist ? v.dist[i] : 0.0;
  return EA_OK;
}
static int check_view(const ea_view& v, int level) {
  if (!v.ref || !v.now) return ea_fail(EA_ERR_INVALID_ARG, "view with a null frameset");
  if (v.ref->ctx->device != v.now->ctx->device) return ea_fail(EA_ERR_INVALID_ARG, "view framesets on different devices");
  if (level < 0 || level >= v.ref->p.n_levels || level >= v.now->p.n_levels) return ea_fail(EA_ERR_INVALID_ARG, "bad level");
  if (v.ref_slot < 0 || v.ref_slot >= v.ref->n_slots || v.now_slot < 0 || v.now_slot >= v.now->n_slots) return ea_fail(EA_ERR_INVALID_ARG, "bad slot");
  return EA_OK;
}

int ea_eval_views(ea_context* c, int n_views, const ea_view* views, int level, const double* pose7, const ea_solve_params* sp,
                  int* n_residuals, double* raw, double* residuals, double* jac, double* sums28, int* failed) {
  if (!c || !views || n_views < 1 || !pose7 || !sp) return ea_fail(EA_ERR_INVALID_ARG, "null argument");
  { const int prc = ea_check_solve_params(sp); if (prc) return prc; }
  CU(cudaSetDevice(c->device));
  cudaStream_t st = c->stream;
  std::vector<int> nres(n_views);
  int total = 0;
  for (int i = 0; i < n_views; ++i) {
    int rc = check_view(views[i], level);
    if (rc) return rc;
    int n_pts = 0;
    rc = ea_frameset_get_num_points(views[i].ref, views[i].ref_slot, level, &n_pts);
    if (rc) return rc;
    nres[i] = (n_pts + sp->point_stride - 1) / sp->point_stride;
    total += nres[i];
  }
  if (n_residuals) *n_residuals = total;
  CU(cudaMemcpyAsync(c->d_pose, pose7, 56, cudaMemcpyHostToDevice, st));
  CU(cudaMemsetAsync(c->d_failed, 0, sizeof(int), st));
  int rc = ea_ensure_tmp(c, size_t(std::max(total, 1)) * 8 * sizeof(double) + size_t(n_views) * 64 * EA_SUMS * 8);
  if (rc) return rc;
  double* d_raw = (double*)c->d_tmp; double* d_res = d_raw + total; double* d_jac = d_res + total; double* d_part = d_jac + size_t(total) * 6;
  int off = 0, nb_total = 0;
  for (int i = 0; i < n_views; ++i) {
    const ea_view& v = views[i];
    const EaLevelDesc& rd = v.ref->h_desc[size_t(v.ref_slot) * EA_MAX_LEVELS + level];
    const EaLevelDesc& nd = v.now->h_desc[size_t(v.now_slot) * EA_MAX_LEVELS + level];
    EaViewXf X; view_xf(v, X);
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
  if (sums28) {
    double t[EA_SUMS] = {0};
    for (int b2 = 0; b2 < nb_total; ++b2) for (int k = 0; k < EA_SUMS; ++k) t[k] += h[size_t(b2) * EA_SUMS + k];
    sums28[0] = t[28];
    for (int k = 0; k < 6; ++k) sums28[1 + k] = t[21 + k];
    for (int k = 0; k < 21; ++k) sums28[7 + k] = t[k];
  }
  return EA_OK;
}

int ea_solve_views(ea_context* c, int n_views, const ea_view* views, int level, double* pose7, const ea_solve_params* sp,
                   ea_summary* summary) {
  if (!c || !views || n_views < 1 || !pose7 || !sp) return ea_fail(EA_ERR_INVALID_ARG, "null argument");
  { const int prc = ea_check_solve_params(sp); if (prc) return prc; }
  CU(cudaSetDevice(c->device));
  cudaStream_t st = c->stream;
  std::vector<int> nres(n_views), nb(n_views);
  int total = 0, nb_total = 0;
  for (int i = 0; i < n_views; ++i) {
    int rc = check_view(views[i], level);
    if (rc) return rc;
    int n_pts = 0;
    rc = ea_frameset_get_num_points(views[i].ref, views[i].ref_slot, level, &n_pts);
    if (rc) return rc;
    nres[i] = (n_pts + sp->point_stride - 1) / sp->point_stride;
    nb[i] = nres[i] > 0 ? std::max(1, std::min(c->sm_count, (nres[i] + 2047) / 2048)) : 0;
    total += nres[i]; nb_total += nb[i];
  }
  // One persistent cooperative kernel for the whole solve (k_views_solve).  View descriptors, control block and CTA totals live
  // in the context's scratch (allocated on first use, grown on demand): no allocation on the path of a solve.
  const int grid = std::max(1, std::min(c->sm_count, (total + 1023) / 1024));
  const size_t off_ctl = (size_t(n_views) * sizeof(ViewDev) + 255) & ~size_t(255);
  const size_t off_part = off_ctl + ((sizeof(ShardCtl) + 255) & ~size_t(255));
  const size_t need = off_part + size_t(grid) * 32 * 8;
  if (c->views_cap < need) {
    CU(cudaStreamSynchronize(st));
    if (c->d_views) { cudaFree(c->d_views); c->d_views = nullptr; c->views_cap = 0; }
    CU(cudaMalloc(&c->d_views, need));
    c->views_cap = need;
  }
  char* vb = static_cast<char*>(c->d_views);
  ViewDev* d_vd = reinterpret_cast<ViewDev*>(vb);
  ShardCtl* d_ctl = reinterpret_cast<ShardCtl*>(vb + off_ctl);
  double* d_partials = reinterpret_cast<double*>(vb + off_part);
  std::vector<ViewDev> hv(static_cast<size_t>(n_views));
  for (int i = 0; i < n_views; ++i) {
    const ea_view& v = views[i];
    ViewDev& D = hv[size_t(i)];
    D.rd = v.ref->h_desc[size_t(v.ref_slot) * EA_MAX_LEVELS + level];
    D.nd = v.now->h_desc[size_t(v.now_slot) * EA_MAX_LEVELS + level];
    D.rg = v.ref->geom[level]; D.ng = v.now->geom[level];
    view_xf(v, D.X);
    D.inv_depth_scale = v.ref->inv_depth_unit;
    D.n_res = nres[i]; D.xyz = D.rd.pts_mode == EA_POINTS_XYZ ? 1 : 0;
  }
  (void)nb; (void)nb_total;
  CU(cudaMemcpyAsync(d_vd, hv.data(), hv.size() * sizeof(ViewDev), cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(c->d_pose, pose7, 56, cudaMemcpyHostToDevice, st));
  k_shard_ctl_init<<<1, 1, 0, st>>>(d_ctl, c->d_pose, hv[0].rg, hv[0].ng, hv[0].xyz);
  ea_solve_params spv = *sp;
  const ViewDev* vd_arg = d_vd; int nv = n_views;
  void* args[] = {&vd_arg, &nv, &spv, &d_ctl, &d_partials};
  cudaError_t le = cudaLaunchCooperativeKernel((const void*)k_views_solve, dim3(unsigned(grid)), dim3(GV_THREADS), args, 0, st);
  c->launches += 2;
  if (le != cudaSuccess) return ea_fail(EA_ERR_CUDA, "views solve launch: %s", cudaGetErrorString(le));
  ShardCtl h;
  CU(cudaMemcpyAsync(&h, d_ctl, sizeof h, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));      // (hv must outlive the upload)
  if (h.error) return ea_fail(EA_ERR_CUDA, "views solve: the persistent kernel lost a CTA (bounded wait expired)");
  for (int i = 0; i < 7; ++i) pose7[i] = h.lm.x[i];
  if (summary) {
    summary->termination = h.done ? h.lm.term : EA_TERM_NO_CONVERGENCE;
    summary->iterations = h.lm.iter; summary->accepted = h.lm.accepted; summary->rejected = h.lm.rejected;
    summary->n_residuals = total; summary->evaluations = h.lm.evals;
    summary->initial_cost = h.lm.initial_cost; summary->final_cost = h.lm.cost;
  }
  return EA_OK;
}

}  // extern "C"
