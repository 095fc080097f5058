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
  ea_lm_load_warp(lm, st->lm, lane);
  __syncwarp();
  const int cmd = ea_lm_advance_warp(lm, local, sp, lane);
  __syncwarp();
  ea_lm_store_warp(st->lm, lm, lane);
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
// Every wait is bounded (EA_GRID_SPIN_LIMIT polls): a lost peer ends the solve with EA_TERM_FAILURE_PEER instead of hanging
// the GPU.
#define EA_SHARD_MAX_WORLD 8
struct ShardXchg {                                  // lives in cudaIpc-shared device memory, one per rank
  // Self-validating 8-byte packets {32 data bits, 32-bit epoch tag}, two per double (the "LL" idea of NCCL): a packet is one
  // store and one load, so there is no flag to order behind the data -- no system-scope fence, no second NVLink round trip.
  unsigned long long ll[2][EA_SHARD_MAX_WORLD][64]; // [evaluation parity][source rank][2 x 32 sums]
};
struct ShardPeers { ShardXchg* p[EA_SHARD_MAX_WORLD]; };
template <int THREADS>
__global__ void __launch_bounds__(THREADS, 1) k_shard_solve(EaLevelDesc rd, EaLevelDesc nd, EaLevelGeom rg, EaLevelGeom ng,
                                                            double inv_depth_scale, ea_solve_params sp, EaEvalConsts loss, EaGridCtl* ctl,
                                                            double* partials /*[grid][32]*/, ShardPeers peers, int rank, int world,
                                                            unsigned long long epoch0, int j_begin, int j_end) {
  __shared__ double part[THREADS / 32][EA_NSUM];
  __shared__ double cpart[THREADS / 32];
  __shared__ double wsum[THREADS / 32][32];
  __shared__ int s_stop, s_late;
  __shared__ EaLmState s_lm;      // CTA 0 only: the LM state stays in its shared memory for the whole solve
  __shared__ __align__(2 * EA_STAGE_SLOT * 8) uint2 stage[2][EA_STAGE_SLOT];   // cp.async staging of the point stream (ea_eval_slice: aligned to its size)
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n = j_end - j_begin;
  const int j0 = j_begin + int((long long)n * blockIdx.x / gridDim.x), j1 = j_begin + int((long long)n * (blockIdx.x + 1) / gridDim.x);
  const float2 affine = *nd.dt_affine;
  const float* dt_pad = nd.dt - ea_dt_origin_offset(nd.w);
  const bool xyz = rd.pts_mode == EA_POINTS_XYZ;
  if (blockIdx.x == 0 && warp == 0) ea_lm_load_warp(s_lm, ctl->lm, lane);   // the reducer CTA keeps the LM state (initialised by k_shard_ctl_init)
  for (unsigned long long e = 1;; ++e) {
    if (ea_grid_wait(ctl, e, s_stop)) break;   // (e == 1 is released by the host-side initialisation)
    long long t0 = 0;
    if (blockIdx.x == 0 && tid == 0) t0 = clock64();
    EaPose P;
    {   // the candidate's folded pose, written by the LM thread of the previous round (L2: bypass the non-coherent L1)
      const double* src = reinterpret_cast<const double*>(&ctl->P);
      double* dst = reinterpret_cast<double*>(&P);
#pragma unroll
      for (int i = 0; i < int(sizeof(EaPose) / 8); ++i) dst[i] = __ldcg(src + i);
    }
    if (xyz) ea_eval_slice<true, THREADS>(rd.pts, dt_pad, affine, ng, inv_depth_scale, loss, sp.point_stride, P, j0, j1, part, cpart, !(e & 1));
    else {
      const bool rev = !(e & 1);
      ea_eval_slice<false, THREADS>(rd.pts, dt_pad, affine, ng, inv_depth_scale, loss, sp.point_stride, P, j0, j1, part, cpart, rev, &stage[0][0], e > 1, true, !rev);
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
          while (ea_ld_acquire(&ctl->ticket) < want) { if (++spins > EA_GRID_SPIN_LIMIT) { late = 1; break; } }
          s_late = late;
        }
      }
    }
    if (blockIdx.x != 0) continue;
    __syncthreads();
    // ---- CTA 0: grid reduce ----
    __threadfence();
    long long t1 = clock64();
    double tot = ea_grid_total<THREADS / 32>(partials, wsum, warp, lane);
    if (warp == 0) {
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
            if (++spins > EA_GRID_SPIN_LIMIT) { err = 1; break; }
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
      if (done) ea_lm_store_warp(ctl->lm, s_lm, lane);   // the host reads the final state from global memory
      __threadfence();
      __syncwarp();
      if (lane == 0) {
        ctl->done = done;
        const long long t4 = clock64();
        ctl->prof[1] += t2 - t1; ctl->prof[2] += t3 - t2; ctl->prof[3] += t4 - t3; ctl->prof[4] += 1;
        __threadfence();
        ea_st_release(&ctl->go, e + 1);
      }
    }
  }
  if (s_stop == 2 && tid == 0) ctl->error = 2;   // the release never came (a CTA of this grid or a peer rank is gone)
}

__global__ void k_shard_init(ShardState* st, const double* pose7) {
  EaLmState& L = st->lm;
  ea_lm_restart(L);
  L.cost = 0.0; L.initial_cost = 0.0;   // read by the host even when the solve ends without an evaluation
  for (int i = 0; i < 7; ++i) { L.x[i] = pose7[i]; L.cand[i] = pose7[i]; st->cand[i] = pose7[i]; }
  st->done = 0; st->started = 1;
}

}  // namespace

__global__ void k_shard_ctl_init(EaGridCtl* ctl, const double* pose7, EaLevelGeom rg, EaLevelGeom ng, int xyz) {
  EaLmState& L = ctl->lm;
  ea_lm_restart(L);
  L.cost = 0.0; L.initial_cost = 0.0;   // read by the host even when the solve ends without an evaluation
  for (int i = 0; i < 7; ++i) { L.x[i] = pose7[i]; L.cand[i] = pose7[i]; }
  EaPose P;
  if (xyz) ea_pose_setup<true>(L.cand, rg, ng, P); else ea_pose_setup<false>(L.cand, rg, ng, P);
  ctl->P = P;
  ctl->ticket = 0; ctl->done = 0; ctl->error = 0;
  for (int k = 0; k < 6; ++k) ctl->prof[k] = 0;
  __threadfence();
  ctl->go = 1;
}

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
  EaGridCtl* d_ctl = nullptr;
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
  alloc((void**)&s->d_ctl, sizeof(EaGridCtl));
  alloc((void**)&s->d_cta_sums, size_t(ctx->sm_count) * 32 * 8);
  if (!rc && cudaHostAlloc((void**)&s->h_done, sizeof(int), cudaHostAllocDefault) != cudaSuccess) rc = ea_fail(EA_ERR_CUDA, "ea_shard_create: cudaHostAlloc failed");
  if (!rc) rc = shard_open_peers(s);
  if (!rc) {
    const char* mode = getenv("EA_SHARD_MODE");      // "nccl": force the host-driven path (the one GPUs without peer access take)
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
  EaGridCtl* ctl = s->d_ctl; double* cta = s->d_cta_sums; ShardPeers peers = s->peers; int rank = s->rank, world = s->world;
  unsigned long long epoch0 = s->epoch;
  void* args[] = {&rd, &nd, &rg, &ng, &ids, &spv, &lossv, &ctl, &cta, &peers, &rank, &world, &epoch0, &j0, &j1};
  cudaError_t le = cudaLaunchCooperativeKernel((const void*)k_shard_solve<EA_SOLVE_THREADS>, dim3(unsigned(grid)), dim3(EA_SOLVE_THREADS), args, 0, st);
  cudaEventRecord(e1, st);
  c->launches += 2;
  if (le != cudaSuccess) { cudaEventDestroy(e0); cudaEventDestroy(e1); return ea_fail(EA_ERR_CUDA, "shard solve launch: %s", cudaGetErrorString(le)); }
  EaGridCtl h;
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
  if (summary) *summary = ea_lm_summary(h.lm, n_res, 0);
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
  if (n_res == 0) {   // as ea_solve_batch: nothing to align, pose untouched, no launch (every rank sees the same count)
    for (int i = 0; i < 8; ++i) s->prof[i] = 0.0;
    if (summary) { *summary = ea_summary{}; summary->termination = EA_TERM_SKIPPED_NO_POINTS; }
    return EA_OK;
  }
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
    *summary = ea_lm_summary(h.lm, n_res, 0);
    summary->termination = h.done ? h.lm.term : EA_TERM_NO_CONVERGENCE;
  }
  return EA_OK;
}

}  // extern "C"
