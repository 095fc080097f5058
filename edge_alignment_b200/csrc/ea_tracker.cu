// Multi-stream frame-to-keyframe tracker: the caller of the pose-solve path, re-stated from the reference's
// consumer loop (src/ea.cpp:87-131) and SolveEA's setRefFrame / setNowFrame / setAsCERESProblem sequence
// (src/ea.cpp:184-199), batched over n_streams independent cameras.  Every frame is preprocessed once
// (its DT when it arrives, its edge points only if it becomes a key frame); poses are warm-started from the
// previous frame and never leave the device between steps.
//
// Key-frame policy mode (ea_tracker_set_keyframe_policy) moves the key-frame decision onto the device, per stream: one
// thread per stream (ea_k_keyframe_policy) reads the pose and summary the solve just wrote, applies the rule, composes the
// world pose and rewrites that stream's slot tables.  Every frame after the first is preprocessed for both roles, but its point
// lists are only built (EA_COMPACT_ONLY, after the policy kernel, gated by its key_reasons) if it was promoted; its ref_bits and
// depth pyramid wait in its slot until then, and the level-0 depth is read from the step's input buffer, so the host path
// releases its staging buffers after that compaction.  Slot bookkeeping, stream s owning slots 3s, 3s+1, 3s+2:
//   K_t  key slot solve(t) reads      d_key_tab[t & 1]   written by policy(t-1)
//   N_t  slot frame t lands in        d_new_tab[t % 3]   written by policy(t-2); read by prep(t), solve(t), policy(t-1), policy(t)
//   K_{t+1} = promoted(t) ? N_t : K_t, and N_{t+2} is the slot that is neither K_{t+1} nor N_{t+1}: one of the two solve(t)
//   read, so prep(t+2) -- which already waits for ev_solved of frame t, recorded after policy(t) -- may overwrite it.
// Prep(t+1) runs beside policy(t) and reads N_{t+1} while policy(t) writes N_{t+2}: three new-slot tables keep them apart
// (and keep the tables of the latest solve intact for ea_tracker_probe_gather); two key tables keep K_t, which the solve
// read, apart from K_{t+1}.
#include <cmath>
#include <cstring>
#include <new>

#include "ea_internal.h"

// a key frame whose point list was cut at max_points is reported with the results that used it (EA_ERR_CAPACITY; the
// poses and summaries are still delivered)
static int tracker_check_truncated(const ea_summary* s, int n_streams, int n_levels) {
  for (int i = 0; i < n_streams * n_levels; ++i)
    if (s[i].truncated)
      return ea_fail(EA_ERR_CAPACITY, "stream %d level %d: the key frame's point list was truncated at max_points; raise ea_frame_params.max_points",
                     i / n_levels, i % n_levels);
  return EA_OK;
}

struct ea_tracker {
  ea_context* ctx = nullptr;
  ea_frameset* fs = nullptr;       // 3 * n_streams slots: stream s owns slots 3s, 3s+1, 3s+2 (key frame, frame being aligned, frame being preprocessed)
  ea_solve_params sp;
  int n_streams = 0, interval = 1, n_levels = 1;
  int frame = 0;                   // frames seen so far
  int key_set = 0;                 // slot set currently holding the key frames
  int prev_key = 0, prev_now = -1; // slot sets the most recently enqueued solve reads
  int32_t* d_slots[3] = {nullptr, nullptr, nullptr};   // [n_streams] slot ids of set 0 / 1 / 2
  // frame t+1 is preprocessed on its own stream while frame t is still being aligned: its kernels fill the SMs the
  // persistent solve kernel releases during its tail
  cudaStream_t prep_stream = nullptr;
  cudaEvent_t ev_prep[2] = {nullptr, nullptr}, ev_solved[2] = {nullptr, nullptr};
  int inputs_ready = 0;            // ea_tracker_set_inputs_ready: device inputs are complete at call time (not stream-ordered)
  ea_image_layout layout{EA_IMAGE_BGR8, 0, 0, 0};   // of the step functions' image argument (resolved by ea_tracker_create)
  double* d_poses = nullptr;       // warm-start table [n_streams][7]
  double* d_result = nullptr;      // poses of the latest step [n_streams][7]
  double* d_identity = nullptr;    // [n_streams][7]
  ea_summary* d_summaries = nullptr;
  int32_t* d_order = nullptr;      // longest-first processing order derived from the previous step's summaries
  bool have_order = false;
  // host-input pipeline: frame t+1 is uploaded on a copy stream while frame t is being aligned
  cudaStream_t copy_stream = nullptr;
  uint8_t* stage_bgr[2] = {nullptr, nullptr};   // [n_streams] frames packed dense (ea_upload_frames)
  void* stage_depth[2] = {nullptr, nullptr};
  cudaEvent_t ev_copied[2] = {nullptr, nullptr}, ev_consumed[2] = {nullptr, nullptr}, ev_result[2] = {nullptr, nullptr};
  double* h_poses[2] = {nullptr, nullptr};          // pinned result ring
  ea_summary* h_summaries[2] = {nullptr, nullptr};
  int result_frame[2] = {-1, -1};
  // key-frame policy mode (see the top of the file)
  bool policy_on = false;
  ea_keyframe_policy policy{};
  int32_t* d_key_tab[2] = {nullptr, nullptr};           // [n_streams] K_t in table t & 1
  int32_t* d_new_tab[3] = {nullptr, nullptr, nullptr};  // [n_streams] N_t in table t % 3
  int32_t* d_key_frame = nullptr;  // [n_streams] frame index of the current key frame
  double* d_world = nullptr;       // [n_streams][7] world_T_frame of the latest frame
  double* d_world_key = nullptr;   // [n_streams][7] world_T_key
  ea_track_info* d_info = nullptr; // [n_streams] of the latest frame
  double* h_world[2] = {nullptr, nullptr};              // pinned result ring (ea_tracker_wait_trajectory)
  ea_track_info* h_info[2] = {nullptr, nullptr};
};

// ---- key-frame policy kernel: one thread per stream, fp64 ----------------------------------------------------------------
struct EaKeyPolicyArgs {
  ea_keyframe_policy p;
  int n, frame, n_levels, finest;
  const ea_summary* summaries;     // [n][n_levels] of solve(frame)
  const double* pose;              // [n][7] key_T_frame of solve(frame)
  double* warm;                    // [n][7] warm-start table: identity for promoted streams
  const int32_t* key_in;           // K_frame
  int32_t* key_out;                // K_{frame+1}
  const int32_t* new_cur;          // N_frame
  const int32_t* new_next;         // N_{frame+1}
  int32_t* new_out;                // N_{frame+2}
  int32_t* key_frame;
  double* world;
  double* world_key;
  ea_track_info* info;
};

__global__ void __launch_bounds__(128) ea_k_keyframe_policy(const EaKeyPolicyArgs A) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= A.n) return;
  const double* q = A.pose + size_t(s) * 7;
  const ea_summary S = A.summaries[size_t(s) * A.n_levels + A.finest];
  const bool lost = S.termination == EA_TERM_FAILURE_EVAL_X0 || S.termination == EA_TERM_FAILURE_INVALID_STEPS ||
                    S.termination == EA_TERM_SKIPPED_NO_POINTS;
  const int key_frame = A.key_frame[s];
  int reasons = 0;
  if (A.p.max_interval > 0 && A.frame - key_frame >= A.p.max_interval) reasons |= EA_KEY_INTERVAL;
  double* w = A.world + size_t(s) * 7;
  if (lost) {
    reasons |= EA_KEY_LOST;        // the pose is not trusted: the world pose stays at the previous frame's
  } else {
    const double tn = sqrt(q[4] * q[4] + q[5] * q[5] + q[6] * q[6]);
    const double ang = 2.0 * atan2(sqrt(q[1] * q[1] + q[2] * q[2] + q[3] * q[3]), fabs(q[0]));
    if (A.p.max_translation > 0.0 && tn > A.p.max_translation) reasons |= EA_KEY_TRANSLATION;
    if (A.p.max_rotation > 0.0 && ang > A.p.max_rotation) reasons |= EA_KEY_ROTATION;
    if (A.p.max_cost_per_residual > 0.0 && S.n_residuals > 0 && S.final_cost / S.n_residuals > A.p.max_cost_per_residual)
      reasons |= EA_KEY_COST;
    // world_T_frame = world_T_key o inverse(key_T_frame): q_w = q_k conj(q), t_w = t_k - R(q_w) t
    const double* k = A.world_key + size_t(s) * 7;
    const double bw = q[0], bx = -q[1], by = -q[2], bz = -q[3];
    double ww = k[0] * bw - k[1] * bx - k[2] * by - k[3] * bz;
    double wx = k[0] * bx + k[1] * bw + k[2] * bz - k[3] * by;
    double wy = k[0] * by - k[1] * bz + k[2] * bw + k[3] * bx;
    double wz = k[0] * bz + k[1] * by - k[2] * bx + k[3] * bw;
    const double inv = 1.0 / sqrt(ww * ww + wx * wx + wy * wy + wz * wz);
    ww *= inv; wx *= inv; wy *= inv; wz *= inv;
    // R(q) v = v + 2 qw (u x v) + 2 u x (u x v), u = q_xyz
    const double vx = q[4], vy = q[5], vz = q[6];
    const double cx = wy * vz - wz * vy, cy = wz * vx - wx * vz, cz = wx * vy - wy * vx;
    const double rx = vx + 2.0 * (ww * cx + wy * cz - wz * cy);
    const double ry = vy + 2.0 * (ww * cy + wz * cx - wx * cz);
    const double rz = vz + 2.0 * (ww * cz + wx * cy - wy * cx);
    w[0] = ww; w[1] = wx; w[2] = wy; w[3] = wz;
    w[4] = k[4] - rx; w[5] = k[5] - ry; w[6] = k[6] - rz;
  }
  A.info[s] = ea_track_info{key_frame, reasons};
  const int32_t key = A.key_in[s], cur = A.new_cur[s];
  const int32_t key1 = reasons ? cur : key;
  A.key_out[s] = key1;
  A.new_out[s] = 3 * (cur - cur % 3) + 3 - key1 - A.new_next[s];   // the stream's third slot
  if (reasons) {
    A.key_frame[s] = A.frame;
    double* k = A.world_key + size_t(s) * 7;
    double* p = A.warm + size_t(s) * 7;
    for (int i = 0; i < 7; ++i) { k[i] = w[i]; p[i] = i == 0 ? 1.0 : 0.0; }
  }
}

// tables and world state of frames 0..2 (policy mode, after create / reset); the caller has synchronised the tracker's streams
static int tracker_policy_init(ea_tracker* t) {
  cudaStream_t s = t->ctx->stream;
  const int n = t->n_streams;
  std::vector<int32_t> tab(size_t(n) * 5);
  std::vector<ea_track_info> info(size_t(n), ea_track_info{0, EA_KEY_FIRST});
  for (int i = 0; i < n; ++i) {
    tab[size_t(i)] = 3 * i;                   // K_1: frame 0
    for (int k = 0; k < 3; ++k) tab[size_t(k + 1) * n + i] = 3 * i + k;   // N_0, N_1, N_2
    tab[size_t(4) * n + i] = 0;               // key frame index
  }
  const size_t ib = size_t(n) * sizeof(int32_t), pb = size_t(n) * 7 * 8;
  CU(cudaMemcpyAsync(t->d_key_tab[1], tab.data(), ib, cudaMemcpyHostToDevice, s));
  for (int k = 0; k < 3; ++k) CU(cudaMemcpyAsync(t->d_new_tab[k], tab.data() + size_t(k + 1) * n, ib, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(t->d_key_frame, tab.data() + size_t(4) * n, ib, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(t->d_info, info.data(), size_t(n) * sizeof(ea_track_info), cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(t->d_world, t->d_identity, pb, cudaMemcpyDeviceToDevice, s));
  CU(cudaMemcpyAsync(t->d_world_key, t->d_identity, pb, cudaMemcpyDeviceToDevice, s));
  CU(cudaStreamSynchronize(s));   // the host tables are released on return
  return EA_OK;
}

extern "C" {

int ea_tracker_create(ea_context* ctx, const ea_frame_params* fp, const ea_solve_params* sp, int n_streams,
                      int keyframe_interval, ea_tracker** out) {
  if (!ctx || !fp || !sp || !out) return ea_fail(EA_ERR_INVALID_ARG, "ea_tracker_create: null argument");
  *out = nullptr;
  if (n_streams <= 0 || keyframe_interval <= 0) return ea_fail(EA_ERR_INVALID_ARG, "n_streams and keyframe_interval must be positive");
  ea_tracker* t = new (std::nothrow) ea_tracker();
  if (!t) return ea_fail(EA_ERR_INVALID_ARG, "out of host memory");
  t->ctx = ctx; t->sp = *sp; t->n_streams = n_streams; t->interval = keyframe_interval; t->n_levels = fp->n_levels;
  struct Guard { ea_tracker* t; ~Guard() { if (t) ea_tracker_destroy(t); } } guard{t};    // a failed create leaves nothing behind
  int rc = ea_frameset_create(ctx, fp, 3 * n_streams, &t->fs);
  if (rc) return rc;
  std::vector<int32_t> ss(n_streams);
  std::vector<double> id(size_t(n_streams) * 7, 0.0);
  for (int i = 0; i < n_streams; ++i) id[size_t(i) * 7] = 1.0;
  for (int k = 0; k < 3; ++k) {
    for (int i = 0; i < n_streams; ++i) ss[i] = 3 * i + k;
    CU(cudaMalloc((void**)&t->d_slots[k], n_streams * sizeof(int32_t)));
    CU(cudaMemcpy(t->d_slots[k], ss.data(), n_streams * sizeof(int32_t), cudaMemcpyHostToDevice));
  }
  CU(cudaMalloc((void**)&t->d_poses, id.size() * 8));
  CU(cudaMalloc((void**)&t->d_result, id.size() * 8));
  CU(cudaMalloc((void**)&t->d_identity, id.size() * 8));
  CU(cudaMalloc((void**)&t->d_summaries, size_t(n_streams) * fp->n_levels * sizeof(ea_summary)));
  CU(cudaMalloc((void**)&t->d_order, size_t(n_streams) * sizeof(int32_t)));
  CU(cudaMemcpy(t->d_identity, id.data(), id.size() * 8, cudaMemcpyHostToDevice));
  CU(cudaStreamCreateWithFlags(&t->copy_stream, cudaStreamNonBlocking));
  CU(cudaStreamCreateWithFlags(&t->prep_stream, cudaStreamNonBlocking));
  for (int b = 0; b < 2; ++b) {
    CU(cudaEventCreateWithFlags(&t->ev_prep[b], cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&t->ev_solved[b], cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&t->ev_copied[b], cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&t->ev_consumed[b], cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&t->ev_result[b], cudaEventDisableTiming));
    CU(cudaHostAlloc((void**)&t->h_poses[b], id.size() * 8, cudaHostAllocDefault));
    CU(cudaHostAlloc((void**)&t->h_summaries[b], size_t(n_streams) * fp->n_levels * sizeof(ea_summary), cudaHostAllocDefault));
    CU(cudaHostAlloc((void**)&t->h_world[b], id.size() * 8, cudaHostAllocDefault));
    CU(cudaHostAlloc((void**)&t->h_info[b], size_t(n_streams) * sizeof(ea_track_info), cudaHostAllocDefault));
    CU(cudaMalloc((void**)&t->d_key_tab[b], n_streams * sizeof(int32_t)));
  }
  for (int k = 0; k < 3; ++k) CU(cudaMalloc((void**)&t->d_new_tab[k], n_streams * sizeof(int32_t)));
  CU(cudaMalloc((void**)&t->d_key_frame, n_streams * sizeof(int32_t)));
  CU(cudaMalloc((void**)&t->d_world, id.size() * 8));
  CU(cudaMalloc((void**)&t->d_world_key, id.size() * 8));
  CU(cudaMalloc((void**)&t->d_info, n_streams * sizeof(ea_track_info)));
  rc = ea_resolve_layout(&t->layout, fp->width, fp->height, true, &t->layout);
  if (rc) return rc;
  rc = ea_tracker_reset(t);
  if (rc) return rc;
  guard.t = nullptr;
  *out = t;
  return EA_OK;
}

int ea_tracker_destroy(ea_tracker* t) {
  if (!t) return EA_OK;
  cudaSetDevice(t->ctx->device);
  cudaStreamSynchronize(t->ctx->stream);
  if (t->prep_stream) { cudaStreamSynchronize(t->prep_stream); cudaStreamDestroy(t->prep_stream); }
  cudaFree(t->d_slots[0]); cudaFree(t->d_slots[1]); cudaFree(t->d_slots[2]); cudaFree(t->d_poses); cudaFree(t->d_result);
  cudaFree(t->d_identity); cudaFree(t->d_summaries); cudaFree(t->d_order);
  cudaFree(t->d_new_tab[0]); cudaFree(t->d_new_tab[1]); cudaFree(t->d_new_tab[2]); cudaFree(t->d_key_frame);
  cudaFree(t->d_world); cudaFree(t->d_world_key); cudaFree(t->d_info);
  if (t->copy_stream) { cudaStreamSynchronize(t->copy_stream); cudaStreamDestroy(t->copy_stream); }
  for (int b = 0; b < 2; ++b) {
    cudaFree(t->stage_bgr[b]); cudaFree(t->stage_depth[b]);
    if (t->ev_copied[b]) cudaEventDestroy(t->ev_copied[b]);
    if (t->ev_consumed[b]) cudaEventDestroy(t->ev_consumed[b]);
    if (t->ev_result[b]) cudaEventDestroy(t->ev_result[b]);
    if (t->ev_prep[b]) cudaEventDestroy(t->ev_prep[b]);
    if (t->ev_solved[b]) cudaEventDestroy(t->ev_solved[b]);
    if (t->h_poses[b]) cudaFreeHost(t->h_poses[b]);
    if (t->h_summaries[b]) cudaFreeHost(t->h_summaries[b]);
    if (t->h_world[b]) cudaFreeHost(t->h_world[b]);
    if (t->h_info[b]) cudaFreeHost(t->h_info[b]);
    cudaFree(t->d_key_tab[b]);
  }
  ea_frameset_destroy(t->fs);
  delete t;
  return EA_OK;
}

int ea_tracker_reset(ea_tracker* t) {
  if (!t) return ea_fail(EA_ERR_INVALID_ARG, "null tracker");
  cudaStream_t s = t->ctx->stream;
  const size_t pb = size_t(t->n_streams) * 7 * 8;
  CU(cudaStreamSynchronize(t->prep_stream));
  CU(cudaStreamSynchronize(s));
  t->frame = 0; t->key_set = 0; t->prev_key = 0; t->prev_now = -1; t->result_frame[0] = t->result_frame[1] = -1; t->have_order = false;
  CU(cudaMemcpyAsync(t->d_poses, t->d_identity, pb, cudaMemcpyDeviceToDevice, s));
  CU(cudaMemcpyAsync(t->d_result, t->d_identity, pb, cudaMemcpyDeviceToDevice, s));
  CU(cudaMemsetAsync(t->d_summaries, 0, size_t(t->n_streams) * t->n_levels * sizeof(ea_summary), s));
  if (t->policy_on) return tracker_policy_init(t);
  return EA_OK;
}

int ea_tracker_set_keyframe_policy(ea_tracker* t, const ea_keyframe_policy* p) {
  if (!t) return ea_fail(EA_ERR_INVALID_ARG, "null tracker");
  if (p) {
    if (p->max_interval < 0) return ea_fail(EA_ERR_INVALID_ARG, "max_interval must not be negative");
    const double v[3] = {p->max_translation, p->max_rotation, p->max_cost_per_residual};
    for (double x : v)
      if (!(x >= 0.0) || !std::isfinite(x)) return ea_fail(EA_ERR_INVALID_ARG, "key-frame thresholds must be finite and not negative");
  }
  if (t->frame != 0) return ea_fail(EA_ERR_STATE, "the key-frame policy can only change before the first step (after create or reset)");
  CU(cudaSetDevice(t->ctx->device));
  t->policy_on = p != nullptr;
  if (p) t->policy = *p;
  return t->policy_on ? tracker_policy_init(t) : EA_OK;
}

}  // extern "C"

// input_ready: event after which the frame buffers are complete (host path: the upload); null => the buffers are ordered by
// the context stream (default) or already complete (inputs_ready).
static int tracker_step(ea_tracker* t, const uint8_t* d_bgr, const ea_image_layout& layout, const void* d_depth, cudaEvent_t input_ready,
                        cudaEvent_t consumed) {
  ea_context* c = t->ctx;
  CU(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  const bool first = (t->frame == 0);
  const bool policy = t->policy_on;
  const bool becomes_key = !policy && (t->frame % t->interval) == 0;
  if (policy && !d_depth) return ea_fail(EA_ERR_INVALID_ARG, "key-frame policy mode: any frame may become a key frame, every step needs depth");
  if (becomes_key && !d_depth) return ea_fail(EA_ERR_INVALID_ARG, "frame %d becomes a key frame and needs depth", t->frame);
  // the new frame lands in the slot set that the solve still in flight (frame - 1) does not read
  int cur = 0;
  if (!first && !policy) { while (cur == t->prev_key || cur == t->prev_now || cur == t->key_set) ++cur; }
  const int roles = (first ? 0 : EA_ROLE_NOW) | (becomes_key || policy ? EA_ROLE_REF : 0);
  // policy mode: per-stream slot tables written on the device (see the top of the file)
  const int32_t* d_key_slots = policy ? t->d_key_tab[t->frame & 1] : t->d_slots[t->key_set];
  const int32_t* d_new_slots = policy ? t->d_new_tab[t->frame % 3] : t->d_slots[cur];
  const int fb = t->frame & 1;
  const bool overlap = input_ready != nullptr || t->inputs_ready != 0;   // frame t+1's preprocessing may run beside frame t's solve
  cudaStream_t ps = t->prep_stream;
  if (input_ready) {
    CU(cudaStreamWaitEvent(ps, input_ready, 0));
  } else if (!t->inputs_ready) {   // inputs produced by work enqueued on the context stream: keep that order (no overlap)
    CU(cudaEventRecord(t->ev_prep[fb], s));
    CU(cudaStreamWaitEvent(ps, t->ev_prep[fb], 0));
  }
  if (t->frame >= 3) CU(cudaStreamWaitEvent(ps, t->ev_solved[fb], 0));   // last reader of this slot set: the solve of frame - 2
  // policy mode: frames after the first build their point lists only once the policy kernel has promoted them
  const bool defer = policy && !first;
  const EaFrameInput in{d_bgr, layout, d_depth, nullptr, nullptr, false};
  int rc = ea_launch_preprocess(t->fs, t->n_streams, d_new_slots, roles, in, ps, defer ? EA_COMPACT_DEFER : EA_COMPACT_INLINE, nullptr);
  if (rc) return rc;
  CU(cudaEventRecord(t->ev_prep[fb], ps));
  if (consumed && !defer) CU(cudaEventRecord(consumed, ps));    // the input buffers may be overwritten from here on
  CU(cudaStreamWaitEvent(s, t->ev_prep[fb], 0));
  const size_t pb = size_t(t->n_streams) * 7 * 8;
  if (!first) {
    // streams that needed the most work last frame go first: hides the launch tail behind the rest of the batch
    rc = ea_solve_batch_device_ordered(c, t->n_streams, t->fs, d_key_slots, t->fs, d_new_slots, t->d_poses, nullptr,
                                       t->have_order ? t->d_order : nullptr, &t->sp, t->d_summaries,
                                       // many pairs per SM and the next frame's preprocessing waiting for the SMs the solve gives
                                       // up in its tail: helpers would only keep those SMs away from it (measured: -7 % throughput)
                                       !(overlap && t->n_streams >= 2 * c->sm_count));
    if (rc) return rc;
    if (t->n_streams > 1 && t->n_streams <= 4096) {
      cudaError_t oe = ea_launch_order_by_work(t->d_summaries, t->n_streams, t->n_levels, t->d_order, s);
      c->launches++;
      if (oe != cudaSuccess) return ea_fail(EA_ERR_CUDA, "order kernel: %s", cudaGetErrorString(oe));
      t->have_order = true;
    }
    CU(cudaMemcpyAsync(t->d_result, t->d_poses, pb, cudaMemcpyDeviceToDevice, s));
    if (policy) {   // decides K_{t+1} and N_{t+2}: before ev_solved, which prep(t+2) waits for
      const int f = t->frame;
      EaKeyPolicyArgs A{t->policy, t->n_streams, f, t->n_levels, t->sp.finest_level, t->d_summaries, t->d_result, t->d_poses,
                        t->d_key_tab[f & 1], t->d_key_tab[(f + 1) & 1], t->d_new_tab[f % 3], t->d_new_tab[(f + 1) % 3],
                        t->d_new_tab[(f + 2) % 3], t->d_key_frame, t->d_world, t->d_world_key, t->d_info};
      ea_k_keyframe_policy<<<(t->n_streams + 127) / 128, 128, 0, s>>>(A);
      c->launches++;
      cudaError_t pe = cudaGetLastError();
      if (pe != cudaSuccess) return ea_fail(EA_ERR_CUDA, "key-frame policy kernel: %s", cudaGetErrorString(pe));
    }
    CU(cudaEventRecord(t->ev_solved[fb], s));
    if (defer) {    // the point lists of the promoted frames (the level-0 depth is still the caller's input)
      rc = ea_launch_preprocess(t->fs, t->n_streams, d_new_slots, EA_ROLE_REF, in, s, EA_COMPACT_ONLY, t->d_info);
      if (rc) return rc;
      if (consumed) CU(cudaEventRecord(consumed, s));
    }
    t->prev_key = t->key_set; t->prev_now = cur;
  }
  if (becomes_key) {
    t->key_set = cur;
    CU(cudaMemcpyAsync(t->d_poses, t->d_identity, pb, cudaMemcpyDeviceToDevice, s));  // pose is relative to the new key frame
  }
  t->frame++;
  return EA_OK;
}

extern "C" {

int ea_tracker_step_device(ea_tracker* t, const uint8_t* d_bgr, const void* d_depth) {
  if (!t || !d_bgr) return ea_fail(EA_ERR_INVALID_ARG, "null argument");
  ea_image_layout L;   // BGR8 with a pitch is only read through the host path's copy
  const int rc = ea_resolve_layout(&t->layout, t->fs->p.width, t->fs->p.height, true, &L);
  if (rc) return rc;
  return tracker_step(t, d_bgr, L, d_depth, nullptr, nullptr);
}

int ea_tracker_set_image_layout(ea_tracker* t, const ea_image_layout* layout) {
  if (!t) return ea_fail(EA_ERR_INVALID_ARG, "null tracker");
  ea_image_layout L;
  const int w = t->fs->p.width, h = t->fs->p.height;
  int rc = ea_resolve_layout(layout, w, h, false, &L);
  if (rc) return rc;
  if (t->frame != 0) return ea_fail(EA_ERR_STATE, "the image layout can only change before the first step (after create or reset)");
  // the host-path staging buffers are sized for the bytes per frame of the layout; the next step_host allocates them anew
  if (ea_layout_row_bytes(L, w) != ea_layout_row_bytes(t->layout, w)) {
    CU(cudaSetDevice(t->ctx->device));
    CU(cudaStreamSynchronize(t->copy_stream));
    for (int b = 0; b < 2; ++b) { CU(cudaFree(t->stage_bgr[b])); t->stage_bgr[b] = nullptr; }
  }
  t->layout = L;
  return EA_OK;
}

int ea_tracker_set_image_format(ea_tracker* t, int image_format) {
  if (!t) return ea_fail(EA_ERR_INVALID_ARG, "null tracker");
  if (image_format != EA_IMAGE_BGR8 && image_format != EA_IMAGE_GRAY8) return ea_fail(EA_ERR_INVALID_ARG, "unknown image format %d", image_format);
  const ea_image_layout dense{image_format, 0, 0, 0};
  return ea_tracker_set_image_layout(t, &dense);
}

int ea_tracker_set_inputs_ready(ea_tracker* t, int ready) {
  if (!t) return ea_fail(EA_ERR_INVALID_ARG, "null tracker");
  t->inputs_ready = ready ? 1 : 0;
  return EA_OK;
}

int ea_tracker_probe_gather(ea_tracker* t, int level, int repeats, float* ms, double* point_gathers) {
  if (!t) return ea_fail(EA_ERR_INVALID_ARG, "null tracker");
  if (t->prev_now < 0) return ea_fail(EA_ERR_STATE, "the tracker has not aligned a frame yet");
  CU(cudaStreamSynchronize(t->prep_stream));
  // the pairs of the most recent alignment: key frames of that solve vs its frames, at the poses it produced
  const int f = t->frame - 1;   // the most recently solved frame
  const int32_t* d_key = t->policy_on ? t->d_key_tab[f & 1] : t->d_slots[t->prev_key];
  const int32_t* d_now = t->policy_on ? t->d_new_tab[f % 3] : t->d_slots[t->prev_now];
  return ea_probe_gather_device(t->ctx, t->n_streams, t->fs, d_key, t->fs, d_now, t->d_result, level, repeats, ms, point_gathers);
}

int ea_tracker_get_poses(ea_tracker* t, double* poses7, ea_summary* summaries) {
  if (!t) return ea_fail(EA_ERR_INVALID_ARG, "null tracker");
  cudaStream_t s = t->ctx->stream;
  std::vector<ea_summary> tmp;
  if (!summaries) { tmp.resize(size_t(t->n_streams) * t->n_levels); summaries = tmp.data(); }
  if (poses7) CU(cudaMemcpyAsync(poses7, t->d_result, size_t(t->n_streams) * 7 * 8, cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(summaries, t->d_summaries, size_t(t->n_streams) * t->n_levels * sizeof(ea_summary), cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  return tracker_check_truncated(summaries, t->n_streams, t->n_levels);
}

int ea_tracker_step_host(ea_tracker* t, const uint8_t* bgr, const void* depth, double* poses7, ea_summary* summaries) {
  if (!t || !bgr) return ea_fail(EA_ERR_INVALID_ARG, "null argument");
  ea_context* c = t->ctx;
  ea_frameset* fs = t->fs;
  CU(cudaSetDevice(c->device));
  const size_t px = size_t(fs->p.width) * fs->p.height;
  const int n = t->n_streams;
  const int frame = t->frame, b = frame & 1;
  // policy mode: any frame may become a key frame, so depth goes up with every frame
  const bool needs_depth = t->policy_on || (frame % t->interval) == 0;
  if (t->policy_on && !depth) return ea_fail(EA_ERR_INVALID_ARG, "key-frame policy mode: any frame may become a key frame, every step needs depth");
  if (needs_depth && !depth) return ea_fail(EA_ERR_INVALID_ARG, "frame %d becomes a key frame and needs depth", frame);
  const size_t frame_bytes = ea_layout_row_bytes(t->layout, fs->p.width) * fs->p.height * n;
  if (!t->stage_bgr[b]) CU(cudaMalloc((void**)&t->stage_bgr[b], frame_bytes));
  if (needs_depth && !t->stage_depth[b]) CU(cudaMalloc((void**)&t->stage_depth[b], px * fs->depth_elem * n));
  // upload on the copy stream once the kernels that read this staging buffer two frames ago are done
  if (frame >= 2) CU(cudaStreamWaitEvent(t->copy_stream, t->ev_consumed[b], 0));
  CU(ea_upload_frames(t->stage_bgr[b], bgr, t->layout, fs->p.width, fs->p.height, n, t->copy_stream));
  if (needs_depth) CU(cudaMemcpyAsync(t->stage_depth[b], depth, px * fs->depth_elem * n, cudaMemcpyHostToDevice, t->copy_stream));
  CU(cudaEventRecord(t->ev_copied[b], t->copy_stream));
  int rc = tracker_step(t, t->stage_bgr[b], ea_staged_layout(t->layout, fs->p.width, fs->p.height), needs_depth ? t->stage_depth[b] : nullptr, t->ev_copied[b], t->ev_consumed[b]);
  if (rc) return rc;
  // results into the pinned ring; the caller reads them now (poses7 given) or later with ea_tracker_wait
  CU(cudaMemcpyAsync(t->h_poses[b], t->d_result, size_t(n) * 7 * 8, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaMemcpyAsync(t->h_summaries[b], t->d_summaries, size_t(n) * t->n_levels * sizeof(ea_summary), cudaMemcpyDeviceToHost, c->stream));
  if (t->policy_on) {
    CU(cudaMemcpyAsync(t->h_world[b], t->d_world, size_t(n) * 7 * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(t->h_info[b], t->d_info, size_t(n) * sizeof(ea_track_info), cudaMemcpyDeviceToHost, c->stream));
  }
  CU(cudaEventRecord(t->ev_result[b], c->stream));
  t->result_frame[b] = frame;
  if (poses7 || summaries) return ea_tracker_wait(t, frame, poses7, summaries);
  return EA_OK;
}

int ea_tracker_wait(ea_tracker* t, int frame, double* poses7, ea_summary* summaries) {
  if (!t) return ea_fail(EA_ERR_INVALID_ARG, "null tracker");
  const int b = frame & 1;
  if (frame < 0 || t->result_frame[b] != frame) return ea_fail(EA_ERR_STATE, "results of frame %d are not (or no longer) in the 2-deep ring", frame);
  CU(cudaEventSynchronize(t->ev_result[b]));
  if (poses7) std::memcpy(poses7, t->h_poses[b], size_t(t->n_streams) * 7 * 8);
  if (summaries) std::memcpy(summaries, t->h_summaries[b], size_t(t->n_streams) * t->n_levels * sizeof(ea_summary));
  return tracker_check_truncated(t->h_summaries[b], t->n_streams, t->n_levels);
}

int ea_tracker_get_trajectory(ea_tracker* t, double* world7, ea_track_info* info) {
  if (!t) return ea_fail(EA_ERR_INVALID_ARG, "null tracker");
  if (!t->policy_on) return ea_fail(EA_ERR_STATE, "no key-frame policy is set: the tracker keeps no trajectory");
  cudaStream_t s = t->ctx->stream;
  CU(cudaSetDevice(t->ctx->device));
  if (world7) CU(cudaMemcpyAsync(world7, t->d_world, size_t(t->n_streams) * 7 * 8, cudaMemcpyDeviceToHost, s));
  if (info) CU(cudaMemcpyAsync(info, t->d_info, size_t(t->n_streams) * sizeof(ea_track_info), cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  return EA_OK;
}

int ea_tracker_wait_trajectory(ea_tracker* t, int frame, double* world7, ea_track_info* info) {
  if (!t) return ea_fail(EA_ERR_INVALID_ARG, "null tracker");
  if (!t->policy_on) return ea_fail(EA_ERR_STATE, "no key-frame policy is set: the tracker keeps no trajectory");
  const int b = frame & 1;
  if (frame < 0 || t->result_frame[b] != frame) return ea_fail(EA_ERR_STATE, "results of frame %d are not (or no longer) in the 2-deep ring", frame);
  CU(cudaEventSynchronize(t->ev_result[b]));
  if (world7) std::memcpy(world7, t->h_world[b], size_t(t->n_streams) * 7 * 8);
  if (info) std::memcpy(info, t->h_info[b], size_t(t->n_streams) * sizeof(ea_track_info));
  return EA_OK;
}

int ea_tracker_frame_index(ea_tracker* t, int* n) {
  if (!t || !n) return ea_fail(EA_ERR_INVALID_ARG, "null argument");
  *n = t->frame;
  return EA_OK;
}

}  // extern "C"
