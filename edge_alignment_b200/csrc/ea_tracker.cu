// Multi-stream frame-to-keyframe tracker: the caller of the pose-solve path, re-stated from the reference's
// consumer loop (src/ea.cpp:87-131) and SolveEA's setRefFrame / setNowFrame / setAsCERESProblem sequence
// (src/ea.cpp:184-199), batched over n_streams independent cameras.  Every frame is preprocessed once
// (its DT when it arrives, its edge points only if it becomes a key frame); poses are warm-started from the
// previous frame and never leave the device between steps.
#include <cstdlib>
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
  int channels = 3;                // image bytes per pixel: 3 (EA_IMAGE_BGR8) or 1 (EA_IMAGE_GRAY8)
  double* d_poses = nullptr;       // warm-start table [n_streams][7]
  double* d_result = nullptr;      // poses of the latest step [n_streams][7]
  double* d_identity = nullptr;    // [n_streams][7]
  ea_summary* d_summaries = nullptr;
  int32_t* d_order = nullptr;      // longest-first processing order derived from the previous step's summaries
  bool have_order = false;
  // host-input pipeline: frame t+1 is uploaded on a copy stream while frame t is being aligned
  cudaStream_t copy_stream = nullptr;
  uint8_t* stage_bgr[2] = {nullptr, nullptr};   // [n_streams][h][w][channels]
  void* stage_depth[2] = {nullptr, nullptr};
  cudaEvent_t ev_copied[2] = {nullptr, nullptr}, ev_consumed[2] = {nullptr, nullptr}, ev_result[2] = {nullptr, nullptr};
  double* h_poses[2] = {nullptr, nullptr};          // pinned result ring
  ea_summary* h_summaries[2] = {nullptr, nullptr};
  int result_frame[2] = {-1, -1};
};

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
  }
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
  return EA_OK;
}

}  // extern "C"

// input_ready: event after which the frame buffers are complete (host path: the upload); null => the buffers are ordered by
// the context stream (default) or already complete (inputs_ready).
static int tracker_step(ea_tracker* t, const uint8_t* d_bgr, const void* d_depth, cudaEvent_t input_ready, cudaEvent_t consumed) {
  ea_context* c = t->ctx;
  CU(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  const bool first = (t->frame == 0);
  const bool becomes_key = (t->frame % t->interval) == 0;
  if (becomes_key && !d_depth) return ea_fail(EA_ERR_INVALID_ARG, "frame %d becomes a key frame and needs depth", t->frame);
  // the new frame lands in the slot set that the solve still in flight (frame - 1) does not read
  int cur = 0;
  if (!first) { while (cur == t->prev_key || cur == t->prev_now || cur == t->key_set) ++cur; }
  const int roles = (first ? 0 : EA_ROLE_NOW) | (becomes_key ? EA_ROLE_REF : 0);
  const int fb = t->frame & 1;
  const bool overlap = input_ready != nullptr || t->inputs_ready != 0;   // frame t+1's preprocessing may run beside frame t's solve
  static const int force_helpers = getenv("EA_TAIL_HELPERS") ? atoi(getenv("EA_TAIL_HELPERS")) : -1;   // experiment knob
  cudaStream_t ps = t->prep_stream;
  if (input_ready) {
    CU(cudaStreamWaitEvent(ps, input_ready, 0));
  } else if (!t->inputs_ready) {   // inputs produced by work enqueued on the context stream: keep that order (no overlap)
    CU(cudaEventRecord(t->ev_prep[fb], s));
    CU(cudaStreamWaitEvent(ps, t->ev_prep[fb], 0));
  }
  if (t->frame >= 3) CU(cudaStreamWaitEvent(ps, t->ev_solved[fb], 0));   // last reader of this slot set: the solve of frame - 2
  int rc = ea_preprocess_impl(t->fs, t->n_streams, t->d_slots[cur], d_bgr, d_depth, roles, nullptr, nullptr, ps, t->channels);
  if (rc) return rc;
  CU(cudaEventRecord(t->ev_prep[fb], ps));
  if (consumed) CU(cudaEventRecord(consumed, ps));              // the input buffers may be overwritten from here on
  CU(cudaStreamWaitEvent(s, t->ev_prep[fb], 0));
  const size_t pb = size_t(t->n_streams) * 7 * 8;
  if (!first) {
    // streams that needed the most work last frame go first: hides the launch tail behind the rest of the batch
    rc = ea_solve_batch_device_ordered(c, t->n_streams, t->fs, t->d_slots[t->key_set], t->fs, t->d_slots[cur], t->d_poses, nullptr,
                                       t->have_order ? t->d_order : nullptr, &t->sp, t->d_summaries,
                                       // many pairs per SM and the next frame's preprocessing waiting for the SMs the solve gives
                                       // up in its tail: helpers would only keep those SMs away from it (measured: -7 % throughput)
                                       force_helpers > 0 || (force_helpers < 0 && !(overlap && t->n_streams >= 2 * c->sm_count)));
    if (rc) return rc;
    if (t->n_streams > 1 && t->n_streams <= 4096) {
      cudaError_t oe = ea_launch_order_by_work(t->d_summaries, t->n_streams, t->n_levels, t->d_order, s);
      c->launches++;
      if (oe != cudaSuccess) return ea_fail(EA_ERR_CUDA, "order kernel: %s", cudaGetErrorString(oe));
      t->have_order = true;
    }
    CU(cudaMemcpyAsync(t->d_result, t->d_poses, pb, cudaMemcpyDeviceToDevice, s));
    CU(cudaEventRecord(t->ev_solved[fb], s));
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
  return tracker_step(t, d_bgr, d_depth, nullptr, nullptr);
}

int ea_tracker_set_image_format(ea_tracker* t, int image_format) {
  if (!t) return ea_fail(EA_ERR_INVALID_ARG, "null tracker");
  if (image_format != EA_IMAGE_BGR8 && image_format != EA_IMAGE_GRAY8) return ea_fail(EA_ERR_INVALID_ARG, "unknown image format %d", image_format);
  if (t->frame != 0) return ea_fail(EA_ERR_STATE, "the image format can only change before the first step (after create or reset)");
  const int channels = image_format == EA_IMAGE_GRAY8 ? 1 : 3;
  if (channels != t->channels) {   // the host-path staging buffers are sized for the format; the next step_host allocates them anew
    CU(cudaSetDevice(t->ctx->device));
    CU(cudaStreamSynchronize(t->copy_stream));
    for (int b = 0; b < 2; ++b) { CU(cudaFree(t->stage_bgr[b])); t->stage_bgr[b] = nullptr; }
    t->channels = channels;
  }
  return EA_OK;
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
  return ea_probe_gather_device(t->ctx, t->n_streams, t->fs, t->d_slots[t->prev_key], t->fs, t->d_slots[t->prev_now], t->d_result, level,
                                repeats, ms, point_gathers);
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
  const bool becomes_key = (frame % t->interval) == 0;
  if (becomes_key && !depth) return ea_fail(EA_ERR_INVALID_ARG, "frame %d becomes a key frame and needs depth", frame);
  const size_t frame_bytes = px * t->channels * n;
  if (!t->stage_bgr[b]) CU(cudaMalloc((void**)&t->stage_bgr[b], frame_bytes));
  if (becomes_key && !t->stage_depth[b]) CU(cudaMalloc((void**)&t->stage_depth[b], px * fs->depth_elem * n));
  // upload on the copy stream once the kernels that read this staging buffer two frames ago are done
  if (frame >= 2) CU(cudaStreamWaitEvent(t->copy_stream, t->ev_consumed[b], 0));
  CU(cudaMemcpyAsync(t->stage_bgr[b], bgr, frame_bytes, cudaMemcpyHostToDevice, t->copy_stream));
  if (becomes_key) CU(cudaMemcpyAsync(t->stage_depth[b], depth, px * fs->depth_elem * n, cudaMemcpyHostToDevice, t->copy_stream));
  CU(cudaEventRecord(t->ev_copied[b], t->copy_stream));
  int rc = tracker_step(t, t->stage_bgr[b], becomes_key ? t->stage_depth[b] : nullptr, t->ev_copied[b], t->ev_consumed[b]);
  if (rc) return rc;
  // results into the pinned ring; the caller reads them now (poses7 given) or later with ea_tracker_wait
  CU(cudaMemcpyAsync(t->h_poses[b], t->d_result, size_t(n) * 7 * 8, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaMemcpyAsync(t->h_summaries[b], t->d_summaries, size_t(n) * t->n_levels * sizeof(ea_summary), cudaMemcpyDeviceToHost, c->stream));
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

int ea_tracker_frame_index(ea_tracker* t, int* n) {
  if (!t || !n) return ea_fail(EA_ERR_INVALID_ARG, "null argument");
  *n = t->frame;
  return EA_OK;
}

}  // extern "C"
