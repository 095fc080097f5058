// Internal host-side declarations shared by the .cu translation units (not part of the ABI).
#pragma once
#include <cuda_runtime.h>

#include <string>
#include <vector>

#include "ea_device.cuh"

#include "ea_solve.cuh"

#define EA_TRACE_DOUBLES 6    // {level, iteration, cost of the accepted iterate, cost at the candidate, radius, decision}

struct EaSolveArgs {
  const EaLevelDesc* ref_desc;  // [ref slots][EA_MAX_LEVELS]
  const EaLevelDesc* now_desc;  // [now slots][EA_MAX_LEVELS]
  const int32_t* ref_slots;     // [n_pairs] device
  const int32_t* now_slots;     // [n_pairs] device
  const int32_t* pose_index;    // [n_pairs] device or null (identity)
  const int32_t* order;         // [n_pairs] device or null: processing order of the work queue (longest first)
  double* poses;                // [*][7] device, in/out
  int* work_counter;            // device: next pair index of the dynamic work queue (zeroed per launch)
  struct EaHelpBoard* boards;   // [grid] tail-helper boards of the persistent kernel (zeroed per launch), or null: no helpers
  unsigned long long* debug;    // null, or [grid][6] cycle counters of each CTA's thread 0 (EA_SOLVE_DEBUG=1, development aid)
  // Coarse / fine split (ea_launch_solve_batch): the coarse phase publishes handoff[pair] = handoff_epoch with release
  // semantics once the pair's pose after level finest + 1 is written; the fine phase acquires it before reading the pose.
  unsigned* handoff;            // [n_pairs] device, or null: no split
  unsigned handoff_epoch;       // tag of this launch (never 0, so that a zeroed array holds no hand-over)
  int handoff_role;             // 0: none; 1: coarse phase (publishes); 2: fine phase (waits)
  ea_summary* summaries;        // [n_pairs][n_levels] device or null
  double* trace;                // [trace_cap][EA_TRACE_DOUBLES] device or null: one record per evaluation (single-pair solves only)
  int* trace_count;             // device counter of records written
  int trace_cap;
  int n_pairs, n_levels, coarsest, finest;
  double inv_depth_scale;
  EaLevelGeom ref_geom[EA_MAX_LEVELS];
  EaLevelGeom now_geom[EA_MAX_LEVELS];
  int ref_cap[EA_MAX_LEVELS];   // point-list capacity per level (guards a truncated list)
  ea_solve_params sp;
  EaEvalConsts loss;                 // sp's loss in fp32 (ea_eval_consts), for the evaluation loop
};

// A split launch runs as a coarse and a fine phase: A.work_counter then holds two counters, and A.debug two blocks of
// EA_DEBUG_ROWS rows (fine phase first).
#define EA_DEBUG_ROWS 1024
struct EaSolveShape {           // what ea_launch_solve_batch enqueued
  int launches = 0;
  int grid[2] = {0, 0};         // CTAs of {the whole launch or the fine phase, the coarse phase (0: no split)}
};
// Chooses the batched solve's launch shape for A.n_pairs pairs (cluster size, coarse / fine split; grows and tags the context's
// hand-over words for a split) and enqueues it on c->stream.
cudaError_t ea_launch_solve_batch(ea_context* c, EaSolveArgs A, EaSolveShape& shape);
size_t ea_help_boards_bytes(int sm_count);
cudaError_t ea_launch_gather_probe(const EaSolveArgs& A, int level, int slices, int repeats, float* d_sink, cudaStream_t stream);
int ea_probe_gather_device(ea_context* c, int n, ea_frameset* ref, const int32_t* d_ref_slots, ea_frameset* now, const int32_t* d_now_slots,
                           const double* d_poses7, int level, int repeats, float* ms, double* point_gathers);
cudaError_t ea_launch_eval_points(const EaLevelDesc& rd, const EaLevelDesc& nd, const EaLevelGeom& rg,
                                  const EaLevelGeom& ng, double inv_depth_scale, const ea_solve_params& sp,
                                  const double* d_pose7, int n_res, double* d_raw, double* d_res, double* d_jac,
                                  int* d_failed, cudaStream_t stream);
cudaError_t ea_launch_eval_sums(const EaLevelDesc& rd, const EaLevelDesc& nd, const EaLevelGeom& rg,
                                const EaLevelGeom& ng, double inv_depth_scale, const ea_solve_params& sp,
                                const double* d_pose7, const int* d_done, int j_begin, int j_end, int n_blocks, double* d_sums,
                                cudaStream_t stream);

// ---- preprocessing (ea_preprocess.cu) ---------------------------------------------------------------
struct EaPrepLevel {            // device pointers of one pyramid level, slot-major pools
  uint8_t* bgr;                 // [slots][h][w][3], or [slots][h][w] for gray input (level 0: null, the caller's input is read directly)
  void* depth;                  // [slots][h][w] u16 or f32 (level 0: null)
  uint32_t* edge_bits;          // [slots][h][words]  raw Laplacian>threshold mask, 1 bit / pixel
  uint32_t* ref_bits;           // [slots][h][words]  edge & depth>0
  uint32_t* med_bits;           // [slots][h][words]  3x3 median of edge_bits
  float* dt;                    // [slots][h + 2 PAD][dt_pitch] replicate-padded (EA_DT_PAD, ea_device.cuh)
  int dt_pitch; size_t dt_slot; // floats per padded row / per slot
  float4* pts;                  // [slots][cap]
  int w, h, words, cap;
};
struct EaCannyCfg { double low, high; int l2, on_color; };
struct EaScratch {              // Canny / exact-EDT work buffers, [n_slots][stride] each (stride = level-0 pixels); after NMS, dxy holds the hysteresis' union-find keys
  uint8_t* gray; int* mag; short2* dxy; uint8_t* map; size_t stride;
};
struct EaPrepArgs {
  EaPrepLevel lv[EA_MAX_LEVELS];
  int n_levels;
  const int32_t* slots;         // [n] device: destination slot of frame i
  const uint8_t* in_img;        // frame i's level-0 image at in_img + i * in_stride, its row y at + y * in_pitch (bytes)
  int in_format;                // EA_IMAGE_BGR8 (dense [h0][w0][3]); EA_IMAGE_GRAY8 (luma plane: gray, NV12); EA_IMAGE_YUYV / _UYVY
                                // (packed 4:2:2, luma read in place).  One-channel input is preprocessed exactly as BGR (g, g, g)
  size_t in_pitch, in_stride;
  const void* in_depth;        // [n][h0][w0] u16 raw units or f32 metres (depth_type), or null
  const uint8_t* in_mask;       // [n][h0][w0] or null: reference points only where mask > 0 (get_aX_mask, utils.cpp:283-369)
  const uint8_t* in_now_mask;   // [n][h0][w0] or null: now-frame edges only where mask > 1 (get_distance_transform2_masked, utils.cpp:124-128)
  int* n_pts;                   // [slots][EA_MAX_LEVELS]
  unsigned* dt_minmax;          // [slots][EA_MAX_LEVELS][2]  (min,max of the fixed-point DT)
  float2* dt_affine;            // [slots][EA_MAX_LEVELS]     {scale, shift} of the min-max normalisation
  int* overflow;                // [slots][EA_MAX_LEVELS]: that point list was truncated at cap (rewritten by every compaction)
  int n, roles, grad_threshold, use_median, dt_normalize;
  int edge_detector, dt_kind;
  int depth_type;               // 0 = u16 raw units, 1 = f32 metres
  int zero_to_one;              // src/SolveEA.cpp:69: an edge pixel without depth is kept at Z = 1
  float depth_one;              // the stored value meaning Z = 1 (depth_scale for u16, 1.0 for f32)
  EaCannyCfg canny;
  EaScratch scratch;
  int compact;                  // the reference-point lists (EA_ROLE_REF): EA_COMPACT_INLINE, _DEFER or _ONLY
  const ea_track_info* compact_gate;   // EA_COMPACT_ONLY: frame i's lists are built only where compact_gate[i].key_reasons != 0
};
// EA_COMPACT_DEFER runs the edge kernels of the reference role (ref_bits and the depth pyramid in the slots) without building the
// point lists; a later EA_COMPACT_ONLY call with the same slots and level-0 depth builds them for the frames its gate selects.
enum { EA_COMPACT_INLINE = 0, EA_COMPACT_DEFER = 1, EA_COMPACT_ONLY = 2 };
// Second lane for big batches: the distance transforms (DRAM / latency-bound, few warps) of one part of the frames run on an
// auxiliary stream beside the edge kernels (issue-bound) of the next part.  Streams and events belong to the context; the
// preprocessing launcher creates them the first time it splits a batch, ea_release_prep_lanes destroys them.
#define EA_PREP_MAX_PARTS 2
struct EaPrepPipe {
  cudaStream_t aux[EA_PREP_MAX_PARTS] = {};
  cudaEvent_t ev_front[EA_PREP_MAX_PARTS] = {}, ev_dt[EA_PREP_MAX_PARTS] = {};
  bool ready = false;
};
void ea_release_prep_lanes(ea_context* c);
// Where the bytes of a level's image lie: channel c of pixel (x, y) of frame (or slot) f at
// base[f * stride + y * pitch + x * step + offset + c].  Level 0 is the caller's image where it lies (GRAY8 / NV12: step 1; YUYV:
// step 2, offset 0; UYVY: step 2, offset 1; BGR: dense, step 3); the pyramid pools above it are dense.
struct EaImage {
  const uint8_t* base;
  size_t stride, pitch;
  int step, offset;
};
inline EaImage ea_level_image(const EaPrepArgs& A, int l) {
  const int cn = A.in_format == EA_IMAGE_BGR8 ? 3 : 1;
  if (l > 0) { const EaPrepLevel& L = A.lv[l]; return {L.bgr, size_t(L.w) * L.h * cn, size_t(L.w) * cn, cn, 0}; }
  const bool packed = A.in_format == EA_IMAGE_YUYV || A.in_format == EA_IMAGE_UYVY;
  return {A.in_img, A.in_stride, A.in_pitch, packed ? 2 : cn, A.in_format == EA_IMAGE_UYVY ? 1 : 0};
}
// ---- image layouts (ea_image_layout, ea_cabi.cu) ----
// Checks `in` for frames of w x h and fills `out` with its row pitch and frame stride made explicit.  on_device: the layout
// describes device memory, where BGR8 must be dense.
int ea_resolve_layout(const ea_image_layout* in, int w, int h, bool on_device, ea_image_layout* out);
size_t ea_layout_row_bytes(const ea_image_layout& L, int w);   // bytes of a row the kernels read: 3w, w, w, 2w, 2w
// The layout of frames that ea_upload_frames has packed dense: NV12 becomes GRAY8 (its luma plane).
ea_image_layout ea_staged_layout(const ea_image_layout& L, int w, int h);
// Copies the rows the kernels read of n host frames in layout L to dst, packed dense, in one copy on `stream`.
cudaError_t ea_upload_frames(uint8_t* dst, const uint8_t* src, const ea_image_layout& L, int w, int h, int n, cudaStream_t stream);

// The frames of one preprocessing call, at the frame set's level-0 geometry.
struct EaFrameInput {
  const uint8_t* image;         // frame i at image + i * layout.frame_stride
  ea_image_layout layout;       // resolved (ea_resolve_layout): row_pitch and frame_stride in bytes
  const void* depth;           // [n][h][w] of the frame set's depth_type, or null; read by the reference role only
  const uint8_t* ref_mask;      // [n][h][w] or null: reference points only where mask > 0
  const uint8_t* now_mask;      // [n][h][w] or null: now-frame edges only where mask > 1
  bool on_host;                 // host buffers (staged through the frame set) rather than device buffers
};
// Enqueues the preprocessing of n frames into the slots d_slots[0..n) (device) on `stream` and counts its launches in the
// context.  The inputs are device buffers (in.on_host is not read); the arguments are the caller's to validate.
int ea_launch_preprocess(ea_frameset* fs, int n, const int32_t* d_slots, int roles, const EaFrameInput& in, cudaStream_t stream,
                         int compact, const ea_track_info* compact_gate);
__host__ __device__ inline float* ea_dt_origin(const EaPrepLevel& L, int slot) {   // pixel (0,0) of a slot's padded DT
  return L.dt + size_t(slot) * L.dt_slot + size_t(EA_DT_PAD) * L.dt_pitch + EA_DT_PAD;
}
cudaError_t ea_launch_dt_normalized_copy(const float* origin, int pitch, const float2* affine, int w, int h, float* out, cudaStream_t stream);
cudaError_t ea_launch_dt_import(const float* src, float* origin, int w, int h, int pitch, cudaStream_t stream);
cudaError_t ea_launch_dt_fill_pad(const EaPrepLevel& L, const int32_t* d_slots, int n, cudaStream_t stream);
cudaError_t ea_launch_canny_level(const EaPrepArgs& A, int l, const EaImage& img, const void* depth, size_t frame_stride_px,
                                  bool slot_indexed, const EaCannyCfg& cfg, const EaScratch& S, cudaStream_t stream, int* launches);
cudaError_t ea_launch_exact_edt_level(const EaPrepArgs& A, int l, const EaScratch& S, cudaStream_t stream, int* launches);
cudaError_t ea_launch_unpack_mask(const uint32_t* bits, int w, int h, int words, int median, uint8_t* out,
                                  cudaStream_t stream);

// ---- host-side objects behind the opaque ABI handles ------------------------------------------------
struct ea_context {
  int device = 0, sm_count = 0, cc_major = 0, cc_minor = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  int64_t launches = 0;
  // small scratch
  double* d_pose = nullptr;      // [7]
  int* d_failed = nullptr;
  int* d_work = nullptr;         // [2] work-queue counters of the batched solve (fine / whole, coarse phase)
  unsigned* d_handoff = nullptr; int handoff_cap = 0; unsigned handoff_epoch = 0;   // coarse -> fine hand-over words (EaSolveArgs)
  void* d_boards = nullptr;       // tail-helper boards of the persistent solve kernel
  // EA_SOLVE_DEBUG=1: [2][EA_DEBUG_ROWS][6] cycle counters, and their sums per phase {fine or whole launch, coarse phase}
  unsigned long long* d_debug = nullptr; double debug_sum[2][6] = {}; long debug_launches[2] = {0, 0};
  double* d_sums = nullptr;      // [max blocks][EA_SUMS]
  int32_t* d_idx = nullptr;      // scratch slot indices
  size_t idx_cap = 0;
  void* d_tmp = nullptr;
  size_t tmp_cap = 0;
  void* d_views = nullptr; size_t views_cap = 0;   // ea_solve_views / ea_solve_views_batch: view descriptors and the persistent kernel's scratch
  EaPrepPipe prep_pipe;           // auxiliary streams of the preprocessing pipeline (created on first use)
  // optional profiling: event pairs around preprocessing pipelines [0] and solve launches [1]
  bool profile = false;
  double* d_trace = nullptr; int* d_trace_count = nullptr; int trace_cap = 0;   // ea_solve_traced
  std::vector<cudaEvent_t> ev[2];
};
struct EaProfileScope {   // records a start/stop event pair on the launching stream when profiling is on
  ea_context* c; int kind; cudaStream_t s;
  EaProfileScope(ea_context* c_, int kind_, cudaStream_t s_ = nullptr) : c(c_), kind(kind_), s(s_ ? s_ : c_->stream) {
    if (c->profile) { cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, s); c->ev[kind].push_back(e); }
  }
  ~EaProfileScope() {
    if (c->profile) { cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, s); c->ev[kind].push_back(e); }
  }
};

struct ea_frameset {
  ea_context* ctx = nullptr;
  ea_frame_params p;
  int n_slots = 0;
  EaPrepLevel lv[EA_MAX_LEVELS];
  EaLevelGeom geom[EA_MAX_LEVELS];
  EaLevelDesc* d_desc = nullptr;          // [n_slots][EA_MAX_LEVELS]
  std::vector<EaLevelDesc> h_desc;
  int* d_npts = nullptr;                  // [n_slots][EA_MAX_LEVELS]
  unsigned* d_minmax = nullptr;
  float2* d_affine = nullptr;             // [n_slots][EA_MAX_LEVELS]
  int* d_overflow = nullptr;
  uint8_t* stage_bgr = nullptr;           // [n_slots][h][w][3]  (host-upload staging; other formats use the first 1 or 2 thirds)
  void* stage_depth = nullptr;
  size_t depth_elem = 2;                  // bytes per depth sample (2: u16, 4: f32)
  double inv_depth_unit = 1.0 / 5000.0;   // metres per stored depth unit
  EaScratch scratch{};                    // only allocated for Canny / exact EDT
  std::vector<void*> allocs;
};


int ea_fail(int code, const char* fmt, ...);
#define CU(call)                                                                                       \
  do {                                                                                                 \
    cudaError_t e_ = (call);                                                                           \
    if (e_ != cudaSuccess) return ea_fail(EA_ERR_CUDA, "%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
  } while (0)
// Scope guards for the entry points: CU() returns early on an error, these release what the call had acquired by then.
struct EaAsyncBuf {   // cudaMallocAsync / cudaFreeAsync on one stream
  void* p = nullptr; cudaStream_t s = nullptr;
  explicit EaAsyncBuf(cudaStream_t s_) : s(s_) {}
  cudaError_t alloc(size_t bytes) { return cudaMallocAsync(&p, bytes, s); }
  template <class T> T* as() const { return static_cast<T*>(p); }
  ~EaAsyncBuf() { if (p) cudaFreeAsync(p, s); }
  EaAsyncBuf(const EaAsyncBuf&) = delete; EaAsyncBuf& operator=(const EaAsyncBuf&) = delete;
};
struct EaDevBuf {     // cudaMalloc / cudaFree
  void* p = nullptr;
  cudaError_t alloc(size_t bytes) { return cudaMalloc(&p, bytes); }
  template <class T> T* as() const { return static_cast<T*>(p); }
  ~EaDevBuf() { if (p) cudaFree(p); }
  EaDevBuf() = default; EaDevBuf(const EaDevBuf&) = delete; EaDevBuf& operator=(const EaDevBuf&) = delete;
};
struct EaEventPair {
  cudaEvent_t a = nullptr, b = nullptr;
  cudaError_t create() { cudaError_t e = cudaEventCreate(&a); return e != cudaSuccess ? e : cudaEventCreate(&b); }
  ~EaEventPair() { if (a) cudaEventDestroy(a); if (b) cudaEventDestroy(b); }
  EaEventPair() = default; EaEventPair(const EaEventPair&) = delete; EaEventPair& operator=(const EaEventPair&) = delete;
};
int ea_ensure_tmp(ea_context* c, size_t bytes);
int ea_ensure_views(ea_context* c, size_t bytes);   // grows c->d_views (after the stream's work on it has finished)
// The C ABI's sums28 ({cost, J^T r [6], upper-tri J^T J [21]}) from n_blocks rows of EA_SUMS partial sums, added in row order.
void ea_fold_sums28(const double* partials, int n_blocks, double* sums28);
// A view's rig transform and distortion in the form the general per-point evaluation takes (identity / zero when unused).
inline void ea_view_xf(const ea_view& v, EaViewXf& X) {
  memset(&X, 0, sizeof X);
  X.use_rig = v.use_rig != 0; X.use_dist = v.use_distortion != 0;
  for (int i = 0; i < 12; ++i) { X.T21[i] = v.cam_T_first[i]; X.T12[i] = v.first_T_cam[i]; }
  if (!X.use_rig) { for (int i = 0; i < 12; ++i) X.T21[i] = X.T12[i] = (i % 5 == 0) ? 1.0 : 0.0; }
  for (int i = 0; i < 5; ++i) X.dist[i] = X.use_dist ? v.dist[i] : 0.0;
}
extern "C" int ea_check_solve_params(const ea_solve_params* sp);   // shared argument validation of every solve entry point
int ea_solve_batch_device_ordered(ea_context* c, int n, ea_frameset* ref, const int32_t* d_ref_slots, ea_frameset* now,
                                   const int32_t* d_now_slots, double* d_poses7, const int32_t* d_pose_index,
                                   const int32_t* d_order, const ea_solve_params* sp, ea_summary* d_summaries, bool tail_helpers = true);
cudaError_t ea_launch_order_by_work(const ea_summary* d_summaries, int n, int n_levels, int32_t* d_order, cudaStream_t stream);
