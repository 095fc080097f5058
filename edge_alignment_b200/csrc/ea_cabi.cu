// C ABI implementation (include/ea_cabi.h): contexts, device-resident framesets, evaluation, batched solve,
// multi-stream tracker.  Host C++ only orchestrates; all arithmetic of the path runs in the kernels of
// ea_preprocess.cu / ea_solve.cu.  No CPU fallback: every entry point fails loudly without a device.
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <algorithm>
#include <cstring>
#include <mutex>
#include <vector>
#include <new>

#include "ea_internal.h"

thread_local std::string g_ea_err;
int ea_fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_ea_err = buf;
  return code;
}

int ea_ensure_tmp(ea_context* c, size_t bytes) {
  if (c->tmp_cap >= bytes) return EA_OK;
  if (c->d_tmp) cudaFree(c->d_tmp);
  c->d_tmp = nullptr; c->tmp_cap = 0;
  CU(cudaMalloc(&c->d_tmp, bytes));
  c->tmp_cap = bytes;
  return EA_OK;
}

int ea_ensure_views(ea_context* c, size_t bytes) {
  if (c->views_cap >= bytes) return EA_OK;
  CU(cudaStreamSynchronize(c->stream));
  if (c->d_views) { cudaFree(c->d_views); c->d_views = nullptr; c->views_cap = 0; }
  CU(cudaMalloc(&c->d_views, bytes));
  c->views_cap = bytes;
  return EA_OK;
}

void ea_fold_sums28(const double* partials, int n_blocks, double* sums28) {
  double t[EA_SUMS] = {0};
  for (int b = 0; b < n_blocks; ++b) for (int k = 0; k < EA_SUMS; ++k) t[k] += partials[size_t(b) * EA_SUMS + k];
  sums28[0] = t[28];                                   // cost
  for (int k = 0; k < 6; ++k) sums28[1 + k] = t[21 + k];  // J^T r
  for (int k = 0; k < 21; ++k) sums28[7 + k] = t[k];      // upper-tri J^T J
}
extern "C" {

int ea_abi_version(void) { return EA_ABI_VERSION; }
const char* ea_last_error(void) { return g_ea_err.c_str(); }

int ea_create(int device, ea_context** out) {
  if (!out) return ea_fail(EA_ERR_INVALID_ARG, "ea_create: out is null");
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0)
    return ea_fail(EA_ERR_NO_DEVICE, "ea_create: no CUDA device (%s); this library has no CPU fallback", cudaGetErrorString(e));
  if (device < 0 || device >= n) return ea_fail(EA_ERR_INVALID_ARG, "ea_create: device %d out of range [0,%d)", device, n);
  CU(cudaSetDevice(device));
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) return ea_fail(EA_ERR_NO_DEVICE, "ea_create: device %d is sm_%d%d; this build is sm_100a only", device, prop.major, prop.minor);
  ea_context* c = new (std::nothrow) ea_context();
  if (!c) return ea_fail(EA_ERR_INVALID_ARG, "out of host memory");
  struct Guard { ea_context* c; ~Guard() { if (c) ea_destroy(c); } } guard{c};    // a failed create leaves nothing behind
  c->device = device; c->sm_count = prop.multiProcessorCount; c->cc_major = prop.major; c->cc_minor = prop.minor;
  CU(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  c->own_stream = true;
  CU(cudaMalloc(&c->d_pose, 7 * sizeof(double)));
  CU(cudaMalloc(&c->d_failed, sizeof(int)));
  CU(cudaMalloc(&c->d_work, 2 * sizeof(int)));
  CU(cudaMalloc(&c->d_sums, size_t(1024) * EA_SUMS * sizeof(double)));
  CU(cudaMalloc(&c->d_boards, ea_help_boards_bytes(c->sm_count)));
  if (getenv("EA_SOLVE_DEBUG")) {
    CU(cudaMalloc(&c->d_debug, size_t(2) * EA_DEBUG_ROWS * 6 * sizeof(unsigned long long)));
    CU(cudaMemset(c->d_debug, 0, size_t(2) * EA_DEBUG_ROWS * 6 * sizeof(unsigned long long)));
  }
  guard.c = nullptr;
  *out = c;
  return EA_OK;
}
int ea_destroy(ea_context* c) {
  if (!c) return EA_OK;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  for (int ph = 0; ph < 2; ++ph) {
    if (!c->d_debug || c->debug_launches[ph] == 0) continue;
    const double n = double(c->debug_launches[ph]);
    const double* d = c->debug_sum[ph];
    fprintf(stderr, "[EA_SOLVE_DEBUG]%s %ld launches; per launch, mean over CTAs, kcycles of thread 0: eval %.1f  wait+totals %.1f  LM %.1f  wait2 %.1f  lifetime %.1f; evaluations %.1f\n",
            ph ? " coarse phase:" : "", c->debug_launches[ph], d[0] / n / 1e3, d[1] / n / 1e3, d[2] / n / 1e3, d[3] / n / 1e3, d[5] / n / 1e3, d[4] / n);
  }
  cudaFree(c->d_handoff); cudaFree(c->d_debug); cudaFree(c->d_boards); cudaFree(c->d_views);
  ea_release_prep_lanes(c);
  cudaFree(c->d_pose); cudaFree(c->d_failed); cudaFree(c->d_work); cudaFree(c->d_sums); cudaFree(c->d_idx); cudaFree(c->d_tmp);
  if (c->own_stream) cudaStreamDestroy(c->stream);
  delete c;
  return EA_OK;
}
int ea_sync(ea_context* c) {
  if (!c) return ea_fail(EA_ERR_INVALID_ARG, "null context");
  CU(cudaStreamSynchronize(c->stream));
  return EA_OK;
}
int ea_set_stream(ea_context* c, void* s) {
  if (!c) return ea_fail(EA_ERR_INVALID_ARG, "null context");
  if (c->own_stream) { cudaStreamSynchronize(c->stream); cudaStreamDestroy(c->stream); c->own_stream = false; }
  c->stream = static_cast<cudaStream_t>(s);
  return EA_OK;
}
int ea_device_info(ea_context* c, int* sm, int* maj, int* min_) {
  if (!c) return ea_fail(EA_ERR_INVALID_ARG, "null context");
  if (sm) *sm = c->sm_count;
  if (maj) *maj = c->cc_major;
  if (min_) *min_ = c->cc_minor;
  return EA_OK;
}
int ea_host_alloc(void** p, size_t bytes) {
  if (!p) return ea_fail(EA_ERR_INVALID_ARG, "null pointer");
  CU(cudaHostAlloc(p, bytes, cudaHostAllocDefault));
  return EA_OK;
}
int ea_host_free(void* p) {
  if (p) CU(cudaFreeHost(p));
  return EA_OK;
}
int ea_launch_count(ea_context* c, int64_t* n) {
  if (!c || !n) return ea_fail(EA_ERR_INVALID_ARG, "null argument");
  *n = c->launches;
  return EA_OK;
}

int ea_profile_enable(ea_context* c, int on) {
  if (!c) return ea_fail(EA_ERR_INVALID_ARG, "null context");
  c->profile = on != 0;
  return EA_OK;
}
int ea_profile_read(ea_context* c, double* pre_ms, int* n_pre, double* solve_ms, int* n_solve) {
  if (!c) return ea_fail(EA_ERR_INVALID_ARG, "null context");
  CU(cudaSetDevice(c->device));
  CU(cudaDeviceSynchronize());        // trackers preprocess on their own stream
  double tot[2] = {0, 0}; int cnt[2] = {0, 0};
  for (int k = 0; k < 2; ++k) {
    for (size_t i = 0; i + 1 < c->ev[k].size(); i += 2) {
      float ms = 0.f;
      cudaEventElapsedTime(&ms, c->ev[k][i], c->ev[k][i + 1]);
      tot[k] += ms; cnt[k]++;
    }
    for (cudaEvent_t e : c->ev[k]) cudaEventDestroy(e);
    c->ev[k].clear();
  }
  if (pre_ms) *pre_ms = tot[0];
  if (n_pre) *n_pre = cnt[0];
  if (solve_ms) *solve_ms = tot[1];
  if (n_solve) *n_solve = cnt[1];
  return EA_OK;
}

void ea_frame_params_default(ea_frame_params* p) {
  if (!p) return;
  std::memset(p, 0, sizeof *p);
  p->width = 640; p->height = 480; p->n_levels = 1; p->grad_threshold = 35; p->use_median = 1;
  p->dt_normalize = EA_NORM_01; p->max_points = 0;
  p->fx = 525.0; p->fy = 525.0; p->cx = 319.5; p->cy = 239.5; p->depth_scale = 5000.0;
  p->edge_detector = EA_EDGE_LAPLACIAN; p->canny_l2 = 0; p->canny_low = 30.0; p->canny_high = 90.0; p->dt_kind = EA_DT_CHAMFER3;
}
void ea_solve_params_default(ea_solve_params* p) {
  if (!p) return;
  std::memset(p, 0, sizeof *p);
  p->point_stride = 30; p->loss_type = EA_LOSS_CAUCHY; p->max_num_iterations = 50; p->jacobi_scaling = 1;
  p->max_consecutive_invalid_steps = 5; p->cluster_size = 0; p->coarsest_level = -1; p->finest_level = 0;
  p->loss_scale = 1.0; p->function_tolerance = 1e-6; p->gradient_tolerance = 1e-10; p->parameter_tolerance = 1e-8;
  p->initial_trust_region_radius = 1e4; p->max_trust_region_radius = 1e16; p->min_trust_region_radius = 1e-32;
  p->min_relative_decrease = 1e-3; p->min_lm_diagonal = 1e-6; p->max_lm_diagonal = 1e32;
}

// ---- framesets ------------------------------------------------------------------------------------------
static int fs_alloc(ea_frameset* fs, void** p, size_t bytes) {
  CU(cudaMalloc(p, bytes));
  fs->allocs.push_back(*p);
  return EA_OK;
}

int ea_frameset_create(ea_context* ctx, const ea_frame_params* p, int n_slots, ea_frameset** out) {
  if (!ctx || !p || !out) return ea_fail(EA_ERR_INVALID_ARG, "ea_frameset_create: null argument");
  *out = nullptr;
  if (n_slots <= 0) return ea_fail(EA_ERR_INVALID_ARG, "n_slots must be positive");
  if (p->n_levels < 1 || p->n_levels > EA_MAX_LEVELS) return ea_fail(EA_ERR_INVALID_ARG, "n_levels must be in [1,%d]", EA_MAX_LEVELS);
  if (p->width < 8 || p->height < 8) return ea_fail(EA_ERR_INVALID_ARG, "frames must be at least 8x8");
  if ((p->width % (1 << (p->n_levels - 1))) || (p->height % (1 << (p->n_levels - 1))))
    return ea_fail(EA_ERR_INVALID_ARG, "width/height must be divisible by 2^(n_levels-1)");
  if (!(p->fx > 0) || !(p->fy > 0) || !(p->depth_scale > 0)) return ea_fail(EA_ERR_INVALID_ARG, "fx, fy, depth_scale must be positive");
  if (p->edge_detector < 0 || p->edge_detector > EA_EDGE_CANNY_COLOR || p->dt_kind < 0 || p->dt_kind > EA_DT_EXACT) return ea_fail(EA_ERR_INVALID_ARG, "unknown edge_detector / dt_kind");
  if (p->depth_type < 0 || p->depth_type > EA_DEPTH_F32) return ea_fail(EA_ERR_INVALID_ARG, "unknown depth_type");
  CU(cudaSetDevice(ctx->device));
  ea_frameset* fs = new (std::nothrow) ea_frameset();
  if (!fs) return ea_fail(EA_ERR_INVALID_ARG, "out of host memory");
  fs->ctx = ctx; fs->p = *p; fs->n_slots = n_slots;
  fs->depth_elem = (p->depth_type == EA_DEPTH_F32) ? 4 : 2;
  fs->inv_depth_unit = (p->depth_type == EA_DEPTH_F32) ? 1.0 : 1.0 / p->depth_scale;
  const int cap0 = p->max_points > 0 ? p->max_points : (p->width * p->height) / 4;
  int rc = EA_OK;
  for (int l = 0; l < p->n_levels && rc == EA_OK; ++l) {
    EaPrepLevel& L = fs->lv[l];
    L.w = p->width >> l; L.h = p->height >> l; L.words = (L.w + 31) / 32;
    // coarse levels have a much higher edge density (and are small): give them every pixel
    L.cap = (l == 0) ? std::max(64, std::min(L.w * L.h, cap0)) : std::min(L.w * L.h, std::max(cap0, 64));
    const size_t px = size_t(L.w) * L.h;
    L.bgr = nullptr; L.depth = nullptr;
    if (l > 0) {
      rc = fs_alloc(fs, (void**)&L.bgr, px * 3 * n_slots);
      if (rc == EA_OK) rc = fs_alloc(fs, (void**)&L.depth, px * (p->depth_type == EA_DEPTH_F32 ? 4 : 2) * n_slots);
    }
    if (rc == EA_OK) rc = fs_alloc(fs, (void**)&L.edge_bits, size_t(L.h) * L.words * 4 * n_slots);
    if (rc == EA_OK) rc = fs_alloc(fs, (void**)&L.ref_bits, size_t(L.h) * L.words * 4 * n_slots);
    if (rc == EA_OK) rc = fs_alloc(fs, (void**)&L.med_bits, size_t(L.h) * L.words * 4 * n_slots);
    // replicate-padded rows (EA_DT_PAD); + one row of slack so that vector accesses of a row's tail stay inside the pool
    L.dt_pitch = ea_dt_pitch(L.w); L.dt_slot = ea_dt_slot_floats(L.w, L.h);
    if (rc == EA_OK) rc = fs_alloc(fs, (void**)&L.dt, (L.dt_slot * n_slots + L.dt_pitch) * 4);
    if (rc == EA_OK) rc = fs_alloc(fs, (void**)&L.pts, size_t(L.cap) * 16 * n_slots);
    const double s = 1.0 / double(1 << l);
    EaLevelGeom& G = fs->geom[l];
    G.fx = p->fx * s; G.fy = p->fy * s;
    G.cx = (p->cx + 0.5) * s - 0.5; G.cy = (p->cy + 0.5) * s - 0.5;   // pixel-centre convention (DESIGN.md "Pyramid")
    G.inv_fx = 1.0 / G.fx; G.inv_fy = 1.0 / G.fy; G.w = L.w; G.h = L.h;
  }
  if (rc == EA_OK && (p->edge_detector != EA_EDGE_LAPLACIAN || p->dt_kind == EA_DT_EXACT)) {
    const size_t px0 = size_t(p->width) * p->height;
    fs->scratch.stride = px0;
    rc = fs_alloc(fs, (void**)&fs->scratch.gray, px0 * n_slots);
    if (rc == EA_OK) rc = fs_alloc(fs, (void**)&fs->scratch.mag, px0 * 4 * n_slots);
    if (rc == EA_OK) rc = fs_alloc(fs, (void**)&fs->scratch.dxy, px0 * 4 * n_slots);
    if (rc == EA_OK) rc = fs_alloc(fs, (void**)&fs->scratch.map, px0 * n_slots);
  }
  if (rc == EA_OK) rc = fs_alloc(fs, (void**)&fs->d_npts, size_t(n_slots) * EA_MAX_LEVELS * sizeof(int));
  if (rc == EA_OK) rc = fs_alloc(fs, (void**)&fs->d_minmax, size_t(n_slots) * EA_MAX_LEVELS * 2 * sizeof(unsigned));
  if (rc == EA_OK) rc = fs_alloc(fs, (void**)&fs->d_overflow, size_t(n_slots) * EA_MAX_LEVELS * sizeof(int));
  if (rc == EA_OK) rc = fs_alloc(fs, (void**)&fs->d_affine, size_t(n_slots) * EA_MAX_LEVELS * sizeof(float2));
  if (rc == EA_OK) rc = fs_alloc(fs, (void**)&fs->d_desc, size_t(n_slots) * EA_MAX_LEVELS * sizeof(EaLevelDesc));
  if (rc != EA_OK) { ea_frameset_destroy(fs); return rc; }
  cudaMemsetAsync(fs->d_npts, 0, size_t(n_slots) * EA_MAX_LEVELS * sizeof(int), ctx->stream);
  cudaMemsetAsync(fs->d_overflow, 0, size_t(n_slots) * EA_MAX_LEVELS * sizeof(int), ctx->stream);
  {
    std::vector<float2> ones(size_t(n_slots) * EA_MAX_LEVELS, make_float2(1.0f, 0.0f));
    cudaMemcpy(fs->d_affine, ones.data(), ones.size() * sizeof(float2), cudaMemcpyHostToDevice);
  }
  fs->h_desc.assign(size_t(n_slots) * EA_MAX_LEVELS, EaLevelDesc{});
  for (int s = 0; s < n_slots; ++s)
    for (int l = 0; l < p->n_levels; ++l) {
      EaLevelDesc& D = fs->h_desc[size_t(s) * EA_MAX_LEVELS + l];
      const EaPrepLevel& L = fs->lv[l];
      D.pts = L.pts + size_t(s) * L.cap;
      D.n_pts = fs->d_npts + size_t(s) * EA_MAX_LEVELS + l;
      D.dt = ea_dt_origin(L, s);
      D.dt_affine = fs->d_affine + size_t(s) * EA_MAX_LEVELS + l;
      D.w = L.w; D.h = L.h; D.pts_mode = EA_POINTS_PIXEL; D.dt_pitch = L.dt_pitch;
      D.truncated = fs->d_overflow + size_t(s) * EA_MAX_LEVELS + l;
    }
  CU(cudaMemcpyAsync(fs->d_desc, fs->h_desc.data(), fs->h_desc.size() * sizeof(EaLevelDesc), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  *out = fs;
  return EA_OK;
}

int ea_frameset_destroy(ea_frameset* fs) {
  if (!fs) return EA_OK;
  cudaSetDevice(fs->ctx->device);
  cudaStreamSynchronize(fs->ctx->stream);
  for (void* p : fs->allocs) cudaFree(p);
  if (fs->stage_bgr) cudaFree(fs->stage_bgr);
  if (fs->stage_depth) cudaFree(fs->stage_depth);
  delete fs;
  return EA_OK;
}

static int check_slots(ea_frameset* fs, int n, const int32_t* slots) {
  if (!fs || n <= 0 || !slots) return ea_fail(EA_ERR_INVALID_ARG, "frameset/slots: null or empty");
  if (n > fs->n_slots) return ea_fail(EA_ERR_INVALID_ARG, "more frames (%d) than slots (%d)", n, fs->n_slots);
  for (int i = 0; i < n; ++i)
    if (slots[i] < 0 || slots[i] >= fs->n_slots) return ea_fail(EA_ERR_INVALID_ARG, "slot %d out of range [0,%d)", slots[i], fs->n_slots);
  return EA_OK;
}

}  // extern "C"

// The compaction kernel writes packed pixel points: a slot that held caller-supplied 3-D points (ea_frameset_set_points with
// EA_POINTS_XYZ) goes back to pixel mode when it is preprocessed as a reference frame.
static int reset_points_mode(ea_frameset* fs, int n, const int32_t* slots) {
  ea_context* c = fs->ctx;
  for (int i = 0; i < n; ++i)
    for (int l = 0; l < fs->p.n_levels; ++l) {
      EaLevelDesc& D = fs->h_desc[size_t(slots[i]) * EA_MAX_LEVELS + l];
      if (D.pts_mode == EA_POINTS_PIXEL) continue;
      D.pts_mode = EA_POINTS_PIXEL;
      CU(cudaMemcpyAsync(fs->d_desc + size_t(slots[i]) * EA_MAX_LEVELS + l, &D, sizeof D, cudaMemcpyHostToDevice, c->stream));
      CU(cudaStreamSynchronize(c->stream));       // D lives in pageable host memory owned by the frameset
    }
  return EA_OK;
}

// ---- image layouts -------------------------------------------------------------------------------------------------------
size_t ea_layout_row_bytes(const ea_image_layout& L, int w) {
  static const int bpp[] = {3, 1, 1, 2, 2};   // BGR8, GRAY8, NV12 (luma), YUYV, UYVY
  return size_t(w) * bpp[L.format];
}

int ea_resolve_layout(const ea_image_layout* in, int w, int h, bool on_device, ea_image_layout* out) {
  if (!in) return ea_fail(EA_ERR_INVALID_ARG, "image layout is null");
  ea_image_layout L = *in;
  if (L.format < EA_IMAGE_BGR8 || L.format > EA_IMAGE_UYVY) return ea_fail(EA_ERR_INVALID_ARG, "unknown image format %d", L.format);
  if (L.reserved != 0) return ea_fail(EA_ERR_INVALID_ARG, "ea_image_layout.reserved must be 0");
  if (L.format == EA_IMAGE_NV12 && (h & 1)) return ea_fail(EA_ERR_INVALID_ARG, "NV12 frames need an even height (h = %d)", h);
  if ((L.format == EA_IMAGE_YUYV || L.format == EA_IMAGE_UYVY) && (w & 1))
    return ea_fail(EA_ERR_INVALID_ARG, "YUYV / UYVY frames need an even width (w = %d)", w);
  const int64_t row = int64_t(ea_layout_row_bytes(L, w));
  if (L.row_pitch == 0) L.row_pitch = row;
  if (L.row_pitch < row || L.row_pitch > INT32_MAX)
    return ea_fail(EA_ERR_INVALID_ARG, "row_pitch %lld: must be in [%lld, 2^31)", (long long)L.row_pitch, (long long)row);
  if (L.frame_stride == 0) L.frame_stride = L.format == EA_IMAGE_NV12 ? 3 * int64_t(h) * L.row_pitch / 2 : int64_t(h) * L.row_pitch;
  // the host path copies the frames as one 3-D copy of rows that are row_pitch apart, frames included
  if (L.frame_stride < int64_t(h) * L.row_pitch || L.frame_stride % L.row_pitch != 0)
    return ea_fail(EA_ERR_INVALID_ARG, "frame_stride %lld: must be a multiple of row_pitch %lld and at least h * row_pitch",
                   (long long)L.frame_stride, (long long)L.row_pitch);
  // the BGR kernels on device memory read dense frames only
  if (on_device && L.format == EA_IMAGE_BGR8 && (L.row_pitch != row || L.frame_stride != int64_t(h) * row))
    return ea_fail(EA_ERR_INVALID_ARG, "BGR8 frames in device memory must be dense");
  *out = L;
  return EA_OK;
}

ea_image_layout ea_staged_layout(const ea_image_layout& L, int w, int h) {
  ea_image_layout S = L;
  if (S.format == EA_IMAGE_NV12) S.format = EA_IMAGE_GRAY8;
  S.row_pitch = int64_t(ea_layout_row_bytes(L, w));
  S.frame_stride = int64_t(h) * S.row_pitch;
  return S;
}

cudaError_t ea_upload_frames(uint8_t* dst, const uint8_t* src, const ea_image_layout& L, int w, int h, int n, cudaStream_t stream) {
  const size_t row = ea_layout_row_bytes(L, w), pitch = size_t(L.row_pitch), rows = size_t(L.frame_stride) / pitch;
  if (pitch == row && rows == size_t(h)) return cudaMemcpyAsync(dst, src, row * h * n, cudaMemcpyHostToDevice, stream);   // dense
  if (rows == size_t(h))        // rows evenly spaced across frames
    return cudaMemcpy2DAsync(dst, row, src, pitch, row, size_t(h) * n, cudaMemcpyHostToDevice, stream);
  cudaMemcpy3DParms p = {};
  p.srcPtr = make_cudaPitchedPtr(const_cast<uint8_t*>(src), pitch, row, rows);
  p.dstPtr = make_cudaPitchedPtr(dst, row, row, size_t(h));
  p.extent = make_cudaExtent(row, size_t(h), size_t(n));
  p.kind = cudaMemcpyHostToDevice;
  return cudaMemcpy3DAsync(&p, stream);
}

// Behind every preprocessing entry point: checks the call, stages host buffers in the frame set (the staging area is sized for
// BGR frames; the other formats take the first third or two of it), copies the slot list to the device and launches.
static int preprocess_frames(ea_frameset* fs, int n, const int32_t* slots, int roles, EaFrameInput in) {
  int rc = check_slots(fs, n, slots);
  if (rc) return rc;
  if (!in.image) return ea_fail(EA_ERR_INVALID_ARG, "image is null");
  rc = ea_resolve_layout(&in.layout, fs->p.width, fs->p.height, !in.on_host, &in.layout);
  if (rc) return rc;
  if (roles != EA_ROLE_REF && roles != EA_ROLE_NOW && roles != EA_ROLE_BOTH)
    return ea_fail(EA_ERR_INVALID_ARG, "roles must be EA_ROLE_REF, EA_ROLE_NOW or EA_ROLE_BOTH");
  const bool ref = (roles & EA_ROLE_REF) != 0;
  if (ref && !in.depth) return ea_fail(EA_ERR_INVALID_ARG, "EA_ROLE_REF needs depth");
  if (in.ref_mask && !ref) return ea_fail(EA_ERR_INVALID_ARG, "a reference mask only applies to the reference role");
  if (in.now_mask && !(roles & EA_ROLE_NOW)) return ea_fail(EA_ERR_INVALID_ARG, "a now mask only applies to the now role");
  if (!ref) in.depth = nullptr;     // nothing else reads it
  ea_context* c = fs->ctx;
  CU(cudaSetDevice(c->device));
  EaAsyncBuf d_masks(c->stream), d_slots(c->stream);      // released on every return path
  if (in.on_host) {
    const size_t px = size_t(fs->p.width) * fs->p.height;
    if (!fs->stage_bgr) CU(cudaMalloc((void**)&fs->stage_bgr, px * 3 * fs->n_slots));
    CU(ea_upload_frames(fs->stage_bgr, in.image, in.layout, fs->p.width, fs->p.height, n, c->stream));
    in.image = fs->stage_bgr;
    in.layout = ea_staged_layout(in.layout, fs->p.width, fs->p.height);
    if (in.depth) {
      if (!fs->stage_depth) CU(cudaMalloc(&fs->stage_depth, px * fs->depth_elem * fs->n_slots));
      CU(cudaMemcpyAsync(fs->stage_depth, in.depth, px * fs->depth_elem * n, cudaMemcpyHostToDevice, c->stream));
      in.depth = fs->stage_depth;
    }
    const int n_masks = (in.ref_mask ? 1 : 0) + (in.now_mask ? 1 : 0);
    if (n_masks) CU(d_masks.alloc(px * n * n_masks));
    uint8_t* m = d_masks.as<uint8_t>();
    if (in.ref_mask) { CU(cudaMemcpyAsync(m, in.ref_mask, px * n, cudaMemcpyHostToDevice, c->stream)); in.ref_mask = m; m += px * n; }
    if (in.now_mask) { CU(cudaMemcpyAsync(m, in.now_mask, px * n, cudaMemcpyHostToDevice, c->stream)); in.now_mask = m; }
    in.on_host = false;
  }
  // the slot list goes through a buffer of the call's own, so the caller may reuse its array at once
  CU(d_slots.alloc(size_t(n) * sizeof(int32_t)));
  CU(cudaMemcpyAsync(d_slots.p, slots, size_t(n) * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream));
  rc = ea_launch_preprocess(fs, n, d_slots.as<int32_t>(), roles, in, c->stream, EA_COMPACT_INLINE, nullptr);
  if (rc == EA_OK && ref) rc = reset_points_mode(fs, n, slots);
  return rc;
}

static ea_image_layout dense(int format) { return ea_image_layout{format, 0, 0, 0}; }

extern "C" {
int ea_frameset_preprocess_host(ea_frameset* fs, int n, const int32_t* slots, const uint8_t* bgr, const void* depth, int roles) {
  return preprocess_frames(fs, n, slots, roles, {bgr, dense(EA_IMAGE_BGR8), depth, nullptr, nullptr, true});
}

int ea_frameset_preprocess_device(ea_frameset* fs, int n, const int32_t* slots, const uint8_t* d_bgr, const void* d_depth, int roles) {
  return preprocess_frames(fs, n, slots, roles, {d_bgr, dense(EA_IMAGE_BGR8), d_depth, nullptr, nullptr, false});
}

int ea_frameset_preprocess_masked(ea_frameset* fs, int n, const int32_t* slots, const uint8_t* bgr, const void* depth,
                                  const uint8_t* mask, int roles) {
  if (!mask) return ea_fail(EA_ERR_INVALID_ARG, "mask is null");
  return preprocess_frames(fs, n, slots, roles, {bgr, dense(EA_IMAGE_BGR8), depth, mask, nullptr, true});
}

int ea_frameset_preprocess_now_masked(ea_frameset* fs, int n, const int32_t* slots, const uint8_t* bgr, const uint8_t* mask) {
  if (!mask) return ea_fail(EA_ERR_INVALID_ARG, "mask is null");
  return preprocess_frames(fs, n, slots, EA_ROLE_NOW, {bgr, dense(EA_IMAGE_BGR8), nullptr, nullptr, mask, true});
}

// ---- 8-bit gray input: the same pipeline as on BGR (g, g, g), from a third of the bytes -----------------------------------
int ea_frameset_preprocess_gray_host(ea_frameset* fs, int n, const int32_t* slots, const uint8_t* gray, const void* depth,
                                     const uint8_t* ref_mask, const uint8_t* now_mask, int roles) {
  return preprocess_frames(fs, n, slots, roles, {gray, dense(EA_IMAGE_GRAY8), depth, ref_mask, now_mask, true});
}

int ea_frameset_preprocess_gray_device(ea_frameset* fs, int n, const int32_t* slots, const uint8_t* d_gray, const void* d_depth, int roles) {
  return preprocess_frames(fs, n, slots, roles, {d_gray, dense(EA_IMAGE_GRAY8), d_depth, nullptr, nullptr, false});
}

// ---- frames with a row pitch (NV12 / YUYV / UYVY, pitched GRAY8 / BGR8): the luma is read where it lies ---------------------
int ea_frameset_preprocess_image_host(ea_frameset* fs, int n, const int32_t* slots, const ea_image_layout* layout, const uint8_t* image,
                                      const void* depth, const uint8_t* ref_mask, const uint8_t* now_mask, int roles) {
  if (!layout) return ea_fail(EA_ERR_INVALID_ARG, "image layout is null");
  return preprocess_frames(fs, n, slots, roles, {image, *layout, depth, ref_mask, now_mask, true});
}

int ea_frameset_preprocess_image_device(ea_frameset* fs, int n, const int32_t* slots, const ea_image_layout* layout, const uint8_t* d_image,
                                        const void* d_depth, const uint8_t* d_ref_mask, const uint8_t* d_now_mask, int roles) {
  if (!layout) return ea_fail(EA_ERR_INVALID_ARG, "image layout is null");
  return preprocess_frames(fs, n, slots, roles, {d_image, *layout, d_depth, d_ref_mask, d_now_mask, false});
}

static int check_slot_level(ea_frameset* fs, int slot, int level) {
  if (!fs) return ea_fail(EA_ERR_INVALID_ARG, "null frameset");
  if (slot < 0 || slot >= fs->n_slots) return ea_fail(EA_ERR_INVALID_ARG, "slot %d out of range", slot);
  if (level < 0 || level >= fs->p.n_levels) return ea_fail(EA_ERR_INVALID_ARG, "level %d out of range", level);
  return EA_OK;
}

int ea_frameset_set_points(ea_frameset* fs, int slot, int level, const float* pts4, int n, int mode) {
  int rc = check_slot_level(fs, slot, level);
  if (rc) return rc;
  const EaPrepLevel& L = fs->lv[level];
  if (n < 0 || n > L.cap) return ea_fail(EA_ERR_CAPACITY, "%d points exceed the level capacity %d (raise max_points)", n, L.cap);
  if (n > 0 && !pts4) return ea_fail(EA_ERR_INVALID_ARG, "pts4 is null");
  if (mode != EA_POINTS_PIXEL && mode != EA_POINTS_XYZ) return ea_fail(EA_ERR_INVALID_ARG, "bad points mode");
  ea_context* c = fs->ctx;
  CU(cudaSetDevice(c->device));
  EaLevelDesc& D = fs->h_desc[size_t(slot) * EA_MAX_LEVELS + level];
  std::vector<uint2> packed;
  if (mode == EA_POINTS_PIXEL) {      // the device keeps pixel points as 8 bytes {u | v << 16, raw depth}
    packed.resize(size_t(n));
    for (int i = 0; i < n; ++i) {
      const float u = pts4[4 * i], v = pts4[4 * i + 1];
      if (!(u >= 0.0f && u <= 65535.0f && v >= 0.0f && v <= 65535.0f) || u != std::floor(u) || v != std::floor(v))
        return ea_fail(EA_ERR_INVALID_ARG, "EA_POINTS_PIXEL point %d: (%g, %g) is not an integer pixel position (use EA_POINTS_XYZ)", i, u, v);
      packed[size_t(i)] = ea_pack_pixel_point(unsigned(u), unsigned(v), pts4[4 * i + 2]);
    }
    D.pts_mode = mode;     // only now: a rejected list leaves the host and device descriptors untouched
    if (n > 0) CU(cudaMemcpyAsync(const_cast<void*>(D.pts), packed.data(), size_t(n) * 8, cudaMemcpyHostToDevice, c->stream));
  } else {
    D.pts_mode = mode;
  }
  if (mode == EA_POINTS_XYZ && n > 0) {
    CU(cudaMemcpyAsync(const_cast<void*>(D.pts), pts4, size_t(n) * 16, cudaMemcpyHostToDevice, c->stream));
  }
  CU(cudaMemcpyAsync(const_cast<int*>(D.n_pts), &n, sizeof(int), cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemsetAsync(fs->d_overflow + size_t(slot) * EA_MAX_LEVELS + level, 0, sizeof(int), c->stream));   // a complete caller-supplied list
  CU(cudaMemcpyAsync(fs->d_desc + size_t(slot) * EA_MAX_LEVELS + level, &D, sizeof D, cudaMemcpyHostToDevice, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return EA_OK;
}
int ea_frameset_set_dt(ea_frameset* fs, int slot, int level, const float* dt) {
  int rc = check_slot_level(fs, slot, level);
  if (rc) return rc;
  if (!dt) return ea_fail(EA_ERR_INVALID_ARG, "dt is null");
  const EaPrepLevel& L = fs->lv[level];
  ea_context* c = fs->ctx;
  CU(cudaSetDevice(c->device));
  rc = ea_ensure_tmp(c, size_t(L.w) * L.h * 4);
  if (rc) return rc;
  CU(cudaMemcpyAsync(c->d_tmp, dt, size_t(L.w) * L.h * 4, cudaMemcpyHostToDevice, c->stream));
  cudaError_t e = ea_launch_dt_import((const float*)c->d_tmp, ea_dt_origin(L, slot), L.w, L.h, L.dt_pitch, c->stream);   // interior + replicated border
  c->launches++;
  if (e != cudaSuccess) return ea_fail(EA_ERR_CUDA, "dt import: %s", cudaGetErrorString(e));
  const float2 one = make_float2(1.0f, 0.0f);   // the caller's DT is used as is
  CU(cudaMemcpyAsync(fs->d_affine + size_t(slot) * EA_MAX_LEVELS + level, &one, sizeof one, cudaMemcpyHostToDevice, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return EA_OK;
}
int ea_frameset_get_num_points(ea_frameset* fs, int slot, int level, int* n) {
  int rc = check_slot_level(fs, slot, level);
  if (rc) return rc;
  if (!n) return ea_fail(EA_ERR_INVALID_ARG, "n is null");
  ea_context* c = fs->ctx;
  CU(cudaSetDevice(c->device));
  int ovf = 0;
  CU(cudaMemcpyAsync(n, fs->d_npts + size_t(slot) * EA_MAX_LEVELS + level, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaMemcpyAsync(&ovf, fs->d_overflow + size_t(slot) * EA_MAX_LEVELS + level, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  if (ovf) return ea_fail(EA_ERR_CAPACITY, "the point list of slot %d level %d was truncated at max_points; raise ea_frame_params.max_points", slot, level);
  return EA_OK;
}
int ea_frameset_get_points(ea_frameset* fs, int slot, int level, float* pts4, int cap, int* n) {
  int m = 0;
  int rc = ea_frameset_get_num_points(fs, slot, level, &m);
  if (rc && rc != EA_ERR_CAPACITY) return rc;
  if (n) *n = m;
  const int k = std::min(m, cap);
  if (k > 0 && pts4) {
    ea_context* c = fs->ctx;
    const EaLevelDesc& D = fs->h_desc[size_t(slot) * EA_MAX_LEVELS + level];
    if (D.pts_mode == EA_POINTS_PIXEL) {
      std::vector<uint2> packed(static_cast<size_t>(k));
      CU(cudaMemcpyAsync(packed.data(), D.pts, size_t(k) * 8, cudaMemcpyDeviceToHost, c->stream));
      CU(cudaStreamSynchronize(c->stream));
      for (int i = 0; i < k; ++i) {
        float d; std::memcpy(&d, &packed[size_t(i)].y, 4);
        pts4[4 * i] = float(packed[size_t(i)].x & 0xffffu); pts4[4 * i + 1] = float(packed[size_t(i)].x >> 16);
        pts4[4 * i + 2] = d; pts4[4 * i + 3] = 1.0f;
      }
    } else {
      CU(cudaMemcpyAsync(pts4, D.pts, size_t(k) * 16, cudaMemcpyDeviceToHost, c->stream));
      CU(cudaStreamSynchronize(c->stream));
    }
  }
  return rc;
}
int ea_frameset_get_dt(ea_frameset* fs, int slot, int level, float* dt) {
  int rc = check_slot_level(fs, slot, level);
  if (rc) return rc;
  if (!dt) return ea_fail(EA_ERR_INVALID_ARG, "dt is null");
  const EaPrepLevel& L = fs->lv[level];
  ea_context* c = fs->ctx;
  CU(cudaSetDevice(c->device));
  // the device keeps the raw chamfer DT plus the normalisation {scale, shift}; hand back the normalised image
  rc = ea_ensure_tmp(c, size_t(L.w) * L.h * 4);
  if (rc) return rc;
  cudaError_t e = ea_launch_dt_normalized_copy(ea_dt_origin(L, slot), L.dt_pitch, fs->d_affine + size_t(slot) * EA_MAX_LEVELS + level,
                                              L.w, L.h, (float*)c->d_tmp, c->stream);
  c->launches++;
  if (e != cudaSuccess) return ea_fail(EA_ERR_CUDA, "dt copy: %s", cudaGetErrorString(e));
  CU(cudaMemcpyAsync(dt, c->d_tmp, size_t(L.w) * L.h * 4, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return EA_OK;
}
int ea_frameset_get_edge_mask(ea_frameset* fs, int slot, int level, int which, uint8_t* mask) {
  int rc = check_slot_level(fs, slot, level);
  if (rc) return rc;
  if (!mask) return ea_fail(EA_ERR_INVALID_ARG, "mask is null");
  const EaPrepLevel& L = fs->lv[level];
  ea_context* c = fs->ctx;
  CU(cudaSetDevice(c->device));
  rc = ea_ensure_tmp(c, size_t(L.w) * L.h);
  if (rc) return rc;
  cudaError_t e = ea_launch_unpack_mask(L.edge_bits + size_t(slot) * L.h * L.words, L.w, L.h, L.words, which, (uint8_t*)c->d_tmp, c->stream);
  c->launches++;
  if (e != cudaSuccess) return ea_fail(EA_ERR_CUDA, "unpack mask: %s", cudaGetErrorString(e));
  CU(cudaMemcpyAsync(mask, c->d_tmp, size_t(L.w) * L.h, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return EA_OK;
}
int ea_frameset_level_geometry(ea_frameset* fs, int level, int* w, int* h, double k4[4]) {
  int rc = check_slot_level(fs, 0, level);
  if (rc) return rc;
  if (w) *w = fs->lv[level].w;
  if (h) *h = fs->lv[level].h;
  if (k4) { k4[0] = fs->geom[level].fx; k4[1] = fs->geom[level].fy; k4[2] = fs->geom[level].cx; k4[3] = fs->geom[level].cy; }
  return EA_OK;
}

// ---- evaluation / solve -------------------------------------------------------------------------------------
int ea_check_solve_params(const ea_solve_params* sp) {
  if (!sp) return ea_fail(EA_ERR_INVALID_ARG, "solve params are null");
  if (sp->point_stride < 1) return ea_fail(EA_ERR_INVALID_ARG, "point_stride must be >= 1");
  if (sp->loss_type < EA_LOSS_TRIVIAL || sp->loss_type > EA_LOSS_HUBER) return ea_fail(EA_ERR_INVALID_ARG, "unknown loss type");
  if (!(sp->loss_scale > 0)) return ea_fail(EA_ERR_INVALID_ARG, "loss_scale must be positive");
  if (sp->max_num_iterations < 0) return ea_fail(EA_ERR_INVALID_ARG, "max_num_iterations must be >= 0");
  if (sp->trust_region_strategy < 0 || sp->trust_region_strategy > 1) return ea_fail(EA_ERR_INVALID_ARG, "trust_region_strategy must be 0 (LM) or 1 (DOGLEG)");
  const int cs = sp->cluster_size;
  if (!(cs == 0 || cs == 1 || cs == 2 || cs == 4 || cs == 8)) return ea_fail(EA_ERR_INVALID_ARG, "cluster_size must be 0,1,2,4 or 8");
  return EA_OK;
}
static int check_pairable(ea_frameset* ref, ea_frameset* now) {
  if (!ref || !now) return ea_fail(EA_ERR_INVALID_ARG, "null frameset");
  if (ref->ctx->device != now->ctx->device) return ea_fail(EA_ERR_INVALID_ARG, "framesets live on different devices");
  if (ref->p.n_levels != now->p.n_levels || ref->p.width != now->p.width || ref->p.height != now->p.height)
    return ea_fail(EA_ERR_INVALID_ARG, "ref/now framesets differ in geometry");
  return EA_OK;
}

int ea_eval(ea_context* c, ea_frameset* ref, int ref_slot, ea_frameset* now, int now_slot, int level, const double* pose7,
            const ea_solve_params* sp, int* n_residuals, double* raw, double* residuals, double* jac, double* sums28, int* failed) {
  if (!c || !pose7) return ea_fail(EA_ERR_INVALID_ARG, "null argument");
  int rc = ea_check_solve_params(sp);
  if (!rc) rc = check_pairable(ref, now);
  if (!rc) rc = check_slot_level(ref, ref_slot, level);
  if (!rc) rc = check_slot_level(now, now_slot, level);
  if (rc) return rc;
  CU(cudaSetDevice(c->device));
  int n_pts = 0;
  rc = ea_frameset_get_num_points(ref, ref_slot, level, &n_pts);
  if (rc) return rc;
  const int n_res = (n_pts + sp->point_stride - 1) / sp->point_stride;
  if (n_residuals) *n_residuals = n_res;
  const EaLevelDesc& rd = ref->h_desc[size_t(ref_slot) * EA_MAX_LEVELS + level];
  const EaLevelDesc& nd = now->h_desc[size_t(now_slot) * EA_MAX_LEVELS + level];
  CU(cudaMemcpyAsync(c->d_pose, pose7, 7 * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemsetAsync(c->d_failed, 0, sizeof(int), c->stream));
  const double ids = ref->inv_depth_unit;
  if (n_res > 0 && (raw || residuals || jac || failed)) {
    rc = ea_ensure_tmp(c, size_t(n_res) * 8 * sizeof(double));
    if (rc) return rc;
    double* d_raw = (double*)c->d_tmp; double* d_res = d_raw + n_res; double* d_jac = d_res + n_res;
    cudaError_t e = ea_launch_eval_points(rd, nd, ref->geom[level], now->geom[level], ids, *sp, c->d_pose, n_res, d_raw, d_res, d_jac, c->d_failed, c->stream);
    c->launches++;
    if (e != cudaSuccess) return ea_fail(EA_ERR_CUDA, "eval launch: %s", cudaGetErrorString(e));
    if (raw) CU(cudaMemcpyAsync(raw, d_raw, size_t(n_res) * 8, cudaMemcpyDeviceToHost, c->stream));
    if (residuals) CU(cudaMemcpyAsync(residuals, d_res, size_t(n_res) * 8, cudaMemcpyDeviceToHost, c->stream));
    if (jac) CU(cudaMemcpyAsync(jac, d_jac, size_t(n_res) * 48, cudaMemcpyDeviceToHost, c->stream));
    if (failed) CU(cudaMemcpyAsync(failed, c->d_failed, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  } else if (failed) *failed = 0;
  if (sums28) {
    for (int k = 0; k < 28; ++k) sums28[k] = 0.0;
    if (n_res > 0) {
      const int nb = std::max(1, std::min(c->sm_count, (n_res + 2047) / 2048));
      cudaError_t e = ea_launch_eval_sums(rd, nd, ref->geom[level], now->geom[level], ids, *sp, c->d_pose, nullptr, 0, n_res, nb, c->d_sums, c->stream);
      c->launches++;
      if (e != cudaSuccess) return ea_fail(EA_ERR_CUDA, "eval sums launch: %s", cudaGetErrorString(e));
      std::vector<double> h(size_t(nb) * EA_SUMS);
      CU(cudaMemcpyAsync(h.data(), c->d_sums, h.size() * 8, cudaMemcpyDeviceToHost, c->stream));
      CU(cudaStreamSynchronize(c->stream));
      ea_fold_sums28(h.data(), nb, sums28);
    }
  }
  CU(cudaStreamSynchronize(c->stream));
  return EA_OK;
}

static int fill_solve_args(ea_frameset* ref, ea_frameset* now, const ea_solve_params* sp, EaSolveArgs& A) {
  int rc = ea_check_solve_params(sp);
  if (!rc) rc = check_pairable(ref, now);
  if (rc) return rc;
  std::memset(&A, 0, sizeof A);
  A.ref_desc = ref->d_desc; A.now_desc = now->d_desc;
  A.n_levels = ref->p.n_levels;
  A.coarsest = sp->coarsest_level < 0 ? ref->p.n_levels - 1 : sp->coarsest_level;
  A.finest = sp->finest_level;
  if (A.coarsest >= ref->p.n_levels || A.finest < 0 || A.finest > A.coarsest) return ea_fail(EA_ERR_INVALID_ARG, "bad level range [%d..%d]", A.coarsest, A.finest);
  A.inv_depth_scale = ref->inv_depth_unit;
  for (int l = 0; l < ref->p.n_levels; ++l) { A.ref_geom[l] = ref->geom[l]; A.now_geom[l] = now->geom[l]; A.ref_cap[l] = ref->lv[l].cap; }
  A.sp = *sp;
  A.loss = ea_eval_consts(sp->loss_type, sp->loss_scale, sp->point_stride);
  return EA_OK;
}

int ea_solve_batch_device(ea_context* c, int n, ea_frameset* ref, const int32_t* d_ref_slots, ea_frameset* now,
                          const int32_t* d_now_slots, double* d_poses7, const int32_t* d_pose_index,
                          const ea_solve_params* sp, ea_summary* d_summaries) {
  return ea_solve_batch_device_ordered(c, n, ref, d_ref_slots, now, d_now_slots, d_poses7, d_pose_index, nullptr, sp, d_summaries);
}
}  // extern "C"

// Gather-roof probe over n pairs (measurement only, see ea_k_gather_probe): device time of `repeats` sweeps over the
// level's point lists and the number of point-gathers they contain.
int ea_probe_gather_device(ea_context* c, int n, ea_frameset* ref, const int32_t* d_ref_slots, ea_frameset* now, const int32_t* d_now_slots,
                           const double* d_poses7, int level, int repeats, float* ms, double* point_gathers) {
  if (!c || !ref || !now || !d_ref_slots || !d_now_slots || !d_poses7 || !ms || !point_gathers) return ea_fail(EA_ERR_INVALID_ARG, "null argument");
  if (n <= 0 || repeats <= 0) return ea_fail(EA_ERR_INVALID_ARG, "n and repeats must be positive");
  ea_solve_params sp;
  ea_solve_params_default(&sp);
  EaSolveArgs A;
  int rc = fill_solve_args(ref, now, &sp, A);
  if (rc) return rc;
  if (level < 0 || level >= ref->p.n_levels) return ea_fail(EA_ERR_INVALID_ARG, "level %d out of range", level);
  CU(cudaSetDevice(c->device));
  A.ref_slots = d_ref_slots; A.now_slots = d_now_slots; A.poses = const_cast<double*>(d_poses7); A.n_pairs = n;
  const int slices = std::max(1, (c->sm_count * 8 + n - 1) / n);
  EaDevBuf sink;
  EaEventPair ev;
  CU(sink.alloc(size_t(n) * slices * 256 * sizeof(float)));
  CU(ev.create());
  float* d_sink = sink.as<float>();
  cudaError_t e = ea_launch_gather_probe(A, level, slices, 1, d_sink, c->stream);     // warm-up sweep
  CU(cudaEventRecord(ev.a, c->stream));
  if (e == cudaSuccess) e = ea_launch_gather_probe(A, level, slices, repeats, d_sink, c->stream);
  CU(cudaEventRecord(ev.b, c->stream));
  c->launches += 2;
  CU(cudaStreamSynchronize(c->stream));
  if (e != cudaSuccess) return ea_fail(EA_ERR_CUDA, "gather probe: %s", cudaGetErrorString(e));
  CU(cudaEventElapsedTime(ms, ev.a, ev.b));
  // point counts of the level (host copy of the device-resident counters)
  std::vector<int32_t> slots(static_cast<size_t>(n));
  CU(cudaMemcpy(slots.data(), d_ref_slots, size_t(n) * sizeof(int32_t), cudaMemcpyDeviceToHost));
  std::vector<int> npts(size_t(ref->n_slots) * EA_MAX_LEVELS);
  CU(cudaMemcpy(npts.data(), ref->d_npts, npts.size() * sizeof(int), cudaMemcpyDeviceToHost));
  double total = 0.0;
  for (int i = 0; i < n; ++i) total += std::min(npts[size_t(slots[size_t(i)]) * EA_MAX_LEVELS + level], ref->lv[level].cap);
  *point_gathers = total * repeats;
  return EA_OK;
}

int ea_solve_batch_device_ordered(ea_context* c, int n, ea_frameset* ref, const int32_t* d_ref_slots, ea_frameset* now,
                                  const int32_t* d_now_slots, double* d_poses7, const int32_t* d_pose_index,
                                  const int32_t* d_order, const ea_solve_params* sp, ea_summary* d_summaries, bool tail_helpers) {
  if (!c || !d_ref_slots || !d_now_slots || !d_poses7) return ea_fail(EA_ERR_INVALID_ARG, "null argument");
  if (n <= 0) return EA_OK;
  EaSolveArgs A;
  int rc = fill_solve_args(ref, now, sp, A);
  if (rc) return rc;
  CU(cudaSetDevice(c->device));
  A.ref_slots = d_ref_slots; A.now_slots = d_now_slots; A.pose_index = d_pose_index; A.poses = d_poses7;
  A.summaries = d_summaries; A.n_pairs = n; A.work_counter = c->d_work; A.order = d_order;
  A.trace = c->d_trace; A.trace_count = c->d_trace_count; A.trace_cap = c->trace_cap;
  A.debug = c->d_debug;
  // tail helpers: CTAs that find the work queue empty serve the ones still solving.  They shorten the launch, not the work:
  // a caller that has other kernels ready to take over the idle SMs (the tracker's overlapped preprocessing) turns them off.
  A.boards = tail_helpers ? static_cast<EaHelpBoard*>(c->d_boards) : nullptr;
  EaProfileScope prof(c, 1);
  EaSolveShape shape;
  const cudaError_t e = ea_launch_solve_batch(c, A, shape);
  if (c->d_debug && e == cudaSuccess) {   // development aid: synchronous read-back of the cycle counters of every CTA that ran
    cudaStreamSynchronize(c->stream);
    std::vector<unsigned long long> h[2];
    for (int ph = 0; ph < 2; ++ph) {      // {whole launch or fine phase, coarse phase}
      const int grid = shape.grid[ph];
      if (grid == 0) continue;
      h[ph].resize(size_t(grid) * 6);
      cudaMemcpy(h[ph].data(), c->d_debug + size_t(ph) * EA_DEBUG_ROWS * 6, h[ph].size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost);
      for (int k = 0; k < 6; ++k) { double sum = 0; for (int b = 0; b < grid; ++b) sum += double(h[ph][size_t(b) * 6 + k]); c->debug_sum[ph][k] += sum / grid; }
      if (ph == 1) c->debug_launches[1]++;
    }
    {   // owner-lifetime distribution of this launch (the launch ends with the last owner): mean / 75th / 90th percentile / max
      const int grid = shape.grid[0];
      std::vector<double> life(static_cast<size_t>(grid));
      double mean = 0.0;
      for (int b = 0; b < grid; ++b) { life[size_t(b)] = double(h[0][size_t(b) * 6 + 5]); mean += life[size_t(b)] / grid; }
      std::sort(life.begin(), life.end());
      if (c->debug_launches[0] % 7 == 3)
        fprintf(stderr, "[EA_SOLVE_DEBUG] launch %ld: owner lifetimes (kcycles) mean %.0f  p50 %.0f  p75 %.0f  p90 %.0f  p97 %.0f  max %.0f\n", c->debug_launches[0],
                mean / 1e3, life[size_t(grid / 2)] / 1e3, life[size_t(grid * 3 / 4)] / 1e3, life[size_t(grid * 9 / 10)] / 1e3, life[size_t(grid * 97 / 100)] / 1e3, life[size_t(grid - 1)] / 1e3);
    }
    c->debug_launches[0]++;
  }
  c->launches += shape.launches;
  if (e != cudaSuccess) return ea_fail(EA_ERR_CUDA, "solve launch: %s", cudaGetErrorString(e));
  return EA_OK;
}
extern "C" {

int ea_solve_batch(ea_context* c, int n, ea_frameset* ref, const int32_t* ref_slots, ea_frameset* now, const int32_t* now_slots,
                   double* poses7, const ea_solve_params* sp, ea_summary* summaries) {
  if (!c || !ref_slots || !now_slots || !poses7) return ea_fail(EA_ERR_INVALID_ARG, "null argument");
  if (n <= 0) return EA_OK;
  int rc = check_pairable(ref, now);
  if (!rc) rc = check_slots(ref, std::min(n, ref->n_slots), ref_slots);
  if (rc) return rc;
  for (int i = 0; i < n; ++i) {
    if (ref_slots[i] < 0 || ref_slots[i] >= ref->n_slots || now_slots[i] < 0 || now_slots[i] >= now->n_slots)
      return ea_fail(EA_ERR_INVALID_ARG, "pair %d: slot out of range", i);
    double q2 = 0;
    for (int k = 0; k < 4; ++k) q2 += poses7[i * 7 + k] * poses7[i * 7 + k];
    if (!(q2 > 0.999999 && q2 < 1.000001)) return ea_fail(EA_ERR_INVALID_ARG, "pair %d: quaternion is not unit (|q|^2=%g)", i, q2);
  }
  CU(cudaSetDevice(c->device));
  const int L = ref->p.n_levels;
  const size_t bytes = size_t(n) * (2 * sizeof(int32_t) + 7 * sizeof(double)) + size_t(n) * L * sizeof(ea_summary) + 64;
  rc = ea_ensure_tmp(c, bytes);
  if (rc) return rc;
  char* base = (char*)c->d_tmp;
  double* d_poses = (double*)base; base += size_t(n) * 7 * sizeof(double);
  ea_summary* d_sum = (ea_summary*)base; base += size_t(n) * L * sizeof(ea_summary);
  int32_t* d_rs = (int32_t*)base; base += size_t(n) * sizeof(int32_t);
  int32_t* d_ns = (int32_t*)base;
  CU(cudaMemcpyAsync(d_poses, poses7, size_t(n) * 7 * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(d_rs, ref_slots, size_t(n) * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(d_ns, now_slots, size_t(n) * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemsetAsync(d_sum, 0, size_t(n) * L * sizeof(ea_summary), c->stream));
  rc = ea_solve_batch_device(c, n, ref, d_rs, now, d_ns, d_poses, nullptr, sp, d_sum);
  if (rc) return rc;
  CU(cudaMemcpyAsync(poses7, d_poses, size_t(n) * 7 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  if (summaries) CU(cudaMemcpyAsync(summaries, d_sum, size_t(n) * L * sizeof(ea_summary), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  {   // truncated point lists among the reference slots this call used
    std::vector<int> ovf(size_t(ref->n_slots) * EA_MAX_LEVELS);
    CU(cudaMemcpy(ovf.data(), ref->d_overflow, ovf.size() * sizeof(int), cudaMemcpyDeviceToHost));
    const int lc = sp->coarsest_level < 0 ? L - 1 : sp->coarsest_level;
    for (int i = 0; i < n; ++i)
      for (int l = sp->finest_level; l <= lc; ++l)
        if (ovf[size_t(ref_slots[i]) * EA_MAX_LEVELS + l])
          return ea_fail(EA_ERR_CAPACITY, "pair %d: the reference point list (slot %d, level %d) was truncated at max_points; result uses the truncated list", i, ref_slots[i], l);
  }
  return EA_OK;
}

int ea_solve_traced(ea_context* c, ea_frameset* ref, int ref_slot, ea_frameset* now, int now_slot, double* pose7,
                    const ea_solve_params* sp, ea_summary* summaries, double* trace, int cap, int* n_records) {
  if (!c || !trace || cap <= 0 || !n_records) return ea_fail(EA_ERR_INVALID_ARG, "ea_solve_traced: null argument");
  CU(cudaSetDevice(c->device));
  CU(cudaMalloc((void**)&c->d_trace, size_t(cap) * EA_TRACE_DOUBLES * sizeof(double)));
  CU(cudaMalloc((void**)&c->d_trace_count, sizeof(int)));
  CU(cudaMemsetAsync(c->d_trace_count, 0, sizeof(int), c->stream));
  c->trace_cap = cap;
  const int32_t rs = ref_slot, ns = now_slot;
  int rc = ea_solve_batch(c, 1, ref, &rs, now, &ns, pose7, sp, summaries);
  int n = 0;
  cudaMemcpy(&n, c->d_trace_count, sizeof(int), cudaMemcpyDeviceToHost);
  *n_records = n;
  cudaMemcpy(trace, c->d_trace, size_t(std::min(n, cap)) * EA_TRACE_DOUBLES * sizeof(double), cudaMemcpyDeviceToHost);
  cudaFree(c->d_trace); cudaFree(c->d_trace_count);
  c->d_trace = nullptr; c->d_trace_count = nullptr; c->trace_cap = 0;
  return rc;
}

}  // extern "C"
