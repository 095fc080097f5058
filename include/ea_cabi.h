/* =============================================================================
 * ea_cabi.h -- C ABI of the B200-native edge-alignment pose-solve path.
 *
 * The reference (kuwt/edge_alignment) has no FFI: the path is plain in-process C++
 * (class SolveEA include/SolveEA.h:36-71, free functions standalone/utils.h:18-35,
 * functor standalone/utils.h:38-99) calling Ceres/OpenCV on one CPU thread.  This
 * header is the boundary a maintainer binds instead: every entry point cites the
 * reference interface it replaces.  Plain pointers and sizes only; no C++/torch types.
 * The C++ facade with the reference's own class names (SolveEA / Frame / EAResidue)
 * sits on top of this header: include/edge_alignment/{SolveEA,Frame,EAResidue}.h.
 *
 * Conventions
 *   - every function returns ea_status (0 == EA_OK); ea_last_error() gives the text
 *   - images: BGR u8 interleaved row-major (cv::imread order, standalone_edge_align.cpp:118), or 8-bit gray
 *     row-major through the *_gray_* entry points / ea_tracker_set_image_format, or NV12 / YUYV / UYVY frames with a row
 *     pitch through the *_image_* entry points / ea_tracker_set_image_layout; depth u16 row-major (raw units;
 *     metres = raw / depth_scale, utils.cpp:235)
 *   - pose: 7 doubles {qw,qx,qy,qz,tx,ty,tz} = b_T_a, Eigen/Ceres (w,x,y,z) order
 *     (standalone/PoseManipUtils.cpp:16-27)
 *   - there is NO CPU fallback: every compute entry point needs a CUDA device
 * ============================================================================= */
#ifndef EA_CABI_H_
#define EA_CABI_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EA_ABI_VERSION 2
#define EA_MAX_LEVELS 4

typedef struct ea_context ea_context;   /* one per (host thread, CUDA device, stream) */
typedef struct ea_frameset ea_frameset; /* n_slots device-resident frames of one geometry */
typedef struct ea_tracker ea_tracker;   /* n_streams frame-to-keyframe trackers */
typedef struct ea_shard ea_shard;       /* one point-sharded pair across ranks (NCCL) */

typedef enum ea_status {
  EA_OK = 0,
  EA_ERR_INVALID_ARG = 1,
  EA_ERR_CUDA = 2,
  EA_ERR_NO_DEVICE = 3,
  EA_ERR_CAPACITY = 4, /* more edge points than max_points: list truncated */
  EA_ERR_STATE = 5,    /* e.g. solve before the frames were preprocessed */
  EA_ERR_NCCL = 6
} ea_status;

/* ceres::LossFunction attached per residual block (standalone_edge_align.cpp:272 CauchyLoss(1.),
 * :2604 TrivialLoss, src/SolveEA.cpp:144 HuberLoss(0.1)) */
typedef enum ea_loss { EA_LOSS_TRIVIAL = 0, EA_LOSS_CAUCHY = 1, EA_LOSS_HUBER = 2 } ea_loss;
typedef enum ea_strategy { EA_STRATEGY_LM = 0, EA_STRATEGY_DOGLEG = 1 } ea_strategy;   /* ceres TrustRegionStrategyType */

/* cv::normalize(NORM_MINMAX) target range: utils.cpp:81 [0,1]; src/SolveEA.cpp:109 [0,255];
 * utils.cpp:142-165 none */
typedef enum ea_norm { EA_NORM_NONE = 0, EA_NORM_01 = 1, EA_NORM_255 = 2 } ea_norm;

/* edge detector feeding both roles */
typedef enum ea_edge {
  EA_EDGE_LAPLACIAN = 0,   /* GaussianBlur3 -> gray -> |Laplacian| > grad_threshold (+ median for the DT): utils.cpp:49-75, 214-220 */
  EA_EDGE_CANNY_GRAY = 1,  /* blur 3x3 -> gray -> Canny(low, high): get_distance_transform2 / get_aX_canny, utils.cpp:85-106, 371-462 */
  EA_EDGE_CANNY_COLOR = 2  /* Canny on the BGR image itself: src/SolveEA.cpp:46,102 */
} ea_edge;
typedef enum ea_depth { EA_DEPTH_U16 = 0, EA_DEPTH_F32 = 1 } ea_depth;
typedef enum ea_dt {
  EA_DT_CHAMFER3 = 0,      /* cv::distanceTransform(DIST_L2, 3): utils.cpp:80 */
  EA_DT_EXACT = 1          /* cv::distanceTransform(DIST_L2, DIST_MASK_PRECISE): src/SolveEA.cpp:108 */
} ea_dt;

/* what a frame is preprocessed for */
typedef enum ea_role {
  EA_ROLE_REF = 1, /* edge points with depth   (get_aX, utils.cpp:201-281) */
  EA_ROLE_NOW = 2, /* edge distance transform  (get_distance_transform, utils.cpp:38-83) */
  EA_ROLE_BOTH = 3
} ea_role;

/* layout of the float4 point stream */
typedef enum ea_points_mode {
  EA_POINTS_PIXEL = 0, /* {u, v, raw depth, 1}: lossless; X,Y,Z rebuilt in fp64 in registers */
  EA_POINTS_XYZ = 1    /* {X, Y, Z, 1} metres (fp32): CAD / externally supplied points */
} ea_points_mode;

/* ceres::TerminationType + message, condensed */
typedef enum ea_termination {
  EA_TERM_NONE = 0,
  EA_TERM_CONVERGENCE_GRADIENT = 1,
  EA_TERM_CONVERGENCE_FUNCTION = 2,
  EA_TERM_CONVERGENCE_PARAMETER = 3,
  EA_TERM_CONVERGENCE_MIN_RADIUS = 4,
  EA_TERM_NO_CONVERGENCE = 5,
  EA_TERM_FAILURE_EVAL_X0 = 6, /* functor returned false at x0 (utils.h:70-73) */
  EA_TERM_FAILURE_INVALID_STEPS = 7,
  EA_TERM_SKIPPED_NO_POINTS = 8,
  EA_TERM_FAILURE_PEER = 9      /* point-sharded solve: a peer rank stopped answering the all-reduce; batched solve: the
                                   coarse levels of the pair were never handed over to its finest level */
} ea_termination;

/* Preprocessing configuration: every literal of utils.cpp:38-83,201-281 and
 * standalone_edge_align.cpp:151-161 as a field.  Defaults reproduce edge_align_test1. */
typedef struct ea_frame_params {
  int32_t width, height;
  int32_t n_levels;       /* 1 = reference behaviour; >1 = coarse-to-fine pyramid (extension) */
  int32_t grad_threshold; /* 35: utils.cpp:65,258 */
  int32_t use_median;     /* 1: medianBlur(B,3) utils.cpp:75 */
  int32_t dt_normalize;   /* ea_norm; EA_NORM_01: utils.cpp:81 */
  int32_t max_points;     /* level-0 capacity of the point list; 0 => width*height/4 */
  int32_t depth_type;     /* ea_depth: EA_DEPTH_U16 raw units (/depth_scale = metres, utils.cpp:235) or EA_DEPTH_F32 metres
                           * (src/SolveEA.cpp:27,68) */
  double fx, fy, cx, cy;  /* 525,525,319.5,239.5: standalone_edge_align.cpp:152 */
  double depth_scale;     /* 5000: standalone_edge_align.cpp:160 */
  /* edge detector / distance transform selection (defaults 0 = the standalone test1 pipeline) */
  int32_t edge_detector;  /* ea_edge */
  int32_t canny_l2;       /* L2gradient flag of cv::Canny (src/SolveEA.cpp:46: true) */
  double canny_low, canny_high; /* cv::Canny thresholds as passed (swapped if low > high, like OpenCV) */
  int32_t dt_kind;        /* ea_dt */
  int32_t zero_depth_to_one; /* src/SolveEA.cpp:69: edge pixels without depth are kept at Z = 1 instead of dropped */
} ea_frame_params;

/* Problem assembly + ceres::Solver::Options (standalone_edge_align.cpp:265-286; Ceres defaults). */
typedef struct ea_solve_params {
  int32_t point_stride;       /* 30: standalone_edge_align.cpp:267 */
  int32_t loss_type;          /* ea_loss; Cauchy: standalone_edge_align.cpp:272 */
  int32_t max_num_iterations; /* 50 (per pyramid level) */
  int32_t jacobi_scaling;     /* 1 */
  int32_t max_consecutive_invalid_steps; /* 5 */
  int32_t cluster_size;       /* 1 = one persistent CTA per pair; 2,4,8 = thread-block cluster per pair (DSMEM
                               * reduction); 0 = auto (clusters of 8/4/2 while pairs are fewer than SMs/8, /4, /2;
                               * else one CTA per pair) */
  int32_t coarsest_level;     /* first level solved; -1 => n_levels-1 */
  int32_t finest_level;       /* last level solved; 0 */
  double loss_scale;          /* 1.0 */
  double function_tolerance;  /* 1e-6 */
  double gradient_tolerance;  /* 1e-10 */
  double parameter_tolerance; /* 1e-8 */
  double initial_trust_region_radius; /* 1e4 */
  double max_trust_region_radius;     /* 1e16 */
  double min_trust_region_radius;     /* 1e-32 */
  double min_relative_decrease;       /* 1e-3 */
  double min_lm_diagonal;             /* 1e-6 */
  double max_lm_diagonal;             /* 1e32 */
  int32_t trust_region_strategy;      /* 0 LEVENBERG_MARQUARDT (Ceres default, standalone); 1 DOGLEG, traditional (src/SolveEA.cpp:192) */
  int32_t reserved;
} ea_solve_params;

/* ceres::Solver::Summary, condensed; one per (pair, level) */
typedef struct ea_summary {
  int32_t termination;  /* ea_termination */
  int32_t iterations;   /* LM iterations (incl. rejected / invalid) */
  int32_t accepted, rejected;
  int32_t n_residuals;  /* residual blocks = ceil(N/stride) */
  int32_t evaluations;  /* fused residual+Jacobian passes over the n_residuals points */
  double initial_cost, final_cost;
  int32_t truncated;    /* 1: the reference point list was cut at ea_frame_params.max_points (result uses the cut list) */
  int32_t reserved;
} ea_summary;

/* ---- library / context ------------------------------------------------------ */
int ea_abi_version(void);
const char* ea_last_error(void);
int ea_create(int device, ea_context** out);
int ea_destroy(ea_context* ctx);
int ea_sync(ea_context* ctx);                       /* wait for the context's stream */
int ea_set_stream(ea_context* ctx, void* cuda_stream); /* borrow a cudaStream_t (e.g. torch's) */
int ea_device_info(ea_context* ctx, int* sm_count, int* cc_major, int* cc_minor);
/* pinned host memory for the upload paths (cudaHostAlloc / cudaFreeHost) */
int ea_host_alloc(void** p, size_t bytes);
int ea_host_free(void* p);
/* number of kernel launches issued by this context since creation (bench.py gpu_launches) */
int ea_launch_count(ea_context* ctx, int64_t* n);

/* Optional device-side timing (CUDA events on the context stream around each preprocessing pipeline and each
 * solve launch).  ea_profile_read syncs, returns the totals since the last read and resets them. */
int ea_profile_enable(ea_context* ctx, int on);
int ea_profile_read(ea_context* ctx, double* preprocess_ms, int* n_preprocess, double* solve_ms, int* n_solve);

void ea_frame_params_default(ea_frame_params* p);
void ea_solve_params_default(ea_solve_params* p);

/* ---- frames ------------------------------------------------------------------ */
/* Replaces the per-frame state the reference keeps in SolveEA (include/SolveEA.h:52-64:
 * ref_im/ref_depth/now_im/ref_edge/now_dist_transform/list_edge_ref) and gives the empty
 * class Frame (include/Frame.h:42-46) its body. */
int ea_frameset_create(ea_context* ctx, const ea_frame_params* p, int n_slots, ea_frameset** out);
int ea_frameset_destroy(ea_frameset* fs);

/* get_aX (utils.cpp:201-281) and/or get_distance_transform (utils.cpp:38-83) for n frames.
 * HOST buffers: bgr [n][h][w][3] u8, depth [n][h][w] u16 or f32 per ea_frame_params.depth_type (may be NULL when
 * roles==EA_ROLE_NOW).
 * Asynchronous on the context stream (host buffers should be pinned for true overlap). */
int ea_frameset_preprocess_host(ea_frameset* fs, int n, const int32_t* slots, const uint8_t* bgr,
                                const void* depth, int roles);
/* get_aX_mask (utils.cpp:283-369): as above from HOST buffers, reference points only where mask [n][h][w] u8 is > 0 */
int ea_frameset_preprocess_masked(ea_frameset* fs, int n, const int32_t* slots, const uint8_t* bgr,
                                  const void* depth, const uint8_t* mask, int roles);
/* get_distance_transform2_masked[_NoNormalize] (utils.cpp:108-141,166-199): distance transform of the now-frame edges
 * that lie where mask [n][h][w] u8 is > 1 (the reference's threshold(mask, 1, 1, THRESH_BINARY)); HOST buffers, EA_ROLE_NOW.
 * With edge_detector = EA_EDGE_CANNY_GRAY (30, 90), dt_kind = EA_DT_CHAMFER3 and dt_normalize = EA_NORM_255 / EA_NORM_NONE
 * this is the reference's pair of functions; the mask composes with every other detector / DT choice the same way. */
int ea_frameset_preprocess_now_masked(ea_frameset* fs, int n, const int32_t* slots, const uint8_t* bgr, const uint8_t* mask);
/* same as ea_frameset_preprocess_host, inputs already resident in device memory */
int ea_frameset_preprocess_device(ea_frameset* fs, int n, const int32_t* slots, const uint8_t* d_bgr,
                                  const void* d_depth, int roles);

/* 8-bit gray input (grayscale / IR cameras, the Y plane of YUV frames): a third of the bytes of BGR.  A gray frame g is
 * preprocessed exactly as the BGR entry points preprocess (g, g, g) -- every level, every edge detector, DT kind, mask and
 * depth type -- so points, distance transforms and solves are bit-identical: OpenCV's 8-bit RGB2GRAY weights sum to 2^15
 * (9798 + 19235 + 3735) with half of that as rounding constant, so three equal channels convert back to the same value, the
 * 2x2 pyramid mean is per channel, and CANNY_COLOR's channel of largest gradient is that value itself.
 * HOST buffers: gray [n][h][w] u8; depth as ea_frameset_preprocess_host (may be NULL unless roles include EA_ROLE_REF);
 * ref_mask [n][h][w] u8 or NULL: reference points only where ref_mask > 0 (get_aX_mask, needs EA_ROLE_REF); now_mask
 * [n][h][w] u8 or NULL: now-frame edges only where now_mask > 1 (get_distance_transform2_masked, needs EA_ROLE_NOW).
 * roles: EA_ROLE_REF, EA_ROLE_NOW or EA_ROLE_BOTH.  Asynchronous on the context stream. */
typedef enum ea_image_format {
  EA_IMAGE_BGR8 = 0, EA_IMAGE_GRAY8 = 1,
  EA_IMAGE_NV12 = 2, EA_IMAGE_YUYV = 3, EA_IMAGE_UYVY = 4   /* luma read in place: ea_image_layout below */
} ea_image_format;
int ea_frameset_preprocess_gray_host(ea_frameset* fs, int n, const int32_t* slots, const uint8_t* gray, const void* depth,
                                     const uint8_t* ref_mask, const uint8_t* now_mask, int roles);
/* same, inputs already resident in device memory (d_gray 4-byte aligned for the word-wide kernels; any address works) */
int ea_frameset_preprocess_gray_device(ea_frameset* fs, int n, const int32_t* slots, const uint8_t* d_gray,
                                       const void* d_depth, int roles);

/* Camera and decoder frames read in place: only their luma is preprocessed, and chroma and padding bytes are never read.
 *   EA_IMAGE_NV12  the luma plane comes first, one byte per pixel at row_pitch; whatever follows it is ignored.  I420, YV12
 *                  and NV21 frames are therefore passed as EA_IMAGE_NV12 as they are.
 *   EA_IMAGE_YUYV  packed 4:2:2, bytes Y0 U Y1 V per pixel pair (UVC webcams, RGB-D colour streams); w must be even
 *   EA_IMAGE_UYVY  packed 4:2:2, bytes U Y0 V Y1 per pixel pair; w must be even
 * A frame in one of these formats gives exactly what the *_gray_* entry points give on its dense Y plane (points, truncation
 * flags, edge and median planes, distance transforms, solves).  Caution: a video Y plane (BT.601 or BT.709, often limited
 * range 16-235) is not cv::cvtColor(BGR2GRAY) of the decoded BGR frame.  The results are those of the luma as delivered, and
 * grad_threshold applies to those values: there is no range expansion and no colour conversion. */
typedef struct ea_image_layout {
  int32_t format;        /* ea_image_format or EA_IMAGE_NV12 / _YUYV / _UYVY */
  int32_t reserved;      /* 0 */
  int64_t row_pitch;     /* bytes from a row to the next (NV12: of the luma plane); 0 = dense: w * {3, 1, 1, 2, 2} */
  int64_t frame_stride;  /* bytes from a frame to the next; 0 = dense: h * row_pitch, NV12 3 * h * row_pitch / 2 */
} ea_image_layout;
/* The image of frame i starts at image + i * frame_stride.  EA_ERR_INVALID_ARG (and nothing launched) for an unknown format,
 * reserved != 0, row_pitch < w * bytes per pixel, frame_stride < h * row_pitch or not a multiple of row_pitch, NV12 with odd h,
 * YUYV / UYVY with odd w, and BGR8 with a non-dense layout on the device path.  Depth, ref_mask and now_mask are dense
 * [n][h][w] as for ea_frameset_preprocess_gray_host.  The host path uploads only the bytes the kernels read (the luma rows of
 * NV12, the pixel rows of GRAY8 / BGR8, the 2w-byte rows of YUYV / UYVY), packed dense, in one copy per call.  The device path
 * reads the frames where they lie: word-wide loads need a 4-byte (planar) or 8-byte (packed) aligned image, row_pitch and
 * frame_stride; any other layout takes the byte kernels with the same results. */
int ea_frameset_preprocess_image_host(ea_frameset* fs, int n, const int32_t* slots, const ea_image_layout* layout,
                                      const uint8_t* image, const void* depth, const uint8_t* ref_mask,
                                      const uint8_t* now_mask, int roles);
/* same, every buffer (masks too) already resident in device memory */
int ea_frameset_preprocess_image_device(ea_frameset* fs, int n, const int32_t* slots, const ea_image_layout* layout,
                                        const uint8_t* d_image, const void* d_depth, const uint8_t* d_ref_mask,
                                        const uint8_t* d_now_mask, int roles);

/* Bypass hooks (parity on oracle-made inputs; CAD point sets as in edge_align_test5..8). */
int ea_frameset_set_points(ea_frameset* fs, int slot, int level, const float* pts4, int n, int mode);
int ea_frameset_set_dt(ea_frameset* fs, int slot, int level, const float* dt /* [h_l][w_l] */);
/* Read-back (synchronous) for parity tests. */
int ea_frameset_get_num_points(ea_frameset* fs, int slot, int level, int* n);
int ea_frameset_get_points(ea_frameset* fs, int slot, int level, float* pts4, int cap, int* n);
int ea_frameset_get_dt(ea_frameset* fs, int slot, int level, float* dt);
int ea_frameset_get_edge_mask(ea_frameset* fs, int slot, int level, int which /*0 raw,1 median*/, uint8_t* mask);
int ea_frameset_level_geometry(ea_frameset* fs, int level, int* w, int* h, double k4[4]);

/* ---- evaluation / solve ------------------------------------------------------- */
/* One Ceres-style evaluation at `pose` (EAResidue::operator() utils.h:48-80 + autodiff Jacobian +
 * QuaternionParameterization + loss corrector).  All outputs optional (host pointers):
 * raw[n] plain DT lookups, residuals[n] robustified, jac[n*6] local robustified,
 * sums[28] = {cost, J^T r (6), upper-tri J^T J (21 row-major)}, failed = #points with |z'|<0.01. */
int ea_eval(ea_context* ctx, ea_frameset* ref, int ref_slot, ea_frameset* now, int now_slot, int level,
            const double* pose7, const ea_solve_params* sp, int* n_residuals, double* raw, double* residuals,
            double* jac, double* sums28, int* failed);

/* ceres::Solve for n independent pairs (standalone_edge_align.cpp:256-301, batched).
 * poses7 [n][7] in/out (HOST); summaries [n][n_levels] (HOST, may be NULL).  Synchronous. */
int ea_solve_batch(ea_context* ctx, int n, ea_frameset* ref, const int32_t* ref_slots, ea_frameset* now,
                   const int32_t* now_slots, double* poses7, const ea_solve_params* sp, ea_summary* summaries);
/* One pair with the iteration log Ceres prints under minimizer_progress_to_stdout (standalone_edge_align.cpp:284): one record
 * of 6 doubles per evaluation, in order, over all pyramid levels: {level, iterations done so far at this level, cost of the
 * accepted iterate, cost at the evaluated candidate, trust-region radius after the update, decision (1 accepted, 0 rejected,
 * -1 none: first evaluation of a level or termination)}.  trace [cap][6] (HOST), n_records = evaluations made. */
int ea_solve_traced(ea_context* ctx, ea_frameset* ref, int ref_slot, ea_frameset* now, int now_slot, double* pose7,
                    const ea_solve_params* sp, ea_summary* summaries, double* trace, int cap, int* n_records);
/* Same with DEVICE-resident slot indices / poses / summaries; asynchronous on the context stream.
 * d_pose_index[n] maps pair i to a row of d_poses (in/out) so chained solves need no host round trip. */
int ea_solve_batch_device(ea_context* ctx, int n, ea_frameset* ref, const int32_t* d_ref_slots, ea_frameset* now,
                          const int32_t* d_now_slots, double* d_poses7, const int32_t* d_pose_index,
                          const ea_solve_params* sp, ea_summary* d_summaries);

/* ---- residual variants / multi-camera problems (standalone/utils.h:101-421) ------------------------------------------
 * Every view adds its residual blocks to the same 6-DoF problem, as the reference does with one AddResidualBlock loop per
 * camera (standalone_edge_align.cpp:791-803, 3204-3219):
 *   plain view                      EAResidue             utils.h:38-99
 *   use_distortion                  EAResidueEx           utils.h:101-178  (k1,k2,p1,p2,k3 as the functor takes them)
 *   use_rig                         EAResidueSecondCam    utils.h:180-298  b_T_a_SecCam = cam_T_first * b_T_a * first_T_cam
 *   use_rig + use_distortion        EAResidueSecondCamEx  utils.h:300-421
 * Intrinsics of a view are those of its `now` frameset.  Transforms are 3x4 row-major [R | t]. */
typedef struct ea_view {
  ea_frameset* ref; int32_t ref_slot;
  ea_frameset* now; int32_t now_slot;
  int32_t use_distortion, use_rig;
  double dist[5];         /* k1, k2, p1, p2, k3 */
  double cam_T_first[12]; /* trans_1to2     (standalone_edge_align.cpp: trans_1to2) */
  double first_T_cam[12]; /* trans_1to2_inv */
} ea_view;
int ea_eval_views(ea_context* ctx, int n_views, const ea_view* views, int level, const double* pose7,
                  const ea_solve_params* sp, int* n_residuals, double* raw, double* residuals, double* jac,
                  double* sums28, int* failed);
int ea_solve_views(ea_context* ctx, int n_views, const ea_view* views, int level, double* pose7,
                   const ea_solve_params* sp, ea_summary* summary);
/* n independent multi-camera problems, each solved coarse-to-fine (sp->coarsest_level .. sp->finest_level, as
 * ea_solve_batch).  Problem i is views[view_offsets[i] .. view_offsets[i+1]) (1..EA_MAX_VIEWS_PER_PROBLEM views); at level l its
 * residual blocks are exactly those ea_solve_views(..., level = l) would use.  The pose found at level l starts level l-1.
 * poses7 [n][7] in/out (HOST); summaries [n][L] (HOST, may be NULL), L = n_levels shared by every frameset of the call.
 * One persistent launch: one CTA per problem, largest problem first; cluster_size is ignored.  Point counts are read on the
 * device.  A truncated reference list is solved with the cut list: results are written, then EA_ERR_CAPACITY names the first
 * (problem, view, level).  Synchronous. */
#define EA_MAX_VIEWS_PER_PROBLEM 16
int ea_solve_views_batch(ea_context* ctx, int n_problems, const int32_t* view_offsets /*[n+1]*/, const ea_view* views,
                         double* poses7, const ea_solve_params* sp, ea_summary* summaries);

/* ---- tracker: the caller of the path (src/ea.cpp:87-131 consumer loop, re-stated) ------ */
/* n_streams independent cameras; every step each stream gets one new frame which is aligned
 * to that stream's key frame (warm-started from the previous pose); every keyframe_interval-th
 * frame becomes the new key frame (unless ea_tracker_set_keyframe_policy chose the per-stream rule below). */
int ea_tracker_create(ea_context* ctx, const ea_frame_params* fp, const ea_solve_params* sp, int n_streams,
                      int keyframe_interval, ea_tracker** out);
int ea_tracker_destroy(ea_tracker* tr);
int ea_tracker_reset(ea_tracker* tr);
/* HOST inputs [n_streams][h][w][3] (or [n_streams][h][w], EA_IMAGE_GRAY8) / [n_streams][h][w]; poses7 out [n_streams][7] = keyframe_T_frame
 * (HOST, may be NULL => fetch later with ea_tracker_get_poses); asynchronous unless poses7 given. */
int ea_tracker_step_host(ea_tracker* tr, const uint8_t* bgr, const void* depth, double* poses7,
                         ea_summary* summaries);
/* Pipelined use of ea_tracker_step_host: call it with poses7 == summaries == NULL (asynchronous: the upload of this
 * frame overlaps the alignment of the previous one), then collect frame f's result with ea_tracker_wait(tr, f, ...).
 * Results live in a 2-deep ring: wait for frame f before submitting frame f+2.  The host buffers of a submitted
 * frame must stay valid until its results have been waited for. */
int ea_tracker_wait(ea_tracker* tr, int frame, double* poses7, ea_summary* summaries);
int ea_tracker_step_device(ea_tracker* tr, const uint8_t* d_bgr, const void* d_depth);
/* ea_image_format of the image argument of ea_tracker_step_host / _device: EA_IMAGE_BGR8 (default, [n_streams][h][w][3]) or
 * EA_IMAGE_GRAY8 ([n_streams][h][w] u8; the host path then uploads w*h bytes per stream and frame instead of 3*w*h).  Results
 * are those of BGR frames (g, g, g).  Only before the first step (after ea_tracker_create or ea_tracker_reset), else
 * EA_ERR_STATE. */
int ea_tracker_set_image_format(ea_tracker* tr, int image_format);
/* The general form of ea_tracker_set_image_format: ea_tracker_step_host / _device take the image in this layout (any format of
 * ea_image_layout, with a row pitch and a frame stride), stream s starting at image + s * frame_stride.  Results are those of
 * GRAY8 frames holding the luma.  The same rules as ea_frameset_preprocess_image_*, and the same state rule as
 * ea_tracker_set_image_format (EA_ERR_STATE after the first step until ea_tracker_reset).  BGR8 with a pitch is accepted for
 * ea_tracker_step_host, whose copy packs it dense; ea_tracker_step_device then returns EA_ERR_INVALID_ARG. */
int ea_tracker_set_image_layout(ea_tracker* tr, const ea_image_layout* layout);
/* By default the device buffers passed to ea_tracker_step_device are ordered by the context stream (work enqueued there
 * before the call produces them).  ready != 0 declares instead that they are COMPLETE in memory when the call is made; the
 * tracker then preprocesses frame t+1 on its own stream while frame t is still being aligned (its kernels take over the
 * SMs the persistent solve kernel releases during its tail).  ea_tracker_step_host always overlaps this way. */
int ea_tracker_set_inputs_ready(ea_tracker* t, int ready);
/* Measurement only: the L1/L2-gather roofline of the fused evaluation for the tracker's current frames and poses -- a kernel
 * that streams the level's point lists, projects them and gathers the 16 distance-transform texels per point, and nothing
 * else.  ms = device time of `repeats` sweeps, point_gathers = points x repeats (bench.py: roofline.gather_roof). */
int ea_tracker_probe_gather(ea_tracker* tr, int level, int repeats, float* ms, double* point_gathers);
int ea_tracker_get_poses(ea_tracker* tr, double* poses7, ea_summary* summaries); /* syncs */
int ea_tracker_frame_index(ea_tracker* tr, int* n_frames_seen);

/* Key-frame policy mode (opt-in; the default is the fixed keyframe_interval schedule of ea_tracker_create).  Every stream
 * decides on the device, inside the asynchronous step, when its own key frame changes, and keeps its world trajectory.
 *   poses7 (ea_tracker_get_poses / _wait) keep their meaning: key frame -> frame, X_frame = R X_key + t.
 *   world pose of frame t: frame -> world, X_world = R_w X_frame + t_w; the world is the camera of the stream's frame 0 after
 *   create / reset.  world_T_frame = world_T_key o inverse(pose7), composed in fp64 with a normalised quaternion.
 * Rule: frame 0 is a key frame (EA_KEY_FIRST).  Frame t >= 1 is aligned to its stream's current key frame (warm start: the
 * previous pose, identity after the stream's key frame changed); it then becomes the stream's new key frame if any enabled
 * criterion fires (a threshold of 0 turns its criterion off; comparisons are strict):
 *   EA_KEY_INTERVAL     max_interval > 0 and t - key_frame >= max_interval
 *   EA_KEY_TRANSLATION  |t(pose7)| > max_translation (metres)
 *   EA_KEY_ROTATION     2 atan2(|q_xyz|, |q_w|) > max_rotation (radians)
 *   EA_KEY_COST         at sp.finest_level: n_residuals > 0 and final_cost / n_residuals > max_cost_per_residual
 *   EA_KEY_LOST         always on: sp.finest_level terminated with EA_TERM_FAILURE_EVAL_X0, EA_TERM_FAILURE_INVALID_STEPS or
 *                       EA_TERM_SKIPPED_NO_POINTS.  The pose is not trusted: the translation, rotation and cost criteria are not
 *                       evaluated, the frame's world pose is held at the previous frame's, and the frame becomes the new key
 *                       frame there (the stream re-anchors).
 * Any frame may become a key frame, so every step needs depth (NULL depth: EA_ERR_INVALID_ARG) and every frame after the first
 * is preprocessed for both roles; its point lists are built after the policy kernel, only if it was promoted.  The depth passed to
 * ea_tracker_step_device is therefore read until that frame's alignment has finished (ea_tracker_get_poses / ea_sync order it).  The host path uploads depth on every step: for 640x480 GRAY8 frames with u16 depth the upload
 * per stream and frame grows from about 0.37 MB (depth on every 10th frame) to about 0.92 MB (arithmetic from the sizes). */
typedef struct ea_keyframe_policy {
  int32_t max_interval;            /* frames since the key frame; 0 = no limit */
  int32_t reserved;
  double max_translation;          /* metres, 0 = off */
  double max_rotation;             /* radians, 0 = off */
  double max_cost_per_residual;    /* final_cost / n_residuals at the finest solved level, 0 = off */
} ea_keyframe_policy;
enum { EA_KEY_FIRST = 1, EA_KEY_INTERVAL = 2, EA_KEY_TRANSLATION = 4, EA_KEY_ROTATION = 8, EA_KEY_COST = 16, EA_KEY_LOST = 32 };
typedef struct ea_track_info {
  int32_t key_frame;   /* frame index of the key frame this frame was aligned to (frame 0: 0) */
  int32_t key_reasons; /* EA_KEY_* bits that made this frame a key frame; 0 = not one */
} ea_track_info;
/* p == NULL: the fixed interval again.  Only before the first step (after create / reset), else EA_ERR_STATE.  Negative or
 * non-finite thresholds and a negative max_interval: EA_ERR_INVALID_ARG.  ea_tracker_reset keeps the policy. */
int ea_tracker_set_keyframe_policy(ea_tracker* tr, const ea_keyframe_policy* p);
/* world7 [n_streams][7] and info [n_streams] of the latest step (HOST, either may be NULL); syncs.  EA_ERR_STATE outside
 * policy mode. */
int ea_tracker_get_trajectory(ea_tracker* tr, double* world7, ea_track_info* info);
/* the same for frame `frame` submitted with ea_tracker_step_host(..., NULL, NULL): the 2-deep ring of ea_tracker_wait */
int ea_tracker_wait_trajectory(ea_tracker* tr, int frame, double* world7, ea_track_info* info);

/* ---- point-sharded single pair across ranks: one persistent cooperative kernel per rank, the 29 normal-equation sums
 * all-reduced inside the kernel through peer-mapped NVLink memory (NCCL only bootstraps the exchange of the cudaIpc
 * handles; EA_SHARD_MODE=nccl or devices without peer access fall back to launches + ncclAllReduce per evaluation) ---- */
int ea_shard_unique_id(uint8_t id128[128]);
int ea_shard_create(ea_context* ctx, const uint8_t id128[128], int rank, int world, ea_shard** out);
int ea_shard_destroy(ea_shard* sh);
/* every rank holds the full now-frame DT and its contiguous slice of the reference points
 * (slot's point list is sliced [rank*n/world, (rank+1)*n/world)); pose7 in/out identical on all ranks */
int ea_shard_solve(ea_shard* sh, ea_frameset* ref, int ref_slot, ea_frameset* now, int now_slot, int level,
                   double* pose7, const ea_solve_params* sp, ea_summary* summary);
/* Measurement: the last solve of this shard.  out[0] evaluations, out[1] device ms of the whole solve, out[2..5] microseconds
 * per evaluation in {slice evaluation, grid reduce, cross-rank all-reduce, LM step}, out[6] 1 = persistent in-kernel path,
 * out[7] kernel launches */
int ea_shard_profile(ea_shard* sh, double out[8]);

#ifdef __cplusplus
}
#endif
#endif /* EA_CABI_H_ */
