"""ctypes binding of libea_b200.so (the C ABI of include/ea_cabi.h).

There is no CPU fallback: importing works anywhere (so the symbol table can be checked on a CPU box),
but every compute call needs a CUDA device and the library must have been built
(`python -m edge_alignment_b200.build` or `__graft_entry__.build()`).
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(HERE, "libea_b200.so")

EA_MAX_LEVELS = 4
EA_MAX_VIEWS_PER_PROBLEM = 16
EA_OK = 0
LOSS_TRIVIAL, LOSS_CAUCHY, LOSS_HUBER = 0, 1, 2
STRATEGY_LM, STRATEGY_DOGLEG = 0, 1
NORM_NONE, NORM_01, NORM_255 = 0, 1, 2
ROLE_REF, ROLE_NOW, ROLE_BOTH = 1, 2, 3
EDGE_LAPLACIAN, EDGE_CANNY_GRAY, EDGE_CANNY_COLOR = 0, 1, 2
DT_CHAMFER3, DT_EXACT = 0, 1
DEPTH_U16, DEPTH_F32 = 0, 1
POINTS_PIXEL, POINTS_XYZ = 0, 1
IMAGE_BGR8, IMAGE_GRAY8, IMAGE_NV12, IMAGE_YUYV, IMAGE_UYVY = 0, 1, 2, 3, 4
KEY_FIRST, KEY_INTERVAL, KEY_TRANSLATION, KEY_ROTATION, KEY_COST, KEY_LOST = 1, 2, 4, 8, 16, 32
TERMINATION = {0: "NONE", 1: "CONVERGENCE_GRADIENT", 2: "CONVERGENCE_FUNCTION", 3: "CONVERGENCE_PARAMETER",
               4: "CONVERGENCE_MIN_RADIUS", 5: "NO_CONVERGENCE", 6: "FAILURE_EVAL_X0", 7: "FAILURE_INVALID_STEPS",
               8: "SKIPPED_NO_POINTS", 9: "FAILURE_PEER"}


class FrameParams(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("n_levels", C.c_int32), ("grad_threshold", C.c_int32),
                ("use_median", C.c_int32), ("dt_normalize", C.c_int32), ("max_points", C.c_int32),
                ("depth_type", C.c_int32), ("fx", C.c_double), ("fy", C.c_double), ("cx", C.c_double),
                ("cy", C.c_double), ("depth_scale", C.c_double), ("edge_detector", C.c_int32), ("canny_l2", C.c_int32),
                ("canny_low", C.c_double), ("canny_high", C.c_double), ("dt_kind", C.c_int32), ("zero_depth_to_one", C.c_int32)]


class SolveParams(C.Structure):
    _fields_ = [("point_stride", C.c_int32), ("loss_type", C.c_int32), ("max_num_iterations", C.c_int32),
                ("jacobi_scaling", C.c_int32), ("max_consecutive_invalid_steps", C.c_int32),
                ("cluster_size", C.c_int32), ("coarsest_level", C.c_int32), ("finest_level", C.c_int32),
                ("loss_scale", C.c_double), ("function_tolerance", C.c_double), ("gradient_tolerance", C.c_double),
                ("parameter_tolerance", C.c_double), ("initial_trust_region_radius", C.c_double),
                ("max_trust_region_radius", C.c_double), ("min_trust_region_radius", C.c_double),
                ("min_relative_decrease", C.c_double), ("min_lm_diagonal", C.c_double),
                ("max_lm_diagonal", C.c_double), ("trust_region_strategy", C.c_int32), ("reserved", C.c_int32)]


class Summary(C.Structure):
    _fields_ = [("termination", C.c_int32), ("iterations", C.c_int32), ("accepted", C.c_int32),
                ("rejected", C.c_int32), ("n_residuals", C.c_int32), ("evaluations", C.c_int32),
                ("initial_cost", C.c_double), ("final_cost", C.c_double), ("truncated", C.c_int32), ("reserved", C.c_int32)]

    def asdict(self):
        d = {k: getattr(self, k) for k, _ in self._fields_}
        d["termination_name"] = TERMINATION.get(self.termination, "?")
        return d


class View(C.Structure):
    _fields_ = [("ref", C.c_void_p), ("ref_slot", C.c_int32), ("now", C.c_void_p), ("now_slot", C.c_int32),
                ("use_distortion", C.c_int32), ("use_rig", C.c_int32), ("dist", C.c_double * 5),
                ("cam_T_first", C.c_double * 12), ("first_T_cam", C.c_double * 12)]


class KeyframePolicy(C.Structure):
    _fields_ = [("max_interval", C.c_int32), ("reserved", C.c_int32), ("max_translation", C.c_double),
                ("max_rotation", C.c_double), ("max_cost_per_residual", C.c_double)]


class ImageLayout(C.Structure):
    _fields_ = [("format", C.c_int32), ("reserved", C.c_int32), ("row_pitch", C.c_int64), ("frame_stride", C.c_int64)]


class TrackInfo(C.Structure):
    _fields_ = [("key_frame", C.c_int32), ("key_reasons", C.c_int32)]


# every symbol include/ea_cabi.h declares: name -> (restype, argtypes)
_vp, _i, _pi = C.c_void_p, C.c_int, C.POINTER(C.c_int)
_i32p, _u8p, _u16p, _f32p, _f64p = (C.POINTER(C.c_int32), C.POINTER(C.c_uint8), C.POINTER(C.c_uint16),
                                    C.POINTER(C.c_float), C.POINTER(C.c_double))
PROTOTYPES = {
    "ea_abi_version": (_i, []),
    "ea_last_error": (C.c_char_p, []),
    "ea_create": (_i, [_i, C.POINTER(_vp)]),
    "ea_destroy": (_i, [_vp]),
    "ea_sync": (_i, [_vp]),
    "ea_set_stream": (_i, [_vp, _vp]),
    "ea_device_info": (_i, [_vp, _pi, _pi, _pi]),
    "ea_host_alloc": (_i, [C.POINTER(_vp), C.c_size_t]),
    "ea_host_free": (_i, [_vp]),
    "ea_launch_count": (_i, [_vp, C.POINTER(C.c_int64)]),
    "ea_profile_enable": (_i, [_vp, _i]),
    "ea_profile_read": (_i, [_vp, _f64p, _pi, _f64p, _pi]),
    "ea_frame_params_default": (None, [C.POINTER(FrameParams)]),
    "ea_solve_params_default": (None, [C.POINTER(SolveParams)]),
    "ea_frameset_create": (_i, [_vp, C.POINTER(FrameParams), _i, C.POINTER(_vp)]),
    "ea_frameset_destroy": (_i, [_vp]),
    "ea_frameset_preprocess_host": (_i, [_vp, _i, _i32p, _vp, _vp, _i]),
    "ea_frameset_preprocess_masked": (_i, [_vp, _i, _i32p, _vp, _vp, _vp, _i]),
    "ea_frameset_preprocess_now_masked": (_i, [_vp, _i, _i32p, _vp, _vp]),
    "ea_frameset_preprocess_device": (_i, [_vp, _i, _i32p, _vp, _vp, _i]),
    "ea_frameset_preprocess_gray_host": (_i, [_vp, _i, _i32p, _vp, _vp, _vp, _vp, _i]),
    "ea_frameset_preprocess_gray_device": (_i, [_vp, _i, _i32p, _vp, _vp, _i]),
    "ea_frameset_preprocess_image_host": (_i, [_vp, _i, _i32p, C.POINTER(ImageLayout), _vp, _vp, _vp, _vp, _i]),
    "ea_frameset_preprocess_image_device": (_i, [_vp, _i, _i32p, C.POINTER(ImageLayout), _vp, _vp, _vp, _vp, _i]),
    "ea_frameset_set_points": (_i, [_vp, _i, _i, _f32p, _i, _i]),
    "ea_frameset_set_dt": (_i, [_vp, _i, _i, _f32p]),
    "ea_frameset_get_num_points": (_i, [_vp, _i, _i, _pi]),
    "ea_frameset_get_points": (_i, [_vp, _i, _i, _f32p, _i, _pi]),
    "ea_frameset_get_dt": (_i, [_vp, _i, _i, _f32p]),
    "ea_frameset_get_edge_mask": (_i, [_vp, _i, _i, _i, _u8p]),
    "ea_frameset_level_geometry": (_i, [_vp, _i, _pi, _pi, _f64p]),
    "ea_eval": (_i, [_vp, _vp, _i, _vp, _i, _i, _f64p, C.POINTER(SolveParams), _pi, _f64p, _f64p, _f64p, _f64p, _pi]),
    "ea_solve_batch": (_i, [_vp, _i, _vp, _i32p, _vp, _i32p, _f64p, C.POINTER(SolveParams), C.POINTER(Summary)]),
    "ea_solve_traced": (_i, [_vp, _vp, _i, _vp, _i, _f64p, C.POINTER(SolveParams), C.POINTER(Summary), _f64p, _i, _pi]),
    "ea_solve_batch_device": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, C.POINTER(SolveParams), _vp]),
    "ea_eval_views": (_i, [_vp, _i, C.POINTER(View), _i, _f64p, C.POINTER(SolveParams), _pi, _f64p, _f64p, _f64p, _f64p, _pi]),
    "ea_solve_views": (_i, [_vp, _i, C.POINTER(View), _i, _f64p, C.POINTER(SolveParams), C.POINTER(Summary)]),
    "ea_solve_views_batch": (_i, [_vp, _i, _i32p, C.POINTER(View), _f64p, C.POINTER(SolveParams), C.POINTER(Summary)]),
    "ea_tracker_create": (_i, [_vp, C.POINTER(FrameParams), C.POINTER(SolveParams), _i, _i, C.POINTER(_vp)]),
    "ea_tracker_destroy": (_i, [_vp]),
    "ea_tracker_reset": (_i, [_vp]),
    "ea_tracker_step_host": (_i, [_vp, _vp, _vp, _f64p, C.POINTER(Summary)]),
    "ea_tracker_wait": (_i, [_vp, _i, _f64p, C.POINTER(Summary)]),
    "ea_tracker_step_device": (_i, [_vp, _vp, _vp]),
    "ea_tracker_set_inputs_ready": (_i, [_vp, _i]),
    "ea_tracker_set_image_format": (_i, [_vp, _i]),
    "ea_tracker_set_image_layout": (_i, [_vp, C.POINTER(ImageLayout)]),
    "ea_tracker_probe_gather": (_i, [_vp, _i, _i, C.POINTER(C.c_float), C.POINTER(C.c_double)]),
    "ea_tracker_get_poses": (_i, [_vp, _f64p, C.POINTER(Summary)]),
    "ea_tracker_frame_index": (_i, [_vp, _pi]),
    "ea_tracker_set_keyframe_policy": (_i, [_vp, C.POINTER(KeyframePolicy)]),
    "ea_tracker_get_trajectory": (_i, [_vp, _f64p, C.POINTER(TrackInfo)]),
    "ea_tracker_wait_trajectory": (_i, [_vp, _i, _f64p, C.POINTER(TrackInfo)]),
    "ea_shard_unique_id": (_i, [_u8p]),
    "ea_shard_create": (_i, [_vp, _u8p, _i, _i, C.POINTER(_vp)]),
    "ea_shard_destroy": (_i, [_vp]),
    "ea_shard_solve": (_i, [_vp, _vp, _i, _vp, _i, _i, _f64p, C.POINTER(SolveParams), C.POINTER(Summary)]),
    "ea_shard_profile": (_i, [_vp, _f64p]),
}

_lib = None


def lib():
    """Load libea_b200.so; fail loudly if it has not been built (no fallback path exists)."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise RuntimeError("edge_alignment_b200: %s is missing -- build it with `python -m edge_alignment_b200.build` "
                               "(there is no CPU or PyTorch fallback for this path)" % SO_PATH)
        L = C.CDLL(SO_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib
