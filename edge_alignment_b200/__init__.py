"""edge_alignment_b200 -- B200-native (sm_100a) pose-solve hot path of kuwt/edge_alignment.

Product = hand-written CUDA kernels behind the C ABI of include/ea_cabi.h (csrc/), plus the C++ facade with the
reference's class names (include/edge_alignment/).  This Python package only binds that ABI for tests and bench.
It never imports oracle/ and has no CPU fallback.
"""
from . import _lib  # noqa: F401
from .api import (Context, EaError, FrameSet, Shard, Tracker, frame_params, image_layout, pixel_points, solve_params, IDENTITY)  # noqa: F401
from ._lib import (STRATEGY_DOGLEG, STRATEGY_LM, LOSS_CAUCHY, LOSS_HUBER, LOSS_TRIVIAL, NORM_01, NORM_255, NORM_NONE, POINTS_PIXEL, POINTS_XYZ,  # noqa: F401
                   ROLE_BOTH, ROLE_NOW, ROLE_REF, EDGE_LAPLACIAN, EDGE_CANNY_GRAY, EDGE_CANNY_COLOR, DT_CHAMFER3, DT_EXACT, DEPTH_U16, DEPTH_F32,
                   IMAGE_BGR8, IMAGE_GRAY8, IMAGE_NV12, IMAGE_YUYV, IMAGE_UYVY, ImageLayout, KEY_FIRST, KEY_INTERVAL, KEY_TRANSLATION, KEY_ROTATION, KEY_COST, KEY_LOST)
