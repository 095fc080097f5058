"""Thin numpy-facing mirror of the C ABI, used by tests/ and bench.py.

The product boundary is the C ABI (include/ea_cabi.h) and the C++ facade with the reference's class names
(include/edge_alignment/SolveEA.h ...); this module only marshals numpy arrays into those calls.  Names follow
the reference: a *frame* plays the ref role (get_aX, standalone/utils.cpp:201) or the now role
(get_distance_transform, utils.cpp:38); a *pair* is solved for b_T_a (standalone_edge_align.cpp:256-301).
"""
import ctypes as C

import numpy as np

from . import _lib as L

IDENTITY = np.array([1.0, 0, 0, 0, 0, 0, 0])


class EaError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("ea status %d: %s" % (code, msg))
        self.code = code


def _check(rc):
    if rc != L.EA_OK:
        raise EaError(rc, L.lib().ea_last_error().decode("utf-8", "replace"))


def _ptr(a, t):
    return a.ctypes.data_as(C.POINTER(t)) if a is not None else None


def frame_params(**kw):
    p = L.FrameParams()
    L.lib().ea_frame_params_default(C.byref(p))
    for k, v in kw.items():
        if not hasattr(type(p), k):
            raise TypeError('frame_params: unknown field %r' % k)
        setattr(p, k, v)
    return p


def solve_params(**kw):
    p = L.SolveParams()
    L.lib().ea_solve_params_default(C.byref(p))
    for k, v in kw.items():
        if not hasattr(type(p), k):
            raise TypeError('solve_params: unknown field %r' % k)
        setattr(p, k, v)
    return p


def image_layout(fmt, row_pitch=0, frame_stride=0):
    """ea_image_layout: format IMAGE_*, bytes from a row to the next and from a frame to the next (0 = dense)."""
    return L.ImageLayout(format=fmt, reserved=0, row_pitch=row_pitch, frame_stride=frame_stride)


def _image_arg(image, layout):
    """(address, ImageLayout) of an image argument.  image: a numpy array or torch tensor [n][h][...] of u8 whose first two
    strides are the frame stride and the row pitch (bytes within a row dense), or an address (int) with an ImageLayout.
    layout: an ImageLayout as is, or an IMAGE_* format whose row pitch and frame stride are taken from the array."""
    if isinstance(image, int):
        if not isinstance(layout, L.ImageLayout):
            raise TypeError("an image given as an address needs an ImageLayout")
        return image, layout
    if hasattr(image, "data_ptr"):
        addr, shape, strides = image.data_ptr(), tuple(image.shape), [s * image.element_size() for s in image.stride()]
    else:
        addr, shape, strides = image.ctypes.data, image.shape, list(image.strides)
    if isinstance(layout, L.ImageLayout):
        return addr, layout
    inner = 1
    for d in range(len(shape) - 1, 1, -1):
        if strides[d] != inner:
            raise ValueError("the bytes of an image row must be dense (strides %s)" % (strides,))
        inner *= shape[d]
    return addr, image_layout(layout, strides[1], strides[0])


class Context:
    def __init__(self, device=0):
        self._h = C.c_void_p()
        _check(L.lib().ea_create(device, C.byref(self._h)))
        self.device = device

    def close(self):
        if self._h:
            L.lib().ea_destroy(self._h)
            self._h = C.c_void_p()

    def sync(self):
        _check(L.lib().ea_sync(self._h))

    def set_stream(self, cuda_stream_ptr):
        _check(L.lib().ea_set_stream(self._h, C.c_void_p(cuda_stream_ptr)))

    def device_info(self):
        a, b, c = C.c_int(), C.c_int(), C.c_int()
        _check(L.lib().ea_device_info(self._h, C.byref(a), C.byref(b), C.byref(c)))
        return dict(sm_count=a.value, cc=(b.value, c.value))

    def launch_count(self):
        n = C.c_int64()
        _check(L.lib().ea_launch_count(self._h, C.byref(n)))
        return n.value

    def profile_enable(self, on=True):
        _check(L.lib().ea_profile_enable(self._h, 1 if on else 0))

    def profile_read(self):
        a, b = C.c_double(), C.c_double(); na, nb = C.c_int(), C.c_int()
        _check(L.lib().ea_profile_read(self._h, C.byref(a), C.byref(na), C.byref(b), C.byref(nb)))
        return dict(preprocess_ms=a.value, n_preprocess=na.value, solve_ms=b.value, n_solve=nb.value)

    def solve_traced(self, ref, ref_slot, now, now_slot, pose7=None, sp=None, cap=512):
        """One pair with its iteration log: returns (pose7, summaries, trace [n, 6]) -- see ea_solve_traced."""
        sp = sp or solve_params()
        pose = np.array(IDENTITY if pose7 is None else pose7, np.float64).copy()
        S = (L.Summary * ref.params.n_levels)()
        tr = np.zeros((cap, 6)); n = C.c_int()
        _check(L.lib().ea_solve_traced(self._h, ref._h, ref_slot, now._h, now_slot, _ptr(pose, C.c_double), C.byref(sp), S,
                                       _ptr(tr, C.c_double), cap, C.byref(n)))
        return pose, [s.asdict() for s in S], tr[:min(n.value, cap)]

    # ---- evaluation / solve -------------------------------------------------------------------------
    def eval(self, ref, ref_slot, now, now_slot, pose7, sp=None, level=0, want_jac=True):
        sp = sp or solve_params()
        pose7 = np.ascontiguousarray(pose7, np.float64)
        n_pts = ref.num_points(ref_slot, level)
        n = (n_pts + sp.point_stride - 1) // sp.point_stride
        raw = np.empty(n); res = np.empty(n); jac = np.empty((n, 6)) if want_jac else None
        sums = np.empty(28); nres = C.c_int(); failed = C.c_int()
        _check(L.lib().ea_eval(self._h, ref._h, ref_slot, now._h, now_slot, level, _ptr(pose7, C.c_double), C.byref(sp),
                               C.byref(nres), _ptr(raw, C.c_double), _ptr(res, C.c_double), _ptr(jac, C.c_double),
                               _ptr(sums, C.c_double), C.byref(failed)))
        H = np.zeros((6, 6)); k = 7
        for a in range(6):
            for c in range(a, 6):
                H[a, c] = H[c, a] = sums[k]; k += 1
        return dict(raw=raw, residuals=res, J=jac, cost=sums[0], b=sums[1:7].copy(), H=H, sums=sums, failed=failed.value,
                    n_residuals=nres.value)

    def solve_batch(self, ref, ref_slots, now, now_slots, poses7=None, sp=None):
        sp = sp or solve_params()
        rs = np.ascontiguousarray(ref_slots, np.int32); ns = np.ascontiguousarray(now_slots, np.int32)
        n = len(rs)
        poses = np.tile(IDENTITY, (n, 1)) if poses7 is None else np.array(poses7, np.float64).reshape(n, 7).copy()
        nl = ref.params.n_levels
        S = (L.Summary * (n * nl))()
        _check(L.lib().ea_solve_batch(self._h, n, ref._h, _ptr(rs, C.c_int32), now._h, _ptr(ns, C.c_int32),
                                      _ptr(poses, C.c_double), C.byref(sp), S))
        sums = [[S[i * nl + l].asdict() for l in range(nl)] for i in range(n)]
        return poses, sums

    # ---- residual variants / multi-camera problems (standalone/utils.h:101-421) ------------------------------------
    @staticmethod
    def _views(views):
        arr = (L.View * len(views))()
        for i, v in enumerate(views):
            a = arr[i]
            a.ref = v["ref"]._h; a.ref_slot = v["ref_slot"]; a.now = v["now"]._h; a.now_slot = v["now_slot"]
            d = v.get("dist"); T21 = v.get("T21")
            a.use_distortion = 0 if d is None else 1
            a.use_rig = 0 if T21 is None else 1
            for k in range(5):
                a.dist[k] = 0.0 if d is None else float(d[k])
            t21 = np.eye(4) if T21 is None else np.asarray(T21, np.float64)
            t12 = np.linalg.inv(t21)
            for k in range(12):
                a.cam_T_first[k] = float(t21[:3].flat[k]); a.first_T_cam[k] = float(t12[:3].flat[k])
        return arr

    def eval_views(self, views, pose7, sp=None, level=0):
        """views: list of dict(ref, ref_slot, now, now_slot, dist=None (k1,k2,p1,p2,k3), T21=None (4x4 trans_1to2))."""
        sp = sp or solve_params()
        arr = self._views(views)
        pose7 = np.ascontiguousarray(pose7, np.float64)
        n = sum((v["ref"].num_points(v["ref_slot"], level) + sp.point_stride - 1) // sp.point_stride for v in views)
        raw = np.empty(n); res = np.empty(n); jac = np.empty((n, 6)); sums = np.empty(28); nres = C.c_int(); failed = C.c_int()
        _check(L.lib().ea_eval_views(self._h, len(views), arr, level, _ptr(pose7, C.c_double), C.byref(sp), C.byref(nres),
                                     _ptr(raw, C.c_double), _ptr(res, C.c_double), _ptr(jac, C.c_double), _ptr(sums, C.c_double), C.byref(failed)))
        H = np.zeros((6, 6)); k = 7
        for a in range(6):
            for c in range(a, 6):
                H[a, c] = H[c, a] = sums[k]; k += 1
        return dict(raw=raw, residuals=res, J=jac, cost=sums[0], b=sums[1:7].copy(), H=H, sums=sums, failed=failed.value, n_residuals=nres.value)

    def solve_views(self, views, pose7=None, sp=None, level=0):
        sp = sp or solve_params()
        arr = self._views(views)
        pose = np.array(IDENTITY if pose7 is None else pose7, np.float64)
        s = L.Summary()
        _check(L.lib().ea_solve_views(self._h, len(views), arr, level, _ptr(pose, C.c_double), C.byref(sp), C.byref(s)))
        return pose, s.asdict()

    def solve_views_batch(self, problems, poses7=None, sp=None):
        """Many multi-camera problems, each solved coarse to fine in one persistent launch (ea_solve_views_batch).
        problems: list of lists of the view dicts eval_views / solve_views take.  Returns (poses [n, 7], [[summary per level]
        per problem])."""
        sp = sp or solve_params()
        n = len(problems)
        flat = [v for pr in problems for v in pr]
        offsets = np.zeros(n + 1, np.int32)
        offsets[1:] = np.cumsum([len(pr) for pr in problems])
        arr = self._views(flat) if flat else (L.View * 1)()
        poses = np.tile(IDENTITY, (n, 1)) if poses7 is None else np.array(poses7, np.float64).reshape(n, 7).copy()
        nl = flat[0]["ref"].params.n_levels if flat else 1
        S = (L.Summary * max(n * nl, 1))()
        _check(L.lib().ea_solve_views_batch(self._h, n, _ptr(offsets, C.c_int32), arr, _ptr(poses, C.c_double), C.byref(sp), S))
        return poses, [[S[i * nl + l].asdict() for l in range(nl)] for i in range(n)]

    def solve_batch_device(self, n, ref, d_ref_slots, now, d_now_slots, d_poses, sp, d_pose_index=0, d_summaries=0):
        """All pointer arguments are raw device addresses (ints); asynchronous on the context stream."""
        _check(L.lib().ea_solve_batch_device(self._h, n, ref._h, d_ref_slots, now._h, d_now_slots, d_poses,
                                             d_pose_index or None, C.byref(sp), d_summaries or None))


class FrameSet:
    """n_slots device-resident frames (gives the reference's empty `class Frame` its body)."""

    def __init__(self, ctx, params, n_slots):
        self.ctx = ctx
        self.params = params
        self.n_slots = n_slots
        self._h = C.c_void_p()
        _check(L.lib().ea_frameset_create(ctx._h, C.byref(params), n_slots, C.byref(self._h)))

    def close(self):
        if self._h:
            L.lib().ea_frameset_destroy(self._h)
            self._h = C.c_void_p()

    def preprocess_host(self, slots, bgr, depth=None, roles=L.ROLE_BOTH):
        slots = np.ascontiguousarray(slots, np.int32)
        bgr = np.ascontiguousarray(bgr, np.uint8)
        depth = None if depth is None else np.ascontiguousarray(depth, np.float32 if self.params.depth_type == L.DEPTH_F32 else np.uint16)
        assert bgr.size == len(slots) * self.params.width * self.params.height * 3
        _check(L.lib().ea_frameset_preprocess_host(self._h, len(slots), _ptr(slots, C.c_int32), bgr.ctypes.data,
                                                   None if depth is None else depth.ctypes.data, roles))
        self.ctx.sync()   # numpy buffers may be pageable and short-lived

    def preprocess_masked(self, slots, bgr, depth, mask, roles=L.ROLE_BOTH):
        """get_aX_mask (utils.cpp:283-369): reference points only where mask > 0."""
        slots = np.ascontiguousarray(slots, np.int32)
        bgr = np.ascontiguousarray(bgr, np.uint8); mask = np.ascontiguousarray(mask, np.uint8)
        depth = np.ascontiguousarray(depth, np.float32 if self.params.depth_type == L.DEPTH_F32 else np.uint16)
        _check(L.lib().ea_frameset_preprocess_masked(self._h, len(slots), _ptr(slots, C.c_int32), bgr.ctypes.data, depth.ctypes.data,
                                                     mask.ctypes.data, roles))
        self.ctx.sync()

    def preprocess_now_masked(self, slots, bgr, mask):
        """get_distance_transform2_masked[_NoNormalize] (utils.cpp:108-141,166-199): DT of the edges where mask > 1."""
        slots = np.ascontiguousarray(slots, np.int32)
        bgr = np.ascontiguousarray(bgr, np.uint8); mask = np.ascontiguousarray(mask, np.uint8)
        _check(L.lib().ea_frameset_preprocess_now_masked(self._h, len(slots), _ptr(slots, C.c_int32), bgr.ctypes.data, mask.ctypes.data))
        self.ctx.sync()

    def preprocess_device(self, slots, d_bgr, d_depth=0, roles=L.ROLE_BOTH):
        slots = np.ascontiguousarray(slots, np.int32)
        _check(L.lib().ea_frameset_preprocess_device(self._h, len(slots), _ptr(slots, C.c_int32), d_bgr, d_depth or None, roles))

    def preprocess_gray_host(self, slots, gray, depth=None, roles=L.ROLE_BOTH, ref_mask=None, now_mask=None):
        """8-bit gray frames [n][h][w]: the same results as preprocess_host on (g, g, g), from a third of the bytes.
        ref_mask: reference points only where > 0 (get_aX_mask); now_mask: now-frame edges only where > 1."""
        slots = np.ascontiguousarray(slots, np.int32)
        gray = np.ascontiguousarray(gray, np.uint8)
        depth = None if depth is None else np.ascontiguousarray(depth, np.float32 if self.params.depth_type == L.DEPTH_F32 else np.uint16)
        ref_mask = None if ref_mask is None else np.ascontiguousarray(ref_mask, np.uint8)
        now_mask = None if now_mask is None else np.ascontiguousarray(now_mask, np.uint8)
        assert gray.size == len(slots) * self.params.width * self.params.height
        _check(L.lib().ea_frameset_preprocess_gray_host(self._h, len(slots), _ptr(slots, C.c_int32), gray.ctypes.data,
                                                        None if depth is None else depth.ctypes.data,
                                                        None if ref_mask is None else ref_mask.ctypes.data,
                                                        None if now_mask is None else now_mask.ctypes.data, roles))
        self.ctx.sync()   # numpy buffers may be pageable and short-lived

    def preprocess_gray_device(self, slots, d_gray, d_depth=0, roles=L.ROLE_BOTH):
        """d_gray / d_depth: device addresses (ints) of [n][h][w] u8 gray frames and their depth."""
        slots = np.ascontiguousarray(slots, np.int32)
        _check(L.lib().ea_frameset_preprocess_gray_device(self._h, len(slots), _ptr(slots, C.c_int32), d_gray, d_depth or None, roles))

    def _dense(self, a, dtype):
        return None if a is None else np.ascontiguousarray(a, dtype)

    def preprocess_image_host(self, slots, image, layout, depth=None, roles=L.ROLE_BOTH, ref_mask=None, now_mask=None):
        """Host frames in any ea_image_layout (NV12 / YUYV / UYVY, pitched GRAY8 / BGR8): the same results as
        preprocess_gray_host on their luma.  image: see _image_arg (a strided array gives its own pitch and stride).
        depth and the masks are dense [n][h][w]."""
        slots = np.ascontiguousarray(slots, np.int32)
        addr, lay = _image_arg(image, layout)
        depth = self._dense(depth, np.float32 if self.params.depth_type == L.DEPTH_F32 else np.uint16)
        ref_mask, now_mask = self._dense(ref_mask, np.uint8), self._dense(now_mask, np.uint8)
        p = lambda a: None if a is None else a.ctypes.data
        _check(L.lib().ea_frameset_preprocess_image_host(self._h, len(slots), _ptr(slots, C.c_int32), C.byref(lay), addr, p(depth),
                                                         p(ref_mask), p(now_mask), roles))
        self.ctx.sync()   # numpy buffers may be pageable and short-lived

    def preprocess_image_device(self, slots, d_image, layout, d_depth=0, roles=L.ROLE_BOTH, d_ref_mask=0, d_now_mask=0):
        """Device frames in any ea_image_layout, read where they lie.  d_image: a CUDA tensor (see _image_arg) or an address
        with an ImageLayout; d_depth / d_ref_mask / d_now_mask: device addresses (ints) of dense [n][h][w] buffers, or 0."""
        slots = np.ascontiguousarray(slots, np.int32)
        addr, lay = _image_arg(d_image, layout)
        _check(L.lib().ea_frameset_preprocess_image_device(self._h, len(slots), _ptr(slots, C.c_int32), C.byref(lay), addr,
                                                           d_depth or None, d_ref_mask or None, d_now_mask or None, roles))

    def set_points(self, slot, pts4, level=0, mode=L.POINTS_PIXEL):
        pts4 = np.ascontiguousarray(pts4, np.float32).reshape(-1, 4)
        _check(L.lib().ea_frameset_set_points(self._h, slot, level, _ptr(pts4, C.c_float), len(pts4), mode))

    def set_dt(self, slot, dt, level=0):
        dt = np.ascontiguousarray(dt, np.float32)
        w, h, _ = self.level_geometry(level)
        assert dt.shape == (h, w)
        _check(L.lib().ea_frameset_set_dt(self._h, slot, level, _ptr(dt, C.c_float)))

    def num_points(self, slot, level=0):
        n = C.c_int()
        _check(L.lib().ea_frameset_get_num_points(self._h, slot, level, C.byref(n)))
        return n.value

    def points(self, slot, level=0):
        n = self.num_points(slot, level)
        out = np.empty((max(n, 1), 4), np.float32); m = C.c_int()
        _check(L.lib().ea_frameset_get_points(self._h, slot, level, _ptr(out, C.c_float), n, C.byref(m)))
        return out[:n]

    def dt(self, slot, level=0):
        w, h, _ = self.level_geometry(level)
        out = np.empty((h, w), np.float32)
        _check(L.lib().ea_frameset_get_dt(self._h, slot, level, _ptr(out, C.c_float)))
        return out

    def edge_mask(self, slot, level=0, median=False):
        w, h, _ = self.level_geometry(level)
        out = np.empty((h, w), np.uint8)
        _check(L.lib().ea_frameset_get_edge_mask(self._h, slot, level, 1 if median else 0, _ptr(out, C.c_uint8)))
        return out

    def level_geometry(self, level=0):
        w, h = C.c_int(), C.c_int(); k = np.empty(4)
        _check(L.lib().ea_frameset_level_geometry(self._h, level, C.byref(w), C.byref(h), _ptr(k, C.c_double)))
        return w.value, h.value, tuple(k)


class Tracker:
    """n_streams frame-to-keyframe trackers stepped in lock-step (the caller of the path, src/ea.cpp:87-131)."""

    def __init__(self, ctx, fparams, sparams, n_streams, keyframe_interval=10, image_format=L.IMAGE_BGR8):
        self.ctx = ctx; self.n_streams = n_streams; self.n_levels = fparams.n_levels
        self._h = C.c_void_p()
        _check(L.lib().ea_tracker_create(ctx._h, C.byref(fparams), C.byref(sparams), n_streams, keyframe_interval, C.byref(self._h)))
        if image_format != L.IMAGE_BGR8:
            self.set_image_format(image_format)

    def set_image_format(self, image_format):
        """IMAGE_BGR8 ([n_streams][h][w][3]) or IMAGE_GRAY8 ([n_streams][h][w]) for step_host / step_device; only before the
        first step (after creation or reset)."""
        _check(L.lib().ea_tracker_set_image_format(self._h, image_format))

    def set_image_layout(self, fmt, row_pitch=0, frame_stride=0):
        """Frames of step_host / step_device in an ea_image_layout (fmt: IMAGE_*, or an ImageLayout): stream s at
        image + s * frame_stride.  Only before the first step (after creation or reset)."""
        lay = fmt if isinstance(fmt, L.ImageLayout) else image_layout(fmt, row_pitch, frame_stride)
        _check(L.lib().ea_tracker_set_image_layout(self._h, C.byref(lay)))

    def close(self):
        if self._h:
            L.lib().ea_tracker_destroy(self._h)
            self._h = C.c_void_p()

    def reset(self):
        _check(L.lib().ea_tracker_reset(self._h))

    def step_host(self, bgr_ptr, depth_ptr, fetch=True):
        """bgr_ptr/depth_ptr: host addresses (ints) of [n_streams][h][w][3] u8 (IMAGE_BGR8) or [n_streams][h][w] u8
        (IMAGE_GRAY8) / [n_streams][h][w] u16."""
        if fetch:
            poses = np.empty((self.n_streams, 7)); S = (L.Summary * (self.n_streams * self.n_levels))()
            _check(L.lib().ea_tracker_step_host(self._h, bgr_ptr, depth_ptr or None, _ptr(poses, C.c_double), S))
            return poses, S
        _check(L.lib().ea_tracker_step_host(self._h, bgr_ptr, depth_ptr or None, None, None))
        return None

    def wait(self, frame):
        """Results of a frame submitted with step_host(..., fetch=False)."""
        poses = np.empty((self.n_streams, 7)); S = (L.Summary * (self.n_streams * self.n_levels))()
        _check(L.lib().ea_tracker_wait(self._h, frame, _ptr(poses, C.c_double), S))
        return poses, S

    def frame_index(self):
        n = C.c_int()
        _check(L.lib().ea_tracker_frame_index(self._h, C.byref(n)))
        return n.value

    def set_inputs_ready(self, ready=True):
        """Device frames passed to step_device are complete at call time: lets frame t+1's preprocessing overlap frame t's solve."""
        _check(L.lib().ea_tracker_set_inputs_ready(self._h, 1 if ready else 0))

    def probe_gather(self, level=0, repeats=8):
        """Gather-roof probe (measurement only): returns point-gathers per second for the current frames and poses."""
        ms = C.c_float(); n = C.c_double()
        _check(L.lib().ea_tracker_probe_gather(self._h, level, repeats, C.byref(ms), C.byref(n)))
        return n.value / (ms.value * 1e-3), ms.value, n.value

    def step_device(self, d_bgr, d_depth=0):
        """Device addresses of the frames, laid out as for step_host."""
        _check(L.lib().ea_tracker_step_device(self._h, d_bgr, d_depth or None))

    def poses(self, want_summaries=True):
        poses = np.empty((self.n_streams, 7))
        S = (L.Summary * (self.n_streams * self.n_levels))() if want_summaries else None
        _check(L.lib().ea_tracker_get_poses(self._h, _ptr(poses, C.c_double), S))
        return poses, S

    def set_keyframe_policy(self, max_interval=0, max_translation=0.0, max_rotation=0.0, max_cost_per_residual=0.0):
        """Per-stream key frames chosen on the device (ea_tracker_set_keyframe_policy); 0 turns a criterion off.
        set_keyframe_policy(None): the fixed keyframe_interval again.  Only before the first step (after creation or reset)."""
        if max_interval is None:
            _check(L.lib().ea_tracker_set_keyframe_policy(self._h, None))
            return
        p = L.KeyframePolicy(max_interval=max_interval, max_translation=max_translation, max_rotation=max_rotation,
                             max_cost_per_residual=max_cost_per_residual)
        _check(L.lib().ea_tracker_set_keyframe_policy(self._h, C.byref(p)))

    @staticmethod
    def _track(world, info):
        return (world, np.array([i.key_frame for i in info], np.int32), np.array([i.key_reasons for i in info], np.int32))

    def trajectory(self):
        """Latest step in policy mode: (world_T_frame [n_streams, 7], key_frame [n_streams], key_reasons [n_streams])."""
        world = np.empty((self.n_streams, 7)); info = (L.TrackInfo * self.n_streams)()
        _check(L.lib().ea_tracker_get_trajectory(self._h, _ptr(world, C.c_double), info))
        return self._track(world, info)

    def wait_trajectory(self, frame):
        """trajectory() of a frame submitted with step_host(..., fetch=False)."""
        world = np.empty((self.n_streams, 7)); info = (L.TrackInfo * self.n_streams)()
        _check(L.lib().ea_tracker_wait_trajectory(self._h, frame, _ptr(world, C.c_double), info))
        return self._track(world, info)


class Shard:
    """One huge pair solved by all ranks together (BASELINE configs[4]): every rank holds the full distance transform and a
    contiguous slice of the ordered point list; the 29 normal-equation sums are all-reduced inside the solve kernel over
    peer-mapped NVLink memory (ea_shard_*).  id128: the 128-byte NCCL id from Shard.unique_id() on rank 0, passed around by the
    caller (e.g. torch.distributed broadcast); None for world == 1."""

    @staticmethod
    def unique_id():
        buf = (C.c_uint8 * 128)()
        _check(L.lib().ea_shard_unique_id(buf))
        return bytes(buf)

    def __init__(self, ctx, id128=None, rank=0, world=1):
        self.ctx = ctx; self.rank = rank; self.world = world
        self._h = C.c_void_p()
        idbuf = (C.c_uint8 * 128)(*id128) if id128 is not None else None
        _check(L.lib().ea_shard_create(ctx._h, idbuf, rank, world, C.byref(self._h)))

    def close(self):
        if self._h:
            L.lib().ea_shard_destroy(self._h)
            self._h = C.c_void_p()

    def solve(self, ref, ref_slot, now, now_slot, pose7=None, sp=None, level=0):
        pose = np.array(IDENTITY if pose7 is None else pose7, dtype=np.float64)
        s = L.Summary()
        _check(L.lib().ea_shard_solve(self._h, ref._h, ref_slot, now._h, now_slot, level, _ptr(pose, C.c_double),
                                      C.byref(sp if sp is not None else solve_params()), C.byref(s)))
        return pose, s.asdict()

    def profile(self):
        """The last solve: evaluations, device ms, microseconds per evaluation {slice evaluation, grid reduce, cross-rank
        all-reduce, LM step}, in-kernel path?, kernel launches."""
        p = (C.c_double * 8)()
        _check(L.lib().ea_shard_profile(self._h, p))
        return {"evaluations": int(p[0]), "solve_ms": p[1], "eval_us": p[2], "grid_reduce_us": p[3], "allreduce_us": p[4],
                "lm_us": p[5], "in_kernel": bool(p[6]), "launches": int(p[7])}


def pixel_points(uvd):
    """[N,3] integer (u, v, raw depth) -> float4 rows of the EA_POINTS_PIXEL stream."""
    uvd = np.asarray(uvd)
    out = np.ones((len(uvd), 4), np.float32)
    out[:, :3] = uvd
    return out
