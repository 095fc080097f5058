"""Camera and decoder frames read in place: NV12, YUYV, UYVY and pitched GRAY8 / BGR8 (ea_frameset_preprocess_image_*,
ea_tracker_set_image_layout).

The preprocessing only reads luma, so a frame in any of these layouts must give exactly what the gray entry points give on its
dense Y plane: edge and median planes, point lists, truncation flags, distance transforms, poses and summaries, bit for bit.  The
gray path (itself pinned to BGR (g, g, g) by test_gpu_gray.py) is the oracle here.
"""
import ctypes as C
import os
import sys

import numpy as np
import pytest

from conftest import ROOT
from test_gpu_gray import CONFIGS, _summaries_equal, _summary_rows, as_depth, assert_same_frames, make_inputs, to_gray

pytestmark = pytest.mark.gpu

FORMATS = ["GRAY8", "NV12", "YUYV", "UYVY"]


@pytest.fixture(scope="module")
def ea():
    import edge_alignment_b200 as ea
    return ea


@pytest.fixture(scope="module")
def ctx(ea):
    c = ea.Context(0)
    yield c
    c.close()


def embed(ea, gray, fmt, padded, fill=None):
    """gray [n][h][w] as frames of format fmt: (buffer [n][rows][pitch] u8, ImageLayout).  Chroma, padding columns and the rows
    between frames hold `fill` (a uint8 array of the buffer's shape) or 0xFF.  padded: pitch align(row, 256) + 64 and three extra
    rows per frame; else the dense layout, passed as pitch = stride = 0."""
    n, h, w = gray.shape
    packed = fmt in ("YUYV", "UYVY")
    row = 2 * w if packed else w
    pitch = ((row + 255) // 256) * 256 + 64 if padded else row
    rows = (3 * h // 2 if fmt == "NV12" else h) + (3 if padded else 0)
    buf = np.full((n, rows, pitch), 0xFF, np.uint8) if fill is None else fill(n, rows, pitch)
    if packed:
        buf[:, :h, (1 if fmt == "UYVY" else 0):row:2] = gray
    else:
        buf[:, :h, :w] = gray
    code = getattr(ea, "IMAGE_" + fmt)
    return buf, ea.image_layout(code, pitch, rows * pitch) if padded else ea.image_layout(code)


def random_fill(seed):
    rng = np.random.default_rng(seed)
    return lambda n, r, p: rng.integers(0, 256, (n, r, p), dtype=np.uint8)


def fparams(ea, cfg):
    w, h, kw = CONFIGS[cfg]
    return w, h, ea.frame_params(width=w, height=h, fx=525.0 * w / 640, fy=525.0 * w / 640, cx=(w - 1) / 2, cy=(h - 1) / 2, **kw)


def run_image(ea, ctx, fs, entry, slots, buf, layout, depth, roles, ref_mask=None, now_mask=None, base_offset=0):
    """Preprocess buf through the host or the device entry point; base_offset shifts the device image by that many bytes."""
    import torch
    if entry == "host":
        fs.preprocess_image_host(slots, buf, layout, depth, roles, ref_mask=ref_mask, now_mask=now_mask)
        return
    flat = torch.zeros(buf.size + 16, dtype=torch.uint8, device="cuda")
    flat[base_offset:base_offset + buf.size] = torch.from_numpy(buf.reshape(-1)).cuda()
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda() if a is not None else None
    dd, dr, dn = dev(depth), dev(ref_mask), dev(now_mask)
    torch.cuda.synchronize()
    ptr = lambda t: t.data_ptr() if t is not None else 0
    fs.preprocess_image_device(slots, flat.data_ptr() + base_offset, layout, ptr(dd), roles, ptr(dr), ptr(dn))
    ctx.sync()


@pytest.mark.parametrize("padded", [False, True], ids=["dense", "padded"])
@pytest.mark.parametrize("entry", ["host", "device"])
@pytest.mark.parametrize("roles", ["REF", "NOW", "BOTH"])
@pytest.mark.parametrize("cfg", sorted(CONFIGS))
def test_image_preprocess_equals_gray(ea, ctx, frames, cfg, roles, entry, padded):
    w, h, fp = fparams(ea, cfg)
    r = getattr(ea, "ROLE_" + roles)
    gray, d16 = make_inputs(frames, w, h, seed=w + h)
    depth = as_depth(d16, fp.depth_type, ea) if r & ea.ROLE_REF else None
    n = len(gray)
    slots = np.arange(n)[::-1].copy()
    fg = ea.FrameSet(ctx, fp, n + 1)
    try:
        fg.preprocess_gray_host(slots, gray, depth, r)
        for fmt in FORMATS:
            fi = ea.FrameSet(ctx, fp, n + 1)
            try:
                buf, lay = embed(ea, gray, fmt, padded, random_fill(7))
                run_image(ea, ctx, fi, entry, slots, buf, lay, depth, r)
                assert_same_frames(ea, fi, fg, n, r, fp.n_levels)
            finally:
                fi.close()
    finally:
        fg.close()


@pytest.mark.parametrize("cfg", ["lap-640x480-l3-trunc", "lap-322x242-l2-f32", "cannycolor-320x240-l3-exact-f32-z1"])
def test_chroma_and_padding_are_not_read(ea, ctx, frames, cfg):
    """The same luma with chroma, padding and inter-frame rows from a random seed and all 0xFF: identical outputs."""
    w, h, fp = fparams(ea, cfg)
    gray, d16 = make_inputs(frames, w, h, seed=3)
    depth = as_depth(d16, fp.depth_type, ea)
    n = len(gray)
    for fmt in FORMATS:
        for entry in ("host", "device"):
            fa, fb = ea.FrameSet(ctx, fp, n), ea.FrameSet(ctx, fp, n)
            try:
                buf, lay = embed(ea, gray, fmt, True, random_fill(11))
                run_image(ea, ctx, fa, entry, np.arange(n), buf, lay, depth, ea.ROLE_BOTH)
                buf, lay = embed(ea, gray, fmt, True)
                run_image(ea, ctx, fb, entry, np.arange(n), buf, lay, depth, ea.ROLE_BOTH)
                assert_same_frames(ea, fa, fb, n, ea.ROLE_BOTH, fp.n_levels)
            finally:
                fa.close(); fb.close()


@pytest.mark.parametrize("cfg", ["lap-640x480-l3-trunc", "lap-320x240-l1", "cannygray-640x480-l2"])
def test_device_misaligned_images_equal_gray(ea, ctx, frames, cfg):
    """Planar luma at an odd address and with an odd row pitch, packed luma at a 4- but not 8-byte aligned address and with a
    pitch of 4 mod 8: the byte kernels take them, with the aligned results."""
    w, h, fp = fparams(ea, cfg)
    gray, d16 = make_inputs(frames, w, h, seed=9)
    depth = as_depth(d16, fp.depth_type, ea)
    n = len(gray)
    fg = ea.FrameSet(ctx, fp, n)
    try:
        fg.preprocess_gray_host(np.arange(n), gray, depth, ea.ROLE_BOTH)
        cases = []
        for fmt, row in (("GRAY8", w), ("NV12", w)):
            buf, lay = embed(ea, gray, fmt, False)
            cases.append((buf, lay, 1))                                       # odd base
            rows = buf.shape[1]
            odd = np.full((n, rows, row + 1), 0xFF, np.uint8); odd[:, :, :row] = buf
            cases.append((odd, ea.image_layout(lay.format, row + 1, rows * (row + 1)), 0))   # odd pitch
        for fmt in ("YUYV", "UYVY"):
            buf, lay = embed(ea, gray, fmt, False)
            cases.append((buf, lay, 4))                                       # 4-byte aligned base
            wide = np.full((n, h, 2 * w + 4), 0xFF, np.uint8); wide[:, :, :2 * w] = buf
            cases.append((wide, ea.image_layout(lay.format, 2 * w + 4, h * (2 * w + 4)), 0))   # pitch 4 mod 8
        for i, (buf, lay, off) in enumerate(cases):
            fi = ea.FrameSet(ctx, fp, n)
            try:
                run_image(ea, ctx, fi, "device", np.arange(n), buf, lay, depth, ea.ROLE_BOTH, base_offset=off)
                assert_same_frames(ea, fi, fg, n, ea.ROLE_BOTH, fp.n_levels)
            except AssertionError as e:
                raise AssertionError("case %d (format %d, offset %d, pitch %d): %s" % (i, lay.format, off, lay.row_pitch, e))
            finally:
                fi.close()
    finally:
        fg.close()


@pytest.mark.parametrize("cfg", ["lap-640x480-l3-trunc", "lap-322x242-l2-f32", "cannycolor-640x480-l2"])
def test_host_bgr_with_pitch_equals_dense(ea, ctx, frames, cfg):
    """A cv::Mat ROI-style BGR8 view (rows of a wider image, frames of a taller one) on the host path == dense BGR8."""
    from test_gpu_gray import tile_to
    w, h, fp = fparams(ea, cfg)
    bgr = tile_to(frames["bgr"], w, h)
    n = len(bgr)
    depth = as_depth(tile_to(frames["depth"], w, h), fp.depth_type, ea)
    big = np.random.default_rng(5).integers(0, 256, (n, h + 10, w + 20, 3), dtype=np.uint8)
    big[:, 5:5 + h, 7:7 + w] = bgr
    roi = big[:, 5:5 + h, 7:7 + w]
    fa, fb = ea.FrameSet(ctx, fp, n), ea.FrameSet(ctx, fp, n)
    try:
        fa.preprocess_host(np.arange(n), bgr, depth)
        fb.preprocess_image_host(np.arange(n), roi, ea.IMAGE_BGR8, depth)
        assert_same_frames(ea, fb, fa, n, ea.ROLE_BOTH, fp.n_levels)
    finally:
        fa.close(); fb.close()


@pytest.mark.parametrize("entry", ["host", "device"])
def test_image_masks_equal_gray(ea, ctx, frames, entry):
    fp = ea.frame_params(n_levels=3)
    gray, depth = make_inputs(frames, 640, 480, seed=5)
    n = len(gray)
    rng = np.random.default_rng(11)
    yy, xx = np.mgrid[0:480, 0:640]
    ref_mask = np.stack([((xx // (40 + 8 * i) + yy // 50) % 2 * 255).astype(np.uint8) for i in range(n)])
    now_mask = rng.integers(0, 4, (n, 480, 640), dtype=np.uint8)
    slots = np.arange(n)
    fg = ea.FrameSet(ctx, fp, n)
    try:
        for roles, rm, nm in ((ea.ROLE_REF, ref_mask, None), (ea.ROLE_NOW, None, now_mask), (ea.ROLE_BOTH, ref_mask, now_mask)):
            d = depth if roles & ea.ROLE_REF else None
            fg.preprocess_gray_host(slots, gray, d, roles, ref_mask=rm, now_mask=nm)
            for fmt in ("NV12", "YUYV"):
                fi = ea.FrameSet(ctx, fp, n)
                try:
                    buf, lay = embed(ea, gray, fmt, True, random_fill(13))
                    run_image(ea, ctx, fi, entry, slots, buf, lay, d, roles, ref_mask=rm, now_mask=nm)
                    assert_same_frames(ea, fi, fg, n, roles, 3)
                finally:
                    fi.close()
    finally:
        fg.close()


@pytest.mark.parametrize("edge_detector", [0, 2])
def test_image_solves_equal_gray(ea, ctx, frames, edge_detector):
    """solve_batch and solve_views_batch on NV12- and YUYV-preprocessed frame sets == on gray ones, bit for bit."""
    fp = ea.frame_params(n_levels=3, edge_detector=edge_detector, canny_low=150.0, canny_high=100.0, canny_l2=1)
    gray = to_gray(frames["bgr"])
    n = len(gray)
    fg = ea.FrameSet(ctx, fp, n)
    sets = []
    try:
        fg.preprocess_gray_host(np.arange(n), gray, frames["depth"], ea.ROLE_BOTH)
        for fmt, entry in (("NV12", "host"), ("YUYV", "device")):
            fi = ea.FrameSet(ctx, fp, n)
            sets.append(fi)
            buf, lay = embed(ea, gray, fmt, True, random_fill(17))
            run_image(ea, ctx, fi, entry, np.arange(n), buf, lay, frames["depth"], ea.ROLE_BOTH)
        rs, ns = [0, 0, 1, 2, 4, 3], [1, 2, 3, 4, 0, 1]
        T21 = np.eye(4); T21[0, 3] = -0.05
        problems = lambda f: [[dict(ref=f, ref_slot=0, now=f, now_slot=1), dict(ref=f, ref_slot=2, now=f, now_slot=3, T21=T21)],
                              [dict(ref=f, ref_slot=1, now=f, now_slot=2, dist=(0.01, -0.002, 0.0, 0.0, 0.0))],
                              [dict(ref=f, ref_slot=4, now=f, now_slot=3)]]
        for sp in (ea.solve_params(), ea.solve_params(point_stride=1, loss_type=ea.LOSS_HUBER, loss_scale=0.1),
                   ea.solve_params(point_stride=3, trust_region_strategy=ea.STRATEGY_DOGLEG)):
            pg, sg = ctx.solve_batch(fg, rs, fg, ns, None, sp)
            pv, sv = ctx.solve_views_batch(problems(fg), None, sp)
            for fi in sets:
                pi, si = ctx.solve_batch(fi, rs, fi, ns, None, sp)
                np.testing.assert_array_equal(pi, pg)
                _summaries_equal(si, sg)
                pi, si = ctx.solve_views_batch(problems(fi), None, sp)
                np.testing.assert_array_equal(pi, pv)
                _summaries_equal(si, sv)
    finally:
        fg.close()
        for fi in sets:
            fi.close()


def _trajectory(tr):
    w, k, r = tr.trajectory()
    return w.copy(), k.tolist(), r.tolist()


@pytest.mark.parametrize("policy", [False, True], ids=["interval", "keyframe-policy"])
def test_image_tracker_equals_gray(ea, ctx, policy):
    """Over 26 frames: an NV12 tracker (pitch 768, NVDEC-like) and a YUYV tracker give the poses, summaries and (policy mode)
    trajectories and track infos of a GRAY8 tracker on the extracted Y, bit for bit, through step_device and through pipelined
    step_host."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import synth
    S, T, W, H = 6, 26, 640, 480
    bgr, depth, _ = synth.make_sequences(S, T, seed=78, device="cuda")
    b = bgr.to(torch.int64)
    gray = ((b[..., 0] * 9798 + b[..., 1] * 19235 + b[..., 2] * 3735 + 16384) >> 15).to(torch.uint8).contiguous()   # [T][S][H][W]
    del b, bgr
    depth = depth.contiguous()
    # NV12: luma rows 768 bytes apart, chroma plane after it; YUYV dense; chroma bytes random
    g = torch.Generator(device="cuda"); g.manual_seed(3)
    nv12 = torch.randint(0, 256, (T, S, 3 * H // 2, 768), dtype=torch.uint8, device="cuda", generator=g)
    nv12[:, :, :H, :W] = gray
    yuyv = torch.randint(0, 256, (T, S, H, 2 * W), dtype=torch.uint8, device="cuda", generator=g)
    yuyv[..., 0::2] = gray
    torch.cuda.synchronize()
    fp = ea.frame_params(n_levels=3)
    sp = ea.solve_params(point_stride=1, loss_type=ea.LOSS_HUBER, loss_scale=0.1)
    arms = {"gray": (gray, ea.image_layout(ea.IMAGE_GRAY8)),
            "nv12": (nv12, ea.image_layout(ea.IMAGE_NV12, 768, 3 * H // 2 * 768)),
            "yuyv": (yuyv, ea.image_layout(ea.IMAGE_YUYV))}
    trackers = {k: ea.Tracker(ctx, fp, sp, S, 10) for k in arms}
    fd_b = depth[0].numel() * 2
    try:
        for k, tr in trackers.items():
            tr.set_image_layout(arms[k][1])
            if policy:
                tr.set_keyframe_policy(max_interval=8, max_translation=0.02, max_rotation=0.03)
        wants_depth = lambda t: policy or t % 10 == 0
        # device path, stream-ordered inputs
        for t in range(T):
            out = {}
            for k, tr in trackers.items():
                img = arms[k][0]
                tr.step_device(img[t].data_ptr(), depth.data_ptr() + t * fd_b)
                p, Ss = tr.poses()
                out[k] = (p, _summary_rows(Ss), _trajectory(tr) if policy else None)
            for k in ("nv12", "yuyv"):
                np.testing.assert_array_equal(out[k][0], out["gray"][0], err_msg="%s step_device frame %d" % (k, t))
                assert out[k][1] == out["gray"][1], (k, t)
                if policy:
                    np.testing.assert_array_equal(out[k][2][0], out["gray"][2][0])
                    assert out[k][2][1:] == out["gray"][2][1:], (k, t)
        # the layout is fixed once a frame has been stepped; reset opens it again
        for k, tr in trackers.items():
            with pytest.raises(ea.EaError) as e:
                tr.set_image_layout(arms[k][1])
            assert e.value.code == 5
            tr.reset()
            tr.set_image_layout(arms[k][1])
        # host path, pipelined: frame t is submitted before frame t-1's results are read
        host = {k: arms[k][0].cpu().pin_memory() for k in arms}
        hd = depth.cpu().pin_memory()
        res = {k: {} for k in arms}
        for t in range(T):
            for k, tr in trackers.items():
                tr.step_host(host[k][t].data_ptr(), hd.data_ptr() + t * fd_b if wants_depth(t) else 0, fetch=False)
                if t > 0:
                    p, Ss = tr.wait(t - 1)
                    res[k][t - 1] = (p, _summary_rows(Ss), tr.wait_trajectory(t - 1) if policy else None)
        for k, tr in trackers.items():
            p, Ss = tr.wait(T - 1)
            res[k][T - 1] = (p, _summary_rows(Ss), tr.wait_trajectory(T - 1) if policy else None)
        for t in range(T):
            for k in ("nv12", "yuyv"):
                np.testing.assert_array_equal(res[k][t][0], res["gray"][t][0], err_msg="%s step_host frame %d" % (k, t))
                assert res[k][t][1] == res["gray"][t][1], (k, t)
                if policy:
                    for a, bb in zip(res[k][t][2], res["gray"][t][2]):
                        np.testing.assert_array_equal(a, bb)
    finally:
        for tr in trackers.values():
            tr.close()


def test_image_invalid_layouts_launch_nothing(ea, ctx, frames):
    import torch
    from edge_alignment_b200 import _lib as L
    lib = L.lib()
    fs = ea.FrameSet(ctx, ea.frame_params(), 2)
    fs_odd_h = ea.FrameSet(ctx, ea.frame_params(width=640, height=241, cy=120.0), 2)
    fs_odd_w = ea.FrameSet(ctx, ea.frame_params(width=321, height=240, cx=160.0), 2)
    tr = ea.Tracker(ctx, ea.frame_params(), ea.solve_params(), 2, 10)
    gray = np.ascontiguousarray(to_gray(frames["bgr"][:2])); depth = np.ascontiguousarray(frames["depth"][:2])
    big = np.zeros(2 * 480 * 640 * 4, np.uint8)
    dbig = torch.zeros(big.size, dtype=torch.uint8, device="cuda")
    sl = np.ascontiguousarray([0, 1], np.int32).ctypes.data_as(C.POINTER(C.c_int32))
    lay = lambda f, p=0, s=0, r=0: ea.ImageLayout(format=f, reserved=r, row_pitch=p, frame_stride=s)
    host = lambda f, l: lib.ea_frameset_preprocess_image_host(f._h, 2, sl, C.byref(l), big.ctypes.data, depth.ctypes.data, None, None, 3)
    dev = lambda f, l: lib.ea_frameset_preprocess_image_device(f._h, 2, sl, C.byref(l), dbig.data_ptr(), None, None, None, 2)
    bad = [lay(5), lay(-1), lay(ea.IMAGE_NV12, r=1),
           lay(ea.IMAGE_GRAY8, 639), lay(ea.IMAGE_YUYV, 1279), lay(ea.IMAGE_BGR8, 1919), lay(ea.IMAGE_NV12, 639),
           lay(ea.IMAGE_GRAY8, 640, 640 * 479), lay(ea.IMAGE_GRAY8, 768, 768 * 480 + 100),
           lay(ea.IMAGE_YUYV, 1280, 1280 * 480 - 1280), lay(ea.IMAGE_UYVY, 1288, 1288 * 481 + 8)]
    cases = [lambda l=l: host(fs, l) for l in bad] + [lambda l=l: dev(fs, l) for l in bad]
    cases += [
        lambda: host(fs_odd_h, lay(ea.IMAGE_NV12)), lambda: dev(fs_odd_h, lay(ea.IMAGE_NV12)),      # NV12, odd h
        lambda: host(fs_odd_w, lay(ea.IMAGE_YUYV)), lambda: dev(fs_odd_w, lay(ea.IMAGE_UYVY)),      # packed, odd w
        lambda: dev(fs, lay(ea.IMAGE_BGR8, 1920 + 64)),                                             # pitched BGR on the device
        lambda: dev(fs, lay(ea.IMAGE_BGR8, 1920, 1920 * 481)),
        lambda: lib.ea_frameset_preprocess_image_host(fs._h, 2, sl, None, big.ctypes.data, depth.ctypes.data, None, None, 3),
        lambda: lib.ea_frameset_preprocess_image_host(fs._h, 2, sl, C.byref(lay(ea.IMAGE_NV12)), None, depth.ctypes.data, None, None, 3),
        lambda: lib.ea_frameset_preprocess_image_host(fs._h, 2, sl, C.byref(lay(ea.IMAGE_NV12)), big.ctypes.data, None, None, None, 1),
        lambda: lib.ea_frameset_preprocess_image_device(fs._h, 2, sl, C.byref(lay(ea.IMAGE_NV12)), dbig.data_ptr(), None, None, None, 4),
        lambda: lib.ea_tracker_set_image_layout(tr._h, None),
        lambda: lib.ea_tracker_set_image_layout(None, C.byref(lay(ea.IMAGE_NV12))),
    ] + [lambda l=l: lib.ea_tracker_set_image_layout(tr._h, C.byref(l)) for l in bad]
    try:
        torch.cuda.synchronize()
        l0 = ctx.launch_count()
        for i, f in enumerate(cases):
            rc = f()
            assert rc == 1, (i, rc, lib.ea_last_error())          # EA_ERR_INVALID_ARG
        assert ctx.launch_count() == l0
        # a tracker set to pitched BGR8 refuses device frames (its host path copies them)
        assert lib.ea_tracker_set_image_layout(tr._h, C.byref(lay(ea.IMAGE_BGR8, 1920 + 64))) == 0
        assert lib.ea_tracker_step_device(tr._h, dbig.data_ptr(), None) == 1
        assert ctx.launch_count() == l0
        # valid calls afterwards still work
        fs.preprocess_image_host([0, 1], gray, ea.IMAGE_GRAY8, depth)
        assert ctx.launch_count() > l0 and fs.num_points(0) > 0
        tr.set_image_layout(ea.IMAGE_NV12, 768)
    finally:
        tr.close(); fs.close(); fs_odd_h.close(); fs_odd_w.close()
