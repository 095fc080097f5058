"""8-bit gray input (ea_frameset_preprocess_gray_*, ea_tracker_set_image_format, Frame::set on 8UC1).

A gray frame g is preprocessed exactly as the BGR path preprocesses (g, g, g): OpenCV's 8-bit RGB2GRAY weights sum to 2^15, so
three equal blurred channels convert back to the same value; the 2x2 pyramid mean is per channel; CANNY_COLOR's channel of
largest gradient (first on ties) is the single channel.  The BGR path is therefore an exact oracle for the gray one: masks,
point lists, truncation flags, distance transforms, poses and summaries must all be bit-identical.
"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ea():
    import edge_alignment_b200 as ea
    return ea


@pytest.fixture(scope="module")
def ctx(ea):
    c = ea.Context(0)
    yield c
    c.close()


def to_gray(bgr):
    """OpenCV's 8-bit RGB2GRAY on BGR data, the 15-bit fixed-point formula the kernels use."""
    b = np.asarray(bgr, np.int64)
    return ((b[..., 0] * 9798 + b[..., 1] * 19235 + b[..., 2] * 3735 + 16384) >> 15).astype(np.uint8)


def rep3(gray):
    return np.ascontiguousarray(np.repeat(np.asarray(gray, np.uint8)[..., None], 3, -1))


def tile_to(a, w, h):
    """The bundled 640x480 frames cut or tiled to another geometry."""
    reps = (-(-h // a.shape[1]), -(-w // a.shape[2])) + (1,) * (a.ndim - 3)
    return np.ascontiguousarray(np.tile(a, (1,) + reps)[:, :h, :w])


def make_inputs(frames, w, h, seed):
    """Gray frames and depth at w x h: the bundled frames, a random image, a smooth random image, a constant image and two
    single-edge images."""
    rng = np.random.default_rng(seed)
    g = [to_gray(tile_to(frames["bgr"][:3], w, h))[i] for i in range(3)]
    g.append(rng.integers(0, 256, (h, w), dtype=np.uint8))
    sm = rng.integers(0, 256, (h // 8 + 1, w // 8 + 1)).astype(np.float64)
    g.append(np.kron(sm, np.ones((8, 8)))[:h, :w].astype(np.uint8))
    g.append(np.full((h, w), 97, np.uint8))
    e = np.full((h, w), 30, np.uint8); e[:, w // 3:] = 200; g.append(e)
    e = np.full((h, w), 220, np.uint8); e[h // 2 + 1:, :] = 10; g.append(e)
    gray = np.ascontiguousarray(np.stack(g))
    d16 = tile_to(frames["depth"][:1], w, h)[0]
    depth = np.ascontiguousarray(np.stack([np.roll(d16, 7 * i, axis=1) for i in range(len(g))]))
    return gray, depth


def as_depth(depth_u16, depth_type, ea):
    return (depth_u16.astype(np.float32) / 5000.0) if depth_type == ea.DEPTH_F32 else depth_u16


def points_rc(ea, fs, slot, level):
    """(status, point rows) of a slot's list; status EA_ERR_CAPACITY marks a list truncated at max_points."""
    from edge_alignment_b200 import _lib as L
    w, h, _ = fs.level_geometry(level)
    out = np.zeros((w * h, 4), np.float32); n = C.c_int()
    rc = L.lib().ea_frameset_get_points(fs._h, slot, level, out.ctypes.data_as(C.POINTER(C.c_float)), w * h, C.byref(n))
    assert rc in (0, 4), L.lib().ea_last_error()
    return rc, out[:min(n.value, w * h)].copy()


def assert_same_frames(ea, fa, fb, n, roles, n_levels, use_median=True):
    for s in range(n):
        for l in range(n_levels):
            ctx = "slot %d level %d" % (s, l)
            np.testing.assert_array_equal(fa.edge_mask(s, l), fb.edge_mask(s, l), err_msg=ctx)
            if roles & ea.ROLE_REF:
                ra, pa = points_rc(ea, fa, s, l)
                rb, pb = points_rc(ea, fb, s, l)
                assert ra == rb, ctx
                np.testing.assert_array_equal(pa, pb, err_msg=ctx)
            if roles & ea.ROLE_NOW:
                if use_median:
                    np.testing.assert_array_equal(fa.edge_mask(s, l, median=True), fb.edge_mask(s, l, median=True), err_msg=ctx)
                np.testing.assert_array_equal(fa.dt(s, l), fb.dt(s, l), err_msg=ctx)


# name -> (w, h, frame_params); the geometries cover the fused pyramid (640x480), 64-wide tiles (w % 128 <= 64: 576, 320, 1280
# at level 1), several levels below 8 px of tile width, and a width that is not a multiple of 4 (322: byte kernel, unfused
# pyramid)
CONFIGS = {
    "lap-640x480-l3-trunc": (640, 480, dict(n_levels=3, max_points=2000)),
    "lap-640x480-l4-f32-z1-nomedian": (640, 480, dict(n_levels=4, use_median=0, depth_type=1, zero_depth_to_one=1)),
    "lap-320x240-l1": (320, 240, dict(n_levels=1)),
    "lap-1280x720-l2": (1280, 720, dict(n_levels=2)),
    "lap-576x432-l3-exact": (576, 432, dict(n_levels=3, dt_kind=1)),
    "lap-322x242-l2-f32": (322, 242, dict(n_levels=2, depth_type=1)),
    "cannygray-640x480-l2": (640, 480, dict(n_levels=2, edge_detector=1)),
    "cannygray-322x242-l2-exact": (322, 242, dict(n_levels=2, edge_detector=1, dt_kind=1, canny_l2=1)),
    "cannycolor-320x240-l3-exact-f32-z1": (320, 240, dict(n_levels=3, edge_detector=2, dt_kind=1, canny_low=150.0, canny_high=100.0,
                                                          canny_l2=1, depth_type=1, zero_depth_to_one=1, dt_normalize=2)),
    "cannycolor-640x480-l2": (640, 480, dict(n_levels=2, edge_detector=2)),
}


@pytest.mark.parametrize("entry", ["host", "device"])
@pytest.mark.parametrize("roles", ["REF", "NOW", "BOTH"])
@pytest.mark.parametrize("cfg", sorted(CONFIGS))
def test_gray_preprocess_equals_replicated_bgr(ea, ctx, frames, cfg, roles, entry):
    import torch
    w, h, kw = CONFIGS[cfg]
    fp = ea.frame_params(width=w, height=h, fx=525.0 * w / 640, fy=525.0 * w / 640, cx=(w - 1) / 2, cy=(h - 1) / 2, **kw)
    r = getattr(ea, "ROLE_" + roles)
    gray, d16 = make_inputs(frames, w, h, seed=w + h)
    depth = as_depth(d16, fp.depth_type, ea) if r & ea.ROLE_REF else None
    n = len(gray)
    slots = np.arange(n)[::-1].copy()          # frames land in other slots than their index
    fg, fb = ea.FrameSet(ctx, fp, n + 1), ea.FrameSet(ctx, fp, n + 1)
    try:
        fb.preprocess_host(slots, rep3(gray), depth, r)
        if entry == "host":
            fg.preprocess_gray_host(slots, gray, depth, r)
        else:
            dg = torch.from_numpy(gray).cuda()
            dd = torch.from_numpy(depth).cuda() if depth is not None else None
            torch.cuda.synchronize()
            fg.preprocess_gray_device(slots, dg.data_ptr(), dd.data_ptr() if dd is not None else 0, r)
            ctx.sync()
        assert_same_frames(ea, fg, fb, n, r, fp.n_levels)
    finally:
        fg.close(); fb.close()


def test_gray_masks_equal_replicated_bgr(ea, ctx, frames):
    """ref_mask == ea_frameset_preprocess_masked, now_mask == ea_frameset_preprocess_now_masked, and both in one call."""
    fp = ea.frame_params(n_levels=3)
    gray, depth = make_inputs(frames, 640, 480, seed=5)
    n = len(gray)
    rng = np.random.default_rng(11)
    yy, xx = np.mgrid[0:480, 0:640]
    ref_mask = np.stack([((xx // (40 + 8 * i) + yy // 50) % 2 * 255).astype(np.uint8) for i in range(n)])
    now_mask = rng.integers(0, 4, (n, 480, 640), dtype=np.uint8)       # values 0..3 around the "> 1" threshold
    slots = np.arange(n)
    fg, fb = ea.FrameSet(ctx, fp, n), ea.FrameSet(ctx, fp, n)
    try:
        for roles in (ea.ROLE_REF, ea.ROLE_BOTH):
            fb.preprocess_masked(slots, rep3(gray), depth, ref_mask, roles)
            fg.preprocess_gray_host(slots, gray, depth, roles, ref_mask=ref_mask)
            assert_same_frames(ea, fg, fb, n, roles, 3)
        fb.preprocess_now_masked(slots, rep3(gray), now_mask)
        fg.preprocess_gray_host(slots, gray, None, ea.ROLE_NOW, now_mask=now_mask)
        assert_same_frames(ea, fg, fb, n, ea.ROLE_NOW, 3)
        # both masks at once: the reference points of the ref-masked call, the edges and DT of the now-masked one
        fb.preprocess_masked(slots, rep3(gray), depth, ref_mask, ea.ROLE_BOTH)
        fb.preprocess_now_masked(slots, rep3(gray), now_mask)
        fg.preprocess_gray_host(slots, gray, depth, ea.ROLE_BOTH, ref_mask=ref_mask, now_mask=now_mask)
        assert_same_frames(ea, fg, fb, n, ea.ROLE_BOTH, 3)
    finally:
        fg.close(); fb.close()


def test_gray_device_pointer_not_word_aligned(ea, ctx, frames):
    """A gray image at an odd device address takes the byte kernels and gives the same results."""
    import torch
    fp = ea.frame_params(n_levels=3)
    gray, depth = make_inputs(frames, 640, 480, seed=3)
    n = len(gray)
    buf = torch.zeros(gray.size + 1, dtype=torch.uint8, device="cuda")
    buf[1:] = torch.from_numpy(gray.reshape(-1)).cuda()
    dd = torch.from_numpy(depth).cuda()
    torch.cuda.synchronize()
    fg, fb = ea.FrameSet(ctx, fp, n), ea.FrameSet(ctx, fp, n)
    try:
        fb.preprocess_host(np.arange(n), rep3(gray), depth, ea.ROLE_BOTH)
        fg.preprocess_gray_device(np.arange(n), buf.data_ptr() + 1, dd.data_ptr(), ea.ROLE_BOTH)
        ctx.sync()
        assert_same_frames(ea, fg, fb, n, ea.ROLE_BOTH, 3)
    finally:
        fg.close(); fb.close()


def test_gray_level0_matches_cv2(ea, ctx, frames):
    """Independent of the BGR path: the Laplacian edge mask and the chamfer DT of the bundled frames in gray against cv2
    (distanceTransform with IPP off, DESIGN.md section 2)."""
    cv2 = pytest.importorskip("cv2")
    gray = to_gray(frames["bgr"])
    n = len(gray)
    fs = ea.FrameSet(ctx, ea.frame_params(), n)
    ipp = cv2.ipp.useIPP()
    try:
        cv2.ipp.setUseIPP(False)
        fs.preprocess_gray_host(np.arange(n), gray, frames["depth"], ea.ROLE_BOTH)
        for i in range(n):
            blur = cv2.GaussianBlur(gray[i], (3, 3), 0, 0, borderType=cv2.BORDER_DEFAULT)
            lap8 = cv2.convertScaleAbs(cv2.Laplacian(blur, cv2.CV_16S, ksize=3, scale=1, delta=0, borderType=cv2.BORDER_DEFAULT))
            B = np.where(lap8 > 35, 0, 255).astype(np.uint8)
            np.testing.assert_array_equal(fs.edge_mask(i), B)
            Bf = cv2.medianBlur(B, 3)
            np.testing.assert_array_equal(fs.edge_mask(i, median=True), Bf)
            dt = cv2.normalize(cv2.distanceTransform(Bf, cv2.DIST_L2, 3), None, 0, 1.0, cv2.NORM_MINMAX)
            np.testing.assert_array_equal(fs.dt(i), dt)
            vs, us = np.nonzero((B == 0) & (frames["depth"][i] > 0))
            pts = fs.points(i)
            np.testing.assert_array_equal(pts[:, 0], us.astype(np.float32))
            np.testing.assert_array_equal(pts[:, 1], vs.astype(np.float32))
    finally:
        cv2.ipp.setUseIPP(ipp)
        fs.close()


def _summaries_equal(a, b):
    for x, y in zip(a, b):
        for sx, sy in zip(x, y):
            assert sx == sy, (sx, sy)


@pytest.mark.parametrize("edge_detector", [0, 2])
def test_gray_solves_equal_replicated_bgr(ea, ctx, frames, edge_detector):
    """solve_batch and solve_views_batch on gray-preprocessed frame sets == the same calls on replicated BGR, bit for bit."""
    fp = ea.frame_params(n_levels=3, edge_detector=edge_detector, canny_low=150.0, canny_high=100.0, canny_l2=1)
    gray = to_gray(frames["bgr"])
    n = len(gray)
    fg, fb = ea.FrameSet(ctx, fp, n), ea.FrameSet(ctx, fp, n)
    try:
        fg.preprocess_gray_host(np.arange(n), gray, frames["depth"], ea.ROLE_BOTH)
        fb.preprocess_host(np.arange(n), rep3(gray), frames["depth"], ea.ROLE_BOTH)
        rs, ns = [0, 0, 1, 2, 4, 3], [1, 2, 3, 4, 0, 1]
        for sp in (ea.solve_params(), ea.solve_params(point_stride=1, loss_type=ea.LOSS_HUBER, loss_scale=0.1),
                   ea.solve_params(point_stride=3, trust_region_strategy=ea.STRATEGY_DOGLEG)):
            pg, sg = ctx.solve_batch(fg, rs, fg, ns, None, sp)
            pb, sb = ctx.solve_batch(fb, rs, fb, ns, None, sp)
            np.testing.assert_array_equal(pg, pb)
            _summaries_equal(sg, sb)
        T21 = np.eye(4); T21[0, 3] = -0.05
        problems = lambda f: [[dict(ref=f, ref_slot=0, now=f, now_slot=1), dict(ref=f, ref_slot=2, now=f, now_slot=3, T21=T21)],
                              [dict(ref=f, ref_slot=1, now=f, now_slot=2, dist=(0.01, -0.002, 0.0, 0.0, 0.0))],
                              [dict(ref=f, ref_slot=4, now=f, now_slot=3)]]
        sp = ea.solve_params(point_stride=2, loss_type=ea.LOSS_HUBER, loss_scale=0.1)
        pg, sg = ctx.solve_views_batch(problems(fg), None, sp)
        pb, sb = ctx.solve_views_batch(problems(fb), None, sp)
        np.testing.assert_array_equal(pg, pb)
        _summaries_equal(sg, sb)
    finally:
        fg.close(); fb.close()


def _summary_rows(S):
    return [tuple(getattr(s, k) for k, _ in s._fields_) for s in S]


def test_gray_tracker_equals_replicated_bgr(ea, ctx):
    """Over 26 frames (three key-frame intervals of 10): a gray tracker and a BGR tracker fed the replicated frames give
    bit-identical poses and summaries, through step_host (pipelined) and through step_device."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import synth
    S, T = 6, 26
    bgr, depth, _ = synth.make_sequences(S, T, seed=77, device="cuda")
    b = bgr.to(torch.int64)
    gray = ((b[..., 0] * 9798 + b[..., 1] * 19235 + b[..., 2] * 3735 + 16384) >> 15).to(torch.uint8).contiguous()
    rep = gray.unsqueeze(-1).expand(*gray.shape, 3).contiguous()
    depth = depth.contiguous()
    torch.cuda.synchronize()
    fp = ea.frame_params(n_levels=3)
    sp = ea.solve_params(point_stride=1, loss_type=ea.LOSS_HUBER, loss_scale=0.1)
    tg = ea.Tracker(ctx, fp, sp, S, 10, image_format=ea.IMAGE_GRAY8)
    tb = ea.Tracker(ctx, fp, sp, S, 10)
    fg_b, fb_b, fd_b = gray[0].numel(), rep[0].numel(), depth[0].numel() * 2
    try:
        # device path, stream-ordered inputs
        for t in range(T):
            tg.step_device(gray.data_ptr() + t * fg_b, depth.data_ptr() + t * fd_b)
            tb.step_device(rep.data_ptr() + t * fb_b, depth.data_ptr() + t * fd_b)
            pg, Sg = tg.poses(); pb, Sb = tb.poses()
            np.testing.assert_array_equal(pg, pb, err_msg="step_device frame %d" % t)
            assert _summary_rows(Sg) == _summary_rows(Sb), t
        dev_last = pg.copy()
        # the format is fixed once a frame has been stepped; reset opens it again
        with pytest.raises(ea.EaError) as e:
            tg.set_image_format(ea.IMAGE_BGR8)
        assert e.value.code == 5
        tg.reset(); tb.reset()
        tg.set_image_format(ea.IMAGE_BGR8); tg.set_image_format(ea.IMAGE_GRAY8)
        # host path, pipelined: frame t is submitted before frame t-1's results are read
        hg = gray.cpu().pin_memory(); hb = rep.cpu().pin_memory(); hd = depth.cpu().pin_memory()
        res = {"g": {}, "b": {}}
        for t in range(T):
            for k, tr, buf, fbytes in (("g", tg, hg, fg_b), ("b", tb, hb, fb_b)):
                tr.step_host(buf.data_ptr() + t * fbytes, hd.data_ptr() + t * fd_b if t % 10 == 0 else 0, fetch=False)
                if t > 0:
                    p, Ss = tr.wait(t - 1)
                    res[k][t - 1] = (p, _summary_rows(Ss))
        for k, tr in (("g", tg), ("b", tb)):
            p, Ss = tr.wait(T - 1)
            res[k][T - 1] = (p, _summary_rows(Ss))
        for t in range(T):
            np.testing.assert_array_equal(res["g"][t][0], res["b"][t][0], err_msg="step_host frame %d" % t)
            assert res["g"][t][1] == res["b"][t][1], t
        np.testing.assert_array_equal(res["g"][T - 1][0], dev_last)
    finally:
        tg.close(); tb.close()


def test_gray_invalid_input_launches_nothing(ea, ctx, frames):
    from edge_alignment_b200 import _lib as L
    lib = L.lib()
    fs = ea.FrameSet(ctx, ea.frame_params(), 2)
    tr = ea.Tracker(ctx, ea.frame_params(), ea.solve_params(), 2, 10)
    gray = np.ascontiguousarray(to_gray(frames["bgr"][:2])); depth = np.ascontiguousarray(frames["depth"][:2])
    mask = np.full((2, 480, 640), 255, np.uint8)
    p = lambda a: a.ctypes.data if a is not None else None
    I32 = lambda v: np.ascontiguousarray(v, np.int32)
    sl = lambda a: a.ctypes.data_as(C.POINTER(C.c_int32))
    ok, bad_hi, bad_neg = I32([0, 1]), I32([0, 2]), I32([-1, 0])
    l0 = ctx.launch_count()
    cases = [
        lambda: lib.ea_frameset_preprocess_gray_host(fs._h, 2, sl(ok), None, p(depth), None, None, 3),      # null image
        lambda: lib.ea_frameset_preprocess_gray_host(None, 2, sl(ok), p(gray), p(depth), None, None, 3),    # null frame set
        lambda: lib.ea_frameset_preprocess_gray_host(fs._h, 2, None, p(gray), p(depth), None, None, 3),     # null slots
        lambda: lib.ea_frameset_preprocess_gray_host(fs._h, 2, sl(bad_hi), p(gray), p(depth), None, None, 3),
        lambda: lib.ea_frameset_preprocess_gray_host(fs._h, 2, sl(bad_neg), p(gray), p(depth), None, None, 3),
        lambda: lib.ea_frameset_preprocess_gray_host(fs._h, 3, sl(I32([0, 1, 1])), p(gray), p(depth), None, None, 3),   # n > slots
        lambda: lib.ea_frameset_preprocess_gray_host(fs._h, 0, sl(ok), p(gray), p(depth), None, None, 3),
        lambda: lib.ea_frameset_preprocess_gray_host(fs._h, 2, sl(ok), p(gray), p(depth), None, None, 0),   # bad roles
        lambda: lib.ea_frameset_preprocess_gray_host(fs._h, 2, sl(ok), p(gray), p(depth), None, None, 4),
        lambda: lib.ea_frameset_preprocess_gray_host(fs._h, 2, sl(ok), p(gray), p(depth), None, None, 7),
        lambda: lib.ea_frameset_preprocess_gray_host(fs._h, 2, sl(ok), p(gray), None, None, None, 1),       # REF without depth
        lambda: lib.ea_frameset_preprocess_gray_host(fs._h, 2, sl(ok), p(gray), p(depth), p(mask), None, 2),   # ref mask, NOW only
        lambda: lib.ea_frameset_preprocess_gray_host(fs._h, 2, sl(ok), p(gray), p(depth), None, p(mask), 1),   # now mask, REF only
        lambda: lib.ea_frameset_preprocess_gray_device(fs._h, 2, sl(ok), None, None, 2),
        lambda: lib.ea_frameset_preprocess_gray_device(fs._h, 2, sl(bad_hi), 1 << 20, None, 2),
        lambda: lib.ea_frameset_preprocess_gray_device(fs._h, 2, sl(ok), 1 << 20, None, 0),
        lambda: lib.ea_frameset_preprocess_gray_device(fs._h, 2, sl(ok), 1 << 20, None, 1),
        lambda: lib.ea_tracker_set_image_format(tr._h, 2),
        lambda: lib.ea_tracker_set_image_format(tr._h, -1),
        lambda: lib.ea_tracker_set_image_format(None, 1),
    ]
    try:
        for i, f in enumerate(cases):
            rc = f()
            assert rc == 1, (i, rc)          # EA_ERR_INVALID_ARG
        assert ctx.launch_count() == l0
        # and a valid call after all of them still works
        fs.preprocess_gray_host([0, 1], gray, depth)
        assert ctx.launch_count() > l0 and fs.num_points(0) > 0
    finally:
        tr.close(); fs.close()


def test_cpp_facade_gray_frames(frames, tmp_path):
    """Frame::set / SolveEA on 8UC1 == on the same image as 8UC3; an image of another type throws (tests/cpp/gray_facade_test.cpp)."""
    from edge_alignment_b200 import _lib as L
    exe = str(tmp_path / "gray_facade_test")
    lib_dir = os.path.dirname(L.SO_PATH)
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "gray_facade_test.cpp"), "-o", exe,
                           "-L", lib_dir, "-l:libea_b200.so", "-Wl,-rpath," + lib_dir, "-Wl,-rpath,/usr/local/cuda/lib64"])
    gray = to_gray(frames["bgr"])
    gray[0].tofile(tmp_path / "ref.gray"); frames["depth"][0].tofile(tmp_path / "ref.d16"); gray[2].tofile(tmp_path / "now.gray")
    out = subprocess.run([exe, str(tmp_path / "ref.gray"), str(tmp_path / "ref.d16"), str(tmp_path / "now.gray"), "640", "480"],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    rec = {l.split()[0]: l.split()[1:] for l in out.stdout.strip().splitlines()}
    for l in range(3):
        assert rec["frame%d" % l][0] == "1" and int(rec["frame%d" % l][1]) > 0, rec
    assert rec["solve0"][0] == "1" and rec["solve1"][0] == "1", rec
    assert rec["u16"][0] == "1"
