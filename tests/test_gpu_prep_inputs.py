"""The BGR preprocessing entry points (ea_frameset_preprocess_{host,device,masked,now_masked}) share one validated path with
the gray ones: the same argument checks, the same launches, and the same results whichever entry point a frame comes in by."""
import ctypes as C

import numpy as np
import pytest

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


@pytest.fixture(scope="module")
def lib():
    from edge_alignment_b200 import _lib as L
    return L.lib()


def _slots(a):
    a = np.ascontiguousarray(a, np.int32)
    return a, a.ctypes.data_as(C.POINTER(C.c_int32))


def test_bgr_invalid_input_launches_nothing(ea, ctx, lib, frames):
    """Every BGR entry point rejects what the gray ones reject, before any launch: null frame set, slots or image, a slot out
    of range, n outside [1, n_slots], roles other than REF / NOW / BOTH, REF without depth, a mask on a role it does not
    apply to, and a null mask where the entry point's mask is required."""
    import torch
    fs = ea.FrameSet(ctx, ea.frame_params(), 2)
    bgr = np.ascontiguousarray(frames["bgr"][:2]); depth = np.ascontiguousarray(frames["depth"][:2])
    mask = np.full((2, 480, 640), 255, np.uint8)
    d_bgr = torch.from_numpy(bgr).cuda(); d_depth = torch.from_numpy(depth.view(np.int16)).cuda()
    torch.cuda.synchronize()
    host = dict(image=bgr.ctypes.data, depth=depth.ctypes.data)
    dev = dict(image=d_bgr.data_ptr(), depth=d_depth.data_ptr())
    ok, p_ok = _slots([0, 1])
    hi, p_hi = _slots([0, 2])
    neg, p_neg = _slots([-1, 0])
    three, p_three = _slots([0, 1, 1])

    def call(entry, h=fs._h, n=2, slots=p_ok, image="x", depth="x", mask_=mask.ctypes.data, roles=ea.ROLE_BOTH):
        buf = dev if entry == "device" else host
        image = buf["image"] if image == "x" else image
        depth = buf["depth"] if depth == "x" else depth
        if entry == "host":
            return lib.ea_frameset_preprocess_host(h, n, slots, image, depth, roles)
        if entry == "device":
            return lib.ea_frameset_preprocess_device(h, n, slots, image, depth, roles)
        if entry == "masked":
            return lib.ea_frameset_preprocess_masked(h, n, slots, image, depth, mask_, roles)
        return lib.ea_frameset_preprocess_now_masked(h, n, slots, image, mask_)

    cases = {}
    for e in ("host", "device", "masked", "now_masked"):
        cases.update({
            (e, "null image"): lambda e=e: call(e, image=None),
            (e, "null frame set"): lambda e=e: call(e, h=None),
            (e, "null slots"): lambda e=e: call(e, slots=None),
            (e, "slot >= n_slots"): lambda e=e: call(e, slots=p_hi),
            (e, "slot < 0"): lambda e=e: call(e, slots=p_neg),
            (e, "n > n_slots"): lambda e=e: call(e, n=3, slots=p_three),
            (e, "n = 0"): lambda e=e: call(e, n=0),
        })
        if e in ("masked", "now_masked"):
            cases[(e, "null mask")] = lambda e=e: call(e, mask_=None)
        if e != "now_masked":
            cases.update({
                (e, "roles 0"): lambda e=e: call(e, roles=0),
                (e, "roles 4"): lambda e=e: call(e, roles=4),
                (e, "roles 7"): lambda e=e: call(e, roles=7),
                (e, "REF without depth"): lambda e=e: call(e, depth=None, roles=ea.ROLE_REF),
            })
    cases[("masked", "reference mask, NOW only")] = lambda: call("masked", roles=ea.ROLE_NOW)
    try:
        l0 = ctx.launch_count()
        rcs = {k: f() for k, f in cases.items()}
        assert all(rc == 1 for rc in rcs.values()), {k: rc for k, rc in rcs.items() if rc != 1}   # EA_ERR_INVALID_ARG
        assert ctx.launch_count() == l0
        # the rejected calls left nothing behind: a valid call through every entry point still works
        for e in ("host", "device", "masked", "now_masked"):
            assert call(e) == 0, (e, lib.ea_last_error())
        ctx.sync()
        assert ctx.launch_count() > l0 and fs.num_points(0) > 0
    finally:
        fs.close()


# launches per call of each entry point on 64x48 frames over 2 levels (Laplacian, chamfer DT, median): below and at the two-lane
# split (8 frames per SM)
LAUNCHES = {
    "host": (6, 12),
    "device": (6, 12),
    "masked": (8, 16),
    "now_masked": (6, 12),
    "gray_host": (10, 20),
    "gray_device": (6, 12),
}


@pytest.mark.parametrize("entry", sorted(LAUNCHES))
def test_launches_per_entry_point(ea, ctx, entry):
    import torch
    w, h = 64, 48
    n_big = 8 * ctx.device_info()["sm_count"]
    fp = ea.frame_params(width=w, height=h, fx=50.0, fy=50.0, cx=w / 2.0, cy=h / 2.0, n_levels=2, max_points=w * h)
    fs = ea.FrameSet(ctx, fp, n_big)
    rng = np.random.default_rng(3)
    got = []
    try:
        for n in (2, n_big):
            bgr = (rng.integers(0, 4, (n, h, w, 3)) * 64).astype(np.uint8)
            gray = np.ascontiguousarray(bgr[..., 1])
            dep = (rng.integers(0, 3, (n, h, w)) * 700).astype(np.uint16)
            mask = np.full((n, h, w), 255, np.uint8)
            slots = np.arange(n)
            d_bgr, d_gray, d_dep = (torch.from_numpy(a).cuda() for a in (bgr, gray, dep.view(np.int16)))
            torch.cuda.synchronize()
            calls = {
                "host": lambda: fs.preprocess_host(slots, bgr, dep, ea.ROLE_BOTH),
                "device": lambda: fs.preprocess_device(slots, d_bgr.data_ptr(), d_dep.data_ptr(), ea.ROLE_BOTH),
                "masked": lambda: fs.preprocess_masked(slots, bgr, dep, mask, ea.ROLE_BOTH),
                "now_masked": lambda: fs.preprocess_now_masked(slots, bgr, mask),
                "gray_host": lambda: fs.preprocess_gray_host(slots, gray, dep, ea.ROLE_BOTH, ref_mask=mask, now_mask=mask),
                "gray_device": lambda: fs.preprocess_gray_device(slots, d_gray.data_ptr(), d_dep.data_ptr(), ea.ROLE_BOTH),
            }
            l0 = ctx.launch_count()
            calls[entry]()
            ctx.sync()
            got.append(ctx.launch_count() - l0)
        assert tuple(got) == LAUNCHES[entry], (entry, got)
    finally:
        fs.close()


def _assert_same(fa, fb, n, roles, ea, n_levels):
    for s in range(n):
        for l in range(n_levels):
            where = "slot %d level %d" % (s, l)
            np.testing.assert_array_equal(fa.edge_mask(s, l), fb.edge_mask(s, l), err_msg=where)
            if roles & ea.ROLE_REF:
                np.testing.assert_array_equal(fa.points(s, l), fb.points(s, l), err_msg=where)
            if roles & ea.ROLE_NOW:
                np.testing.assert_array_equal(fa.edge_mask(s, l, median=True), fb.edge_mask(s, l, median=True), err_msg=where)
                np.testing.assert_array_equal(fa.dt(s, l), fb.dt(s, l), err_msg=where)


@pytest.mark.parametrize("case", ["device_vs_host", "masked_all_255_vs_ref", "now_masked_all_255_vs_now"])
def test_entry_points_agree(ea, ctx, frames, case):
    """The same frames through two entry points give byte-identical edge masks, point lists and distance transforms at every
    level: host and device BGR buffers; a reference mask of 255 everywhere and no mask; a now mask of 255 and no mask."""
    import torch
    fp = ea.frame_params(n_levels=3, max_points=640 * 480)
    bgr, depth = frames["bgr"], frames["depth"]
    n = len(bgr)
    slots = np.arange(n)[::-1].copy()          # frames land in other slots than their index
    ones = np.full((n, 480, 640), 255, np.uint8)
    fa, fb = ea.FrameSet(ctx, fp, n), ea.FrameSet(ctx, fp, n)
    try:
        if case == "device_vs_host":
            roles = ea.ROLE_BOTH
            d_bgr, d_dep = torch.from_numpy(bgr).cuda(), torch.from_numpy(depth.view(np.int16)).cuda()
            torch.cuda.synchronize()
            fa.preprocess_device(slots, d_bgr.data_ptr(), d_dep.data_ptr(), roles)
            ctx.sync()
            fb.preprocess_host(slots, bgr, depth, roles)
        elif case == "masked_all_255_vs_ref":
            roles = ea.ROLE_REF
            fa.preprocess_masked(slots, bgr, depth, ones, roles)
            fb.preprocess_host(slots, bgr, depth, roles)
        else:
            roles = ea.ROLE_NOW
            fa.preprocess_now_masked(slots, bgr, ones)
            fb.preprocess_host(slots, bgr, None, roles)
        _assert_same(fa, fb, n, roles, ea, fp.n_levels)
    finally:
        fa.close(); fb.close()
