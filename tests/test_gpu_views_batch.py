"""ea_solve_views_batch: many multi-camera problems, each solved coarse to fine in one persistent launch (k_views_batch).

Every problem is checked against the fp64 oracle level by level (oracle.solve_views chained from the coarsest level, with the
bounds of test_gpu_shard_views: pose 1e-4, costs 1e-5 relative, iterations +-2, same termination, same rejected steps for
dogleg), against ea_solve_views and ea_solve_batch on single levels, for bit-for-bit independence from the batch around it, and
against the ground truth of synthetic stereo rigs.  The last test runs without a GPU: the spill guard of the new kernel.
"""
import ctypes as C
import os
import re
import shutil
import subprocess
import sys
import tempfile

import numpy as np
import pytest

from conftest import IDENTITY, ROOT, rot_angle_between

LM, DOGLEG = 0, 1
LOSSES = {"trivial": (0, 1.0), "cauchy": (1, 1.0), "huber": (2, 0.1)}
R_FLOOR = 0.05
ANG = 0.05
T21 = np.eye(4)
T21[:3, :3] = [[np.cos(ANG), 0, np.sin(ANG)], [0, 1, 0], [-np.sin(ANG), 0, np.cos(ANG)]]
T21[:3, 3] = [-0.1, 0.01, 0.02]
DIST = (0.1, -0.2, 0.001, -0.002, 0.05)
N_BIG = 100_003
START = np.array([0.99995, 0.006, -0.004, 0.005, 0.01, -0.01, 0.02])
START[:4] /= np.linalg.norm(START[:4])


# ------------------------------------------------------------------------------------------------------------ fixtures
@pytest.fixture(scope="module")
def ea():
    import edge_alignment_b200 as ea
    return ea


@pytest.fixture(scope="module")
def ctx(ea):
    c = ea.Context(0)
    yield c
    c.close()


def _halve(O, bgr, depth, times):
    for _ in range(times):
        bgr, depth = O.half_linear(bgr), O.half_nearest(depth)
    return bgr, depth


def _backproject(uvd, K, depth_scale=5000.0):
    z = uvd[:, 2] / depth_scale
    return np.stack([(uvd[:, 0] - K[2]) * z / K[0], (uvd[:, 1] - K[3]) * z / K[1], z], 1)


def _xyz4(xyz):
    p4 = np.ones((len(xyz), 4), np.float32)
    p4[:, :3] = xyz
    return p4


@pytest.fixture(scope="module")
def views_data(ea, ctx, frames, oracle):
    """Framesets and oracle inputs of the view layouts, levels 0 and 1 of 2-level framesets.
      A (640 x 480): 0/1 = frames 0 -> 2, 2/3 = frames 3 -> 1, 4 = fp32 XYZ points of frame 0, 5 = no points, 6 = five points
      H (320 x 240, halved K): 0/1 = half-size frames 3 -> 1 (a second frameset of another size)
      B (1280 x 960, the frames' K): 0 = frame 0's points tiled to N_BIG (the capacity of A's level 1 is 320 x 240)"""
    O = oracle
    K = frames["K"]
    A = ea.FrameSet(ctx, ea.frame_params(n_levels=2, max_points=640 * 480), 7)
    A.preprocess_host([0, 1, 2, 3], frames["bgr"][[0, 2, 3, 1]], frames["depth"][[0, 2, 3, 1]], ea.ROLE_BOTH)
    hK = (K[0] / 2, K[1] / 2, (K[2] + 0.5) / 2 - 0.5, (K[3] + 0.5) / 2 - 0.5)
    H = ea.FrameSet(ctx, ea.frame_params(width=320, height=240, fx=hK[0], fy=hK[1], cx=hK[2], cy=hK[3], n_levels=2,
                                         max_points=320 * 240), 2)
    H.preprocess_host([0, 1], np.stack([O.half_linear(frames["bgr"][i]) for i in (3, 1)]),
                      np.stack([O.half_nearest(frames["depth"][i]) for i in (3, 1)]), ea.ROLE_BOTH)
    B = ea.FrameSet(ctx, ea.frame_params(width=1280, height=960, fx=K[0], fy=K[1], cx=K[2], cy=K[3], n_levels=2,
                                         max_points=1280 * 960), 1)
    ov = {}     # (view name, level) -> oracle view without the stride
    for l in range(2):
        KA, KH, KB = A.level_geometry(l)[2], H.level_geometry(l)[2], B.level_geometry(l)[2]
        src = {i: _halve(O, frames["bgr"][i], frames["depth"][i], l) for i in range(4)}
        dts = {i: O.get_distance_transform(src[i][0])[0] for i in (1, 2)}
        xyz0, uvd0 = O.get_aX(src[0][0], src[0][1], KA)
        xyz3, _ = O.get_aX(src[3][0], src[3][1], KA)
        hs = {i: _halve(O, frames["bgr"][i], frames["depth"][i], l + 1) for i in (1, 3)}
        ov["plain", l] = dict(xyz=xyz0, dt=dts[2], K=KA)
        ov["rig_dist", l] = dict(xyz=xyz3, dt=dts[1], K=KA, T21=T21, dist=DIST)
        ov["half", l] = dict(xyz=O.get_aX(hs[3][0], hs[3][1], KH)[0], dt=O.get_distance_transform(hs[1][0])[0], K=KH)
        p4 = _xyz4(xyz0)
        A.set_points(4, p4, level=l, mode=ea.POINTS_XYZ)
        ov["xyz", l] = dict(xyz=p4[:, :3].astype(np.float64), dt=dts[2], K=KA)
        A.set_points(5, np.zeros((0, 4), np.float32), level=l)
        ov["zero", l] = dict(xyz=np.zeros((0, 3)), dt=dts[2], K=KA)
        A.set_points(6, ea.pixel_points(uvd0[:5]), level=l)
        ov["tiny", l] = dict(xyz=xyz0[:5], dt=dts[2], K=KA)
        idx = np.arange(N_BIG) % len(uvd0)
        B.set_points(0, ea.pixel_points(uvd0[idx]), level=l)
        ov["big", l] = dict(xyz=_backproject(uvd0[idx].astype(np.float64), KB), dt=dts[2], K=KA)
    gv = {"plain": dict(ref=A, ref_slot=0, now=A, now_slot=1), "rig_dist": dict(ref=A, ref_slot=2, now=A, now_slot=3, T21=T21, dist=DIST),
          "half": dict(ref=H, ref_slot=0, now=H, now_slot=1), "xyz": dict(ref=A, ref_slot=4, now=A, now_slot=1),
          "zero": dict(ref=A, ref_slot=5, now=A, now_slot=1), "tiny": dict(ref=A, ref_slot=6, now=A, now_slot=1),
          "big": dict(ref=B, ref_slot=0, now=A, now_slot=1)}
    yield gv, ov
    A.close(); H.close(); B.close()


# the problems of a parity batch: an empty view between others, 5 points beside 1e5, one rig + distortion view alone, and a
# view of the 320 x 240 frameset with an XYZ view
PROBLEMS = [["plain", "rig_dist", "zero", "half", "xyz"], ["plain", "tiny", "big", "rig_dist"], ["rig_dist"], ["half", "xyz"]]


def _options(O, loss, strategy=LM, radius=1e4, max_it=50):
    t, s = LOSSES[loss]
    return O.default_options(loss_type=t, loss_scale=s, strategy=strategy, initial_radius=radius, max_num_iterations=max_it)


def _params(ea, loss, stride, strategy=LM, radius=1e4, max_it=50, **kw):
    t, s = LOSSES[loss]
    return ea.solve_params(point_stride=stride, loss_type=t, loss_scale=s, trust_region_strategy=strategy,
                           initial_trust_region_radius=radius, max_num_iterations=max_it, **kw)


def _assert_pose_close(a, b, tol):
    assert rot_angle_between(a[:4], b[:4]) < tol, "rotation off by %g rad" % rot_angle_between(a[:4], b[:4])
    assert np.abs(a[4:] - b[4:]).max() < tol, "translation off by %g m" % np.abs(a[4:] - b[4:]).max()


def _assert_matches_oracle(pose, s, op, os_, dogleg):
    _assert_pose_close(pose, op, 1e-4)
    assert s["n_residuals"] == os_["n_residuals"]
    assert s["termination"] == os_["termination"], (s["termination_name"], os_["termination_name"])
    assert abs(s["iterations"] - os_["iterations"]) <= 2, (s["iterations"], os_["iterations"])
    assert abs(s["final_cost"] - os_["final_cost"]) <= 1e-5 * os_["final_cost"]
    assert abs(s["initial_cost"] - os_["initial_cost"]) <= 1e-5 * os_["initial_cost"]
    if dogleg:
        assert s["rejected"] == os_["rejected"], (s["rejected"], os_["rejected"])


def _assert_own_costs(s, cost_at_start, cost_at_pose):
    """initial_cost / final_cost are the kernel's own evaluations at the start and at the returned pose (test_gpu_shard_views:
    2e-6 relative, plus the suite's residual floor per residual for costs driven to zero)."""
    atol = s["n_residuals"] * 0.5 * (1e-5 * R_FLOOR) ** 2
    np.testing.assert_allclose(s["initial_cost"], cost_at_start, rtol=2e-6, atol=atol, err_msg="initial_cost")
    np.testing.assert_allclose(s["final_cost"], cost_at_pose, rtol=2e-6, atol=atol, err_msg="final_cost")


def _oracle_views(views_data, names, stride, level):
    return [dict(views_data[1][v, level], stride=stride) for v in names]


def _gpu_views(views_data, names):
    return [views_data[0][v] for v in names]


# ------------------------------------------------------------------------------ 1. coarse to fine against the chained oracle
# (strategy, loss, stride, start)
CASES = [(LM, "trivial", 1, "identity"), (DOGLEG, "huber", 7, "xpert"), (LM, "huber", 7, "identity"), (DOGLEG, "trivial", 1, "xpert")]


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=["%s-%s-s%d-%s" % ("lm" if c[0] == LM else "dl", c[1], c[2], c[3]) for c in CASES])
def test_views_batch_matches_chained_oracle(ea, ctx, oracle, numpy_pins, views_data, case):
    O = oracle
    strategy, loss, stride, start = case
    start7 = IDENTITY if start == "identity" else numpy_pins["xpert"]
    max_it = 200 if strategy == DOGLEG else 50
    radius = 1e-2 if strategy == DOGLEG else 1e4
    opts = _options(O, loss, strategy, radius, max_it)
    sp = _params(ea, loss, stride, strategy, radius, max_it)
    poses, S = ctx.solve_views_batch([_gpu_views(views_data, p) for p in PROBLEMS], [start7] * len(PROBLEMS), sp)
    for i, names in enumerate(PROBLEMS):
        op = np.array(start7, np.float64)
        for level in (1, 0):
            ov = _oracle_views(views_data, names, stride, level)
            op, os_ = O.solve_views(ov, op, opts)
            s = S[i][level]
            assert s["n_residuals"] == sum((len(v["xyz"]) + stride - 1) // stride for v in ov)
            assert s["truncated"] == 0 and s["reserved"] == 0
            if level == 1:   # the level's pose is only observable as the next level's start: its initial cost
                for k in ("initial_cost", "final_cost"):
                    assert abs(s[k] - os_[k]) <= 1e-5 * os_[k], (i, level, k, s[k], os_[k])
                assert s["termination"] == os_["termination"] and abs(s["iterations"] - os_["iterations"]) <= 2, (i, level, s, os_)
                assert strategy != DOGLEG or s["rejected"] == os_["rejected"], (i, level, s["rejected"], os_["rejected"])
                np.testing.assert_allclose(S[i][0]["initial_cost"], O.evaluate_views(_oracle_views(views_data, names, stride, 0), op, opts)["cost"],
                                           rtol=1e-5, err_msg="problem %d: level 0 did not start where level 1 ended" % i)
            else:
                _assert_matches_oracle(poses[i], s, op, os_, strategy == DOGLEG)


# --------------------------------------------------------------- 2. one level: the same problem as ea_solve_views / ea_solve_batch
@pytest.mark.gpu
@pytest.mark.parametrize("level", [0, 1])
def test_single_level_matches_solve_views_and_oracle(ea, ctx, oracle, numpy_pins, views_data, level):
    O = oracle
    x = numpy_pins["xpert"]
    for loss, stride in (("huber", 7), ("trivial", 1)):
        sp = _params(ea, loss, stride, coarsest_level=level, finest_level=level)
        opts = _options(O, loss)
        poses, S = ctx.solve_views_batch([_gpu_views(views_data, p) for p in PROBLEMS], [x] * len(PROBLEMS), sp)
        for i, names in enumerate(PROBLEMS):
            s = S[i][level]
            assert all(S[i][l]["termination"] == 0 for l in range(2) if l != level), "a level outside the range was written"
            vp, vs = ctx.solve_views(_gpu_views(views_data, names), x, sp, level=level)
            _assert_pose_close(poses[i], vp, 2e-6)
            assert s["termination"] == vs["termination"] and abs(s["iterations"] - vs["iterations"]) <= 2, (s, vs)
            assert s["n_residuals"] == vs["n_residuals"]
            ov = _oracle_views(views_data, names, stride, level)
            _assert_own_costs(s, O.evaluate_views(ov, x, opts)["cost"], O.evaluate_views(ov, poses[i], opts)["cost"])
    # a single plain view is the batched mono solver's problem
    A = views_data[0]["plain"]["ref"]
    sp = _params(ea, "huber", 1, coarsest_level=level, finest_level=level)
    poses, S = ctx.solve_views_batch([[views_data[0]["plain"]]], [START], sp)
    bp, bS = ctx.solve_batch(A, [0], A, [1], [START], sp)
    _assert_pose_close(poses[0], bp[0], 2e-6)
    assert S[0][level]["termination"] == bS[0][level]["termination"] and S[0][level]["n_residuals"] == bS[0][level]["n_residuals"]


# ------------------------------------------------------------------------------------------ 3. independence, bit for bit
def _raw(ea, ctx, problems, poses, sp, n_levels):
    """ea_solve_views_batch through ctypes: (status, poses, summaries as one byte string per problem)."""
    from edge_alignment_b200 import _lib as L
    n = len(problems)
    flat = [v for p in problems for v in p]
    offsets = np.zeros(n + 1, np.int32)
    offsets[1:] = np.cumsum([len(p) for p in problems])
    arr = ctx._views(flat) if flat else (L.View * 1)()
    poses = np.array(poses, np.float64).reshape(n, 7).copy()
    S = (L.Summary * max(n * n_levels, 1))()
    rc = L.lib().ea_solve_views_batch(ctx._h, n, offsets.ctypes.data_as(C.POINTER(C.c_int32)), arr,
                                      poses.ctypes.data_as(C.POINTER(C.c_double)), C.byref(sp), S)
    raw = bytes(S)
    size = C.sizeof(L.Summary) * n_levels
    return rc, poses, [raw[i * size:(i + 1) * size] for i in range(n)], S


@pytest.mark.gpu
def test_problem_results_do_not_depend_on_the_batch(ea, ctx, numpy_pins, views_data):
    gv = views_data[0]
    kinds = [["plain"], ["rig_dist"], ["half", "xyz"], ["plain", "tiny", "big", "rig_dist"], ["plain", "rig_dist", "zero", "half", "xyz"],
             ["xyz", "rig_dist"], ["tiny"], ["big"]]
    starts = [IDENTITY, numpy_pins["xpert"], START]
    batch = [[gv[v] for v in kinds[k % len(kinds)]] for k in range(72)]
    bstart = [starts[k % len(starts)] for k in range(72)]
    sp = _params(ea, "huber", 3)
    rc, P, S, _ = _raw(ea, ctx, batch, bstart, sp, 2)
    assert rc == 0
    rc, Pr, Sr, _ = _raw(ea, ctx, batch[::-1], bstart[::-1], sp, 2)
    assert rc == 0
    rc, P2, S2, _ = _raw(ea, ctx, batch, bstart, sp, 2)
    assert rc == 0 and P.tobytes() == P2.tobytes() and S == S2, "two identical calls differ"
    for k in range(len(kinds)):
        rc, P1, S1, _ = _raw(ea, ctx, [batch[k]], [bstart[k]], sp, 2)
        assert rc == 0
        assert P1[0].tobytes() == P[k].tobytes() == Pr[71 - k].tobytes(), k
        assert S1[0] == S[k] == Sr[71 - k], k


# --------------------------------------------------------------------------------------------------------- 4. ground truth
@pytest.mark.gpu
def test_synthetic_stereo_rigs_recover_ground_truth(ea, ctx):
    import torch
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import synth
    n_rigs = 16
    fp = ea.frame_params(n_levels=3)
    left = ea.FrameSet(ctx, fp, 2 * n_rigs)
    right = ea.FrameSet(ctx, fp, 2 * n_rigs)
    try:
        gts, problems = [], []
        for r in range(n_rigs):
            Rw, tw = synth.trajectory(2, 900 + r)                        # frame 0 -> frame 1 of the rig
            Rw2, tw2, rig = synth.stereo_rig(Rw, tw)
            bl, dl = synth.render(Rw, tw, 900 + r, device="cuda")
            br, dr = synth.render(Rw2, tw2, 900 + r, device="cuda")
            torch.cuda.synchronize()
            left.preprocess_device([2 * r, 2 * r + 1], bl.contiguous().data_ptr(), dl.contiguous().data_ptr(), ea.ROLE_BOTH)
            right.preprocess_device([2 * r, 2 * r + 1], br.contiguous().data_ptr(), dr.contiguous().data_ptr(), ea.ROLE_BOTH)
            ctx.sync()
            gts.append(synth.relative_pose(Rw, tw, 0, 1))
            problems.append([dict(ref=left, ref_slot=2 * r, now=left, now_slot=2 * r + 1),
                             dict(ref=right, ref_slot=2 * r, now=right, now_slot=2 * r + 1, T21=rig)])
        sp = ea.solve_params(point_stride=1, loss_type=ea.LOSS_HUBER, loss_scale=0.1)
        poses, S = ctx.solve_views_batch(problems, None, sp)
        for r in range(n_rigs):
            assert np.degrees(rot_angle_between(poses[r][:4], gts[r][:4])) < 1.0, (r, poses[r], gts[r])
            assert np.abs(poses[r][4:] - gts[r][4:]).max() < 0.03, (r, poses[r], gts[r])
            assert all(1 <= S[r][l]["termination"] <= 5 for l in range(3)), [s["termination_name"] for s in S[r]]
    finally:
        left.close(); right.close()


# -------------------------------------------------------------------------------------------------- 5. degenerate inputs
@pytest.fixture(scope="module")
def degen(ea, ctx, frames):
    """64 x 48 frames with XYZ points (z-guard), 640 x 480 slots 0 = frame 0 (points), 1 = frame 2, 3 = no points, and a
    truncated 64 x 48 list; all 1-level."""
    rng = np.random.default_rng(5)
    w, h = 64, 48
    K = (40.0, 40.0, 31.5, 23.5)
    small = ea.FrameSet(ctx, ea.frame_params(width=w, height=h, fx=K[0], fy=K[1], cx=K[2], cy=K[3], max_points=w * h), 1)
    small.set_dt(0, rng.random((h, w)).astype(np.float32))
    p4 = np.ones((400, 4), np.float32)
    p4[:, 0] = rng.uniform(-3, 3, 400); p4[:, 1] = rng.uniform(-3, 3, 400); p4[:, 2] = rng.uniform(0.5, 2.0, 400)
    zpose = np.array([1.0, 0, 0, 0, 0.1, -0.1, 0.2])
    p4[5, :3] = (0.1, 0.1, 0.005 - zpose[6])             # |z'| < 0.01 at zpose (utils.h:70-73)
    small.set_points(0, p4, mode=ea.POINTS_XYZ)
    big = ea.FrameSet(ctx, ea.frame_params(), 4)
    big.preprocess_host([0, 1], frames["bgr"][[0, 2]], frames["depth"][[0, 2]], ea.ROLE_BOTH)
    big.set_points(3, np.zeros((0, 4), np.float32))
    trunc = ea.FrameSet(ctx, ea.frame_params(width=64, height=48, max_points=100), 1)
    trunc.preprocess_host([0], rng.integers(0, 256, (1, 48, 64, 3)).astype(np.uint8), np.full((1, 48, 64), 1000, np.uint16), ea.ROLE_BOTH)
    yield dict(small=small, zpose=zpose, big=big, trunc=trunc)
    small.close(); big.close(); trunc.close()


@pytest.mark.gpu
def test_views_batch_degenerate_inputs(ea, ctx, degen, views_data):
    from edge_alignment_b200 import _lib as L
    D = degen
    big, small = D["big"], D["small"]
    sp = ea.solve_params(point_stride=1, loss_type=ea.LOSS_TRIVIAL)
    ok = dict(ref=big, ref_slot=0, now=big, now_slot=1)
    # no problems: nothing launched
    n0 = ctx.launch_count()
    rc, _, _, _ = _raw(ea, ctx, [], np.zeros((0, 7)), sp, 1)
    assert rc == 0 and ctx.launch_count() == n0
    # every invalid call is refused before anything is launched or written
    two = views_data[0]["plain"]                                              # a 2-level frameset
    invalid = [([[]], sp), ([[ok] * 17], sp), ([[ok], [dict(ok, ref_slot=4)]], sp), ([[dict(ok, now_slot=-1)]], sp),
               ([[ok, two]], sp), ([[ok]], ea.solve_params(point_stride=1, coarsest_level=1)),
               ([[ok]], ea.solve_params(point_stride=1, finest_level=-1)), ([[ok]], ea.solve_params(point_stride=0))]
    for problems, spx in invalid:
        pose = np.tile(START, (len(problems), 1))
        n0 = ctx.launch_count()
        rc, got, _, _ = _raw(ea, ctx, problems, pose, spx, 1)
        assert rc == 1 and ctx.launch_count() == n0 and np.array_equal(got, pose), (problems, rc)
    bad_q = np.array([[1.0, 0.1, 0, 0, 0, 0, 0]])
    rc, got, _, _ = _raw(ea, ctx, [[ok]], bad_q, sp, 1)
    assert rc == 1 and np.array_equal(got, bad_q)
    # view_offsets that decrease or do not start at 0, a null frameset
    for offs in ([0, 2, 1], [1, 2]):
        arr = ctx._views([ok, ok])
        o = np.array(offs, np.int32)
        pose = np.tile(START, (len(offs) - 1, 1))
        rc = L.lib().ea_solve_views_batch(ctx._h, len(offs) - 1, o.ctypes.data_as(C.POINTER(C.c_int32)), arr,
                                          pose.ctypes.data_as(C.POINTER(C.c_double)), C.byref(sp), None)
        assert rc == 1 and np.array_equal(pose, np.tile(START, (len(offs) - 1, 1)))
    arr = ctx._views([ok])
    arr[0].now = None
    o = np.array([0, 1], np.int32)
    pose = START.copy()
    rc = L.lib().ea_solve_views_batch(ctx._h, 1, o.ctypes.data_as(C.POINTER(C.c_int32)), arr, pose.ctypes.data_as(C.POINTER(C.c_double)),
                                      C.byref(sp), None)
    assert rc == 1 and np.array_equal(pose, START)
    # zero residuals at every level: skipped, pose unchanged
    gv = views_data[0]
    poses, S = ctx.solve_views_batch([[gv["zero"]], [gv["plain"]]], [START, START], ea.solve_params(point_stride=7))
    assert [s["termination_name"] for s in S[0]] == ["SKIPPED_NO_POINTS"] * 2 and np.array_equal(poses[0], START)
    assert all(s["evaluations"] == 0 and s["n_residuals"] == 0 for s in S[0])
    assert all(1 <= s["termination"] <= 5 for s in S[1])
    # a z-guard failure at the start pose
    poses, S = ctx.solve_views_batch([[dict(ref=small, ref_slot=0, now=small, now_slot=0)]], [D["zpose"]], sp)
    assert S[0][0]["termination_name"] == "FAILURE_EVAL_X0" and np.array_equal(poses[0], D["zpose"])
    # the iteration cap: same iterations and evaluations as ea_solve_views
    sp3 = ea.solve_params(point_stride=1, max_num_iterations=3)
    poses, S = ctx.solve_views_batch([[ok]], [START], sp3)
    vp, vs = ctx.solve_views([ok], START, sp3)
    assert S[0][0]["termination_name"] == "NO_CONVERGENCE" == vs["termination_name"]
    assert S[0][0]["iterations"] == vs["iterations"] and S[0][0]["evaluations"] == vs["evaluations"]
    _assert_pose_close(poses[0], vp, 2e-6)
    # a truncated list is solved with the cut list, then reported
    tv = dict(ref=D["trunc"], ref_slot=0, now=D["trunc"], now_slot=0)
    rc, got, _, S = _raw(ea, ctx, [[ok], [tv]], [START, START], sp, 1)
    assert rc == 4 and "problem 1, view 0" in L.lib().ea_last_error().decode()
    assert S[1].truncated == 1 and S[0].truncated == 0 and 1 <= S[1].termination <= 5 and S[1].n_residuals == 100
    assert not np.array_equal(got[0], START)


def _scratch_sequence(ea, frames, ctx, calls):
    """Framesets on `ctx` and the given subset of a fixed sequence of calls: views batches of 1, 70 and 1 problems with a views
    solve between them (the context's scratch grows on the second batch)."""
    fs = ea.FrameSet(ctx, ea.frame_params(n_levels=2), 4)
    try:
        fs.preprocess_host([0, 1, 2, 3], frames["bgr"][[0, 2, 3, 1]], frames["depth"][[0, 2, 3, 1]], ea.ROLE_BOTH)
        a = dict(ref=fs, ref_slot=0, now=fs, now_slot=1)
        b = dict(ref=fs, ref_slot=2, now=fs, now_slot=3, T21=T21, dist=DIST)
        many = [[a, b] if k % 3 else [b] * (1 + k % 16) for k in range(70)]
        sp = ea.solve_params(point_stride=3)
        out = {}
        for k in calls:
            if k == "one_a":
                out[k] = ctx.solve_views_batch([[a, b]], None, sp)
            elif k == "many":
                out[k] = ctx.solve_views_batch(many, None, sp)
            elif k == "views":
                out[k] = ctx.solve_views([a, b], None, sp)
            elif k == "one_b":
                out[k] = ctx.solve_views_batch([[b]], [START], sp)
        return out
    finally:
        fs.close()


@pytest.mark.gpu
def test_views_batch_scratch_growth_matches_fresh_context(ea, frames):
    seq = ["one_a", "many", "views", "one_b"]
    c = ea.Context(0)
    try:
        got = _scratch_sequence(ea, frames, c, seq)
    finally:
        c.close()
    for k in seq:
        c = ea.Context(0)
        try:
            want = _scratch_sequence(ea, frames, c, [k])[k]
        finally:
            c.close()
        np.testing.assert_array_equal(got[k][0], want[0], err_msg=k)      # poses
        assert got[k][1] == want[1], k                                    # summaries


# ------------------------------------------------------------------------------------- 6. spill guard (no GPU needed)
# ptxas' figures for CUDA 12.9, in bytes: (max spill stores, max spill loads).  k_views_batch's own spills are three words
# stored before the evaluation loop and reloaded after it (tid / lane / warp, live across the boss warp's calls) and one word
# around the LM call: its SASS has no local-memory access between the start and the end of the evaluation loop.
LIMITS = {
    "k_views_batchILi256E": (20, 28),
    "ea_lm_advance_warp": (0, 0),
    "vb_boss_next": (0, 0),
    "vb_fold": (0, 0),
}


def test_views_batch_kernel_spills_are_pinned():
    from edge_alignment_b200 import build
    try:
        nvcc = build.nvcc()
    except RuntimeError:
        pytest.skip("nvcc not found")
    if not (os.path.exists(nvcc) or shutil.which(nvcc)):
        pytest.skip("nvcc not found")
    with tempfile.TemporaryDirectory() as tmp:
        cmd = [nvcc] + build.NVCC_FLAGS + ["-Xptxas", "-v", "-c", os.path.join(build.CSRC, "ea_views_batch.cu"), "-o",
                                           os.path.join(tmp, "ea_views_batch.o")]
        p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert p.returncode == 0, p.stdout[-4000:]
    found, name = [], None
    for line in p.stdout.splitlines():
        m = re.search(r"Function properties for (\S+)", line)
        if m:
            name = m.group(1)
            continue
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and name:
            found.append((name, int(m.group(2)), int(m.group(3))))
            name = None
    for frag, (max_st, max_ld) in LIMITS.items():
        hits = [r for r in found if frag in r[0]]
        assert hits, "ptxas reported no function matching %s" % frag
        for fn, st, ld in hits:
            assert st <= max_st and ld <= max_ld, "%s spills %d B stored / %d B loaded (limit %d / %d)" % (fn, st, ld, max_st, max_ld)
