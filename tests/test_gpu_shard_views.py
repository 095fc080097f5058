"""The point-sharded solve (ea_shard_solve: the persistent kernel k_shard_solve and its host-driven twin selected with
EA_SHARD_MODE=nccl) and the multi-view solve (ea_solve_views: k_views_solve) against the fp64 oracle.

Both kernels share the per-point evaluation and the LM step with the batched solver but own their grid reduce, the slicing of
the point list over CTAs, the control-block set-up and (shard) the cp.async staging with alternating sweep direction.  Every
solve here is checked three ways:
  * against the oracle's solve on the same inputs (pose 1e-4 rad / 1e-4 m, costs 1e-5 relative, iterations +-2, same
    termination; same rejected steps for dogleg),
  * its own evaluations: initial_cost is the oracle's cost at the start pose and final_cost the oracle's cost at the RETURNED
    pose, both to 2e-6 relative (the bound of test_eval_parity).  The final cost comes from a late evaluation, one that ran
    with the reversed sweep and the point the previous evaluation prefetched, so this reaches the staging and the direction
    logic even where the LM paths of GPU and oracle part ways,
  * and, for the slice shapes, twice in a row bit for bit.
World 1 only: the two-rank slicing needs two GPUs (test_gpu_multi.py).
"""
import ctypes as C

import numpy as np
import pytest

from conftest import IDENTITY, rot_angle_between

pytestmark = pytest.mark.gpu

LM, DOGLEG = 0, 1
LOSSES = {"trivial": (0, 1.0), "cauchy": (1, 1.0), "huber": (2, 0.1)}
R_FLOOR = 0.05


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


@pytest.fixture(params=["kernel", "nccl"])
def shard(request, ea, ctx, monkeypatch):
    """A world-1 shard on the persistent cooperative kernel ("kernel") or on the host-driven launch loop ("nccl")."""
    monkeypatch.setenv("EA_SHARD_MODE", request.param)      # read by ea_shard_create
    sh = ea.Shard(ctx)
    sh.mode = request.param
    yield sh
    sh.close()


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


def _options(O, loss, strategy=LM, radius=1e4, max_it=50):
    t, s = LOSSES[loss]
    return O.default_options(loss_type=t, loss_scale=s, strategy=strategy, initial_radius=radius, max_num_iterations=max_it)


def _params(ea, loss, stride, strategy=LM, radius=1e4, max_it=50):
    t, s = LOSSES[loss]
    return ea.solve_params(point_stride=stride, loss_type=t, loss_scale=s, trust_region_strategy=strategy,
                           initial_trust_region_radius=radius, max_num_iterations=max_it)


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
    """initial_cost / final_cost are the kernel's own evaluations at the start pose and at the returned pose.  A relative bound
    means nothing once the solve drives the cost to zero (one residual: 1e-17 on the GPU, exactly 0 in fp64), so each residual
    may also be off by the suite's residual floor, 1e-5 * R_FLOOR, which bounds its cost by (5e-7)^2 / 2 ~ 1.3e-13 near r = 0."""
    atol = s["n_residuals"] * 0.5 * (1e-5 * R_FLOOR) ** 2
    np.testing.assert_allclose(s["initial_cost"], cost_at_start, rtol=2e-6, atol=atol, err_msg="initial_cost")
    np.testing.assert_allclose(s["final_cost"], cost_at_pose, rtol=2e-6, atol=atol, err_msg="final_cost")


def _assert_residual_parity(gpu_raw, ref_raw):
    tol = 1e-5 * np.maximum(np.abs(ref_raw), R_FLOOR)
    bad = np.abs(gpu_raw - ref_raw) > tol
    assert not bad.any(), "max excess %g at %s" % ((np.abs(gpu_raw - ref_raw) / tol).max(), np.nonzero(bad)[0][:8])


# ------------------------------------------------------------------------- 1. the shard solve across the parameter space
PAIRS = ((0, 2), (3, 1))


@pytest.fixture(scope="module")
def pyr(ea, ctx, frames, oracle):
    """Frames 0->2 and 3->1 on a 3-level frameset (slots 0/1 and 2/3), plus the fp32 XYZ points of frames 0 and 3 (slots 4, 5),
    with the oracle's inputs per (pair, level) built as test_preprocess_pyramid_and_variants builds them."""
    O = oracle
    fs = ea.FrameSet(ctx, ea.frame_params(n_levels=3), 6)
    order = [0, 2, 3, 1]
    fs.preprocess_host([0, 1, 2, 3], frames["bgr"][order], frames["depth"][order], ea.ROLE_BOTH)
    inp = {}
    for p, (a, b) in enumerate(PAIRS):
        for l in range(3):
            K = fs.level_geometry(l)[2]
            ba, da = _halve(O, frames["bgr"][a], frames["depth"][a], l)
            bb, _ = _halve(O, frames["bgr"][b], frames["depth"][b], l)
            xyz, _ = O.get_aX(ba, da, K)
            dt, _ = O.get_distance_transform(bb)
            inp[p, l, "pixel"] = dict(xyz=xyz, dt=dt, K=K, ref=2 * p, now=2 * p + 1)
        p4 = _xyz4(inp[p, 0, "pixel"]["xyz"])
        fs.set_points(4 + p, p4, mode=ea.POINTS_XYZ)
        inp[p, 0, "xyz"] = dict(inp[p, 0, "pixel"], xyz=p4[:, :3].astype(np.float64), ref=4 + p)   # the same fp32-rounded points
    yield fs, inp
    fs.close()


# (loss, strategy, radius, stride, start, points, level, pair): every loss with every strategy, and every value of every other
# axis at least once
SOLVE_CASES = [
    ("trivial", LM, 1e4, 1, "identity", "pixel", 0, 0),
    ("trivial", LM, 1e-2, 7, "xpert", "xyz", 0, 1),
    ("trivial", DOGLEG, 1e-2, 7, "identity", "pixel", 1, 0),
    ("cauchy", LM, 1e4, 7, "xpert", "pixel", 2, 1),
    ("cauchy", LM, 1e-2, 1, "identity", "xyz", 0, 0),
    ("cauchy", DOGLEG, 1e-2, 1, "xpert", "pixel", 0, 1),
    ("huber", LM, 1e4, 7, "identity", "xyz", 0, 1),
    ("huber", LM, 1e-2, 1, "xpert", "pixel", 1, 1),
    ("huber", DOGLEG, 1e-2, 7, "xpert", "pixel", 2, 0),
    ("huber", DOGLEG, 1e-2, 1, "identity", "xyz", 0, 0),
]


def _case_id(c):
    return "%s-%s%g-s%d-%s-%s-L%d-p%d" % (c[0], "lm" if c[1] == LM else "dl", c[2], c[3], c[4], c[5], c[6], c[7])


@pytest.mark.parametrize("case", SOLVE_CASES, ids=[_case_id(c) for c in SOLVE_CASES])
def test_shard_solve_matches_oracle(ea, oracle, numpy_pins, pyr, shard, case):
    O = oracle
    loss, strategy, radius, stride, start, points, level, pair = case
    fs, inp = pyr
    d = inp[pair, level, points]
    start7 = IDENTITY if start == "identity" else numpy_pins["xpert"]
    max_it = 200 if strategy == DOGLEG else 50
    opts = _options(O, loss, strategy, radius, max_it)
    pose, s = shard.solve(fs, d["ref"], fs, d["now"], start7, _params(ea, loss, stride, strategy, radius, max_it), level=level)
    op, os_, _ = O.solve(d["xyz"], d["dt"], d["K"], start7, stride=stride, options=opts)
    assert s["evaluations"] > 1 and s["truncated"] == 0
    _assert_matches_oracle(pose, s, op, os_, strategy == DOGLEG)
    _assert_own_costs(s, O.evaluate(d["xyz"], d["dt"], d["K"], start7, stride=stride, options=opts)["cost"],
                      O.evaluate(d["xyz"], d["dt"], d["K"], pose, stride=stride, options=opts)["cost"])
    prof = shard.profile()
    assert prof["in_kernel"] == (shard.mode == "kernel") and prof["evaluations"] == s["evaluations"]


# --------------------------------------------------------------------------------------------------------- 3. slice shapes
# k_shard_solve runs min(sm, ceil(n / 1024)) CTAs of 512 threads: one loop iteration is one 512-point staging slot and the
# fp32 -> fp64 flush comes every 16 iterations.  The counts put the slice boundaries on, just before and just after those
# sizes, and (1024 sm + k) gives uneven slices on the full grid.
BASE_COUNTS = [1, 31, 255, 256, 257, 511, 512, 513, 1023, 1024, 1025, 3 * 1024 + 1, 8191, 8192, 8193]
SM_OFFSETS = [-1, 0, 1, 37]
COUNTS = ["n%d" % n for n in BASE_COUNTS] + ["sm%+d" % k for k in SM_OFFSETS]


def _count(name, sm):
    return int(name[1:]) if name[0] == "n" else 1024 * sm + int(name[2:])


@pytest.fixture(scope="module")
def slices(ea, ctx, frames, oracle):
    """Reference points chosen one by one with set_points: a prefix of frame 0's point list, tiled (duplicates included) for
    the counts above its 44458 points.  The reference frameset is twice as wide as the frames only for its capacity: at stride
    3 the largest count needs 3 (1024 sm + 37) points, more than a 640 x 480 level holds.  Its intrinsics are the frames'.
    The now side is frame 2's distance transform from the oracle."""
    O = oracle
    K = frames["K"]
    sm = ctx.device_info()["sm_count"]
    xyz, uvd = O.get_aX(frames["bgr"][0], frames["depth"][0], K)
    dt, _ = O.get_distance_transform(frames["bgr"][2])
    ref = ea.FrameSet(ctx, ea.frame_params(width=1280, height=480, fx=K[0], fy=K[1], cx=K[2], cy=K[3], max_points=1280 * 480), 1)
    now = ea.FrameSet(ctx, ea.frame_params(max_points=640 * 480), 1)
    now.set_dt(0, dt)
    cache = {}
    yield dict(O=O, K=K, sm=sm, xyz=xyz, uvd=uvd, dt=dt, ref=ref, now=now, cache=cache)
    ref.close(); now.close()


def _load_slice(ea, S, reach, n):
    """Sets the reference list for `n` residuals reached by list length (stride 1) or through stride 3; returns (stride,
    oracle points)."""
    stride = 3 if reach == "stride3" else 1
    m = 3 * n - 2 if stride == 3 else n                   # the last residual is the last point of the list
    idx = np.arange(m) % len(S["uvd"])
    if reach == "xyz":
        p4 = _xyz4(S["xyz"][idx])
        S["ref"].set_points(0, p4, mode=ea.POINTS_XYZ)
        return stride, p4[:, :3].astype(np.float64)
    S["ref"].set_points(0, ea.pixel_points(S["uvd"][idx]), mode=ea.POINTS_PIXEL)
    return stride, S["xyz"][idx]


@pytest.mark.parametrize("count", COUNTS)
@pytest.mark.parametrize("reach", ["length", "stride3", "xyz"])
def test_shard_slice_shapes(ea, slices, shard, reach, count):
    S = slices
    O = S["O"]
    n = _count(count, S["sm"])
    stride, xyz = _load_slice(ea, S, reach, n)
    sp = ea.solve_params(point_stride=stride)
    runs = [shard.solve(S["ref"], 0, S["now"], 0, None, sp) for _ in range(2)]
    (pose, s), (pose2, s2) = runs
    assert np.array_equal(pose, pose2) and s == s2, "two runs differ"
    assert 1 <= s["termination"] <= 5, s["termination_name"]
    assert s["n_residuals"] == n
    opts = O.default_options()
    _assert_own_costs(s, O.evaluate(xyz, S["dt"], S["K"], IDENTITY, stride=stride, options=opts)["cost"],
                      O.evaluate(xyz, S["dt"], S["K"], pose, stride=stride, options=opts)["cost"])
    if n >= 1000:
        key = (reach, n)
        if key not in S["cache"]:
            S["cache"][key] = O.solve(xyz, S["dt"], S["K"], IDENTITY, stride=stride, options=opts)[:2]
        op, os_ = S["cache"][key]
        _assert_matches_oracle(pose, s, op, os_, False)


@pytest.mark.parametrize("count", COUNTS)
def test_shard_modes_agree(ea, ctx, slices, monkeypatch, count):
    """The persistent kernel and the host-driven loop: same solve, different reduction trees (so not bit for bit)."""
    S = slices
    n = _count(count, S["sm"])
    stride, _ = _load_slice(ea, S, "length", n)
    out = {}
    for mode in ("kernel", "nccl"):
        monkeypatch.setenv("EA_SHARD_MODE", mode)
        sh = ea.Shard(ctx)
        try:
            out[mode] = sh.solve(S["ref"], 0, S["now"], 0, None, ea.solve_params(point_stride=stride))
            assert sh.profile()["in_kernel"] == (mode == "kernel")
        finally:
            sh.close()
    (pk, sk), (pn, sn) = out["kernel"], out["nccl"]
    _assert_pose_close(pk, pn, 2e-6)
    assert abs(sk["iterations"] - sn["iterations"]) <= 1
    assert sk["n_residuals"] == sn["n_residuals"] == n


# ------------------------------------------------------------------------------------------------------ 4. multi-view solve
ANG = 0.05
T21 = np.eye(4)
T21[:3, :3] = [[np.cos(ANG), 0, np.sin(ANG)], [0, 1, 0], [-np.sin(ANG), 0, np.cos(ANG)]]
T21[:3, 3] = [-0.1, 0.01, 0.02]
DIST = (0.1, -0.2, 0.001, -0.002, 0.05)
N_BIG = 100_003


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


LAYOUTS = {
    "zero_between": ["plain", "rig_dist", "zero", "half", "xyz"],     # an empty view in the middle of the list
    "tiny_big": ["plain", "tiny", "big", "rig_dist"],                 # 5 points beside 1e5: most CTAs have no slice of the tiny view
}
# (strategy, loss, stride, level, start)
VIEW_CASES = [(LM, "trivial", 1, 0, "identity"), (DOGLEG, "huber", 7, 1, "xpert"), (LM, "huber", 7, 1, "identity"),
              (DOGLEG, "trivial", 1, 0, "xpert")]


def _view_lists(views_data, names, stride, level):
    gv, ov = views_data
    return [gv[v] for v in names], [dict(ov[v, level], stride=stride) for v in names]


@pytest.mark.parametrize("case", VIEW_CASES, ids=["%s-%s-s%d-L%d-%s" % ("lm" if c[0] == LM else "dl", c[1], c[2], c[3], c[4]) for c in VIEW_CASES])
@pytest.mark.parametrize("layout", sorted(LAYOUTS))
def test_views_solve_matches_oracle(ea, ctx, oracle, numpy_pins, views_data, layout, case):
    O = oracle
    strategy, loss, stride, level, start = case
    start7 = IDENTITY if start == "identity" else numpy_pins["xpert"]
    max_it = 200 if strategy == DOGLEG else 50
    radius = 1e-2 if strategy == DOGLEG else 1e4
    gv, ov = _view_lists(views_data, LAYOUTS[layout], stride, level)
    opts = _options(O, loss, strategy, radius, max_it)
    pose, s = ctx.solve_views(gv, start7, _params(ea, loss, stride, strategy, radius, max_it), level=level)
    op, os_ = O.solve_views(ov, start7, opts)
    assert s["n_residuals"] == sum((len(v["xyz"]) + stride - 1) // stride for v in ov)
    _assert_matches_oracle(pose, s, op, os_, strategy == DOGLEG)
    _assert_own_costs(s, O.evaluate_views(ov, start7, opts)["cost"], O.evaluate_views(ov, pose, opts)["cost"])


def test_eval_views_output_offsets(ea, ctx, oracle, numpy_pins, views_data):
    """ea_eval_views writes every view's residuals and Jacobian rows at its offset in the concatenated output: an empty view
    and an XYZ view between others must not shift what follows them."""
    O = oracle
    x = numpy_pins["xpert"]
    for level, stride in ((0, 7), (1, 1)):
        gv, ov = _view_lists(views_data, ["plain", "zero", "xyz", "rig_dist", "zero", "half"], stride, level)
        sp = _params(ea, "huber", stride)
        g = ctx.eval_views(gv, x, sp, level=level)
        o = O.evaluate_views(ov, x, _options(O, "huber"))
        assert g["failed"] == 0 and o["ok"] and g["n_residuals"] == len(o["raw"])
        _assert_residual_parity(g["raw"], o["raw"])
        _assert_residual_parity(g["residuals"], o["residuals"])
        jscale = np.abs(o["J"]).max(0)
        assert (np.abs(g["J"] - o["J"]) <= 3e-5 * jscale + 3e-5 * np.abs(o["J"])).all()
        np.testing.assert_allclose(g["cost"], o["cost"], rtol=3e-6)
        np.testing.assert_allclose(g["H"], o["H"], rtol=0, atol=3e-6 * np.abs(np.diag(o["H"])).max())
        np.testing.assert_allclose(g["b"], o["b"], rtol=0, atol=3e-6 * (np.abs(o["J"]) * np.abs(o["residuals"])[:, None]).sum(0).max())


def _scratch_sequence(ea, frames, ctx, calls):
    """Framesets on `ctx` and the given subset of a fixed sequence of calls: views solves of 1, 6 and 1 views with a shard solve
    and a batched solve between them (the views scratch of the context grows on the second views solve)."""
    fs = ea.FrameSet(ctx, ea.frame_params(), 4)
    try:
        fs.preprocess_host([0, 1, 2, 3], frames["bgr"][[0, 2, 3, 1]], frames["depth"][[0, 2, 3, 1]], ea.ROLE_BOTH)
        one = [dict(ref=fs, ref_slot=0, now=fs, now_slot=1)]
        six = [dict(ref=fs, ref_slot=0, now=fs, now_slot=1), dict(ref=fs, ref_slot=2, now=fs, now_slot=3, T21=T21, dist=DIST),
               dict(ref=fs, ref_slot=0, now=fs, now_slot=3, dist=DIST), dict(ref=fs, ref_slot=2, now=fs, now_slot=1),
               dict(ref=fs, ref_slot=0, now=fs, now_slot=1, T21=T21), dict(ref=fs, ref_slot=2, now=fs, now_slot=3)]
        sp = ea.solve_params(point_stride=1)
        out = {}
        for k in calls:
            if k == "views1a":
                out[k] = ctx.solve_views(one, None, sp)
            elif k == "shard":
                sh = ea.Shard(ctx)
                try:
                    out[k] = sh.solve(fs, 2, fs, 3, None, sp)
                finally:
                    sh.close()
            elif k == "views6":
                out[k] = ctx.solve_views(six, None, sp)
            elif k == "batch":
                out[k] = ctx.solve_batch(fs, [0, 2], fs, [1, 3], None, sp)
            elif k == "views1b":
                out[k] = ctx.solve_views(one, START, sp)
        return out
    finally:
        fs.close()


def test_views_scratch_growth_matches_fresh_context(ea, frames, monkeypatch):
    monkeypatch.setenv("EA_SHARD_MODE", "kernel")
    seq = ["views1a", "shard", "views6", "batch", "views1b"]
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


# -------------------------------------------------------------------------------------------------- 5. degenerate inputs
def _filled_summary(L):
    """A Summary whose every field holds a sentinel: the solver must write all of them."""
    s = L.Summary()
    for name, t in L.Summary._fields_:
        setattr(s, name, -7.0 if t is C.c_double else 0x5A5A5A5A)
    return s


def _raw_shard_solve(L, sh, ref, ref_slot, now, now_slot, pose, sp, level=0):
    s = _filled_summary(L)
    rc = L.lib().ea_shard_solve(sh._h, ref._h, ref_slot, now._h, now_slot, level, pose.ctypes.data_as(C.POINTER(C.c_double)),
                                C.byref(sp), C.byref(s))
    return rc, s.asdict()


def _raw_solve_views(L, ctx, views, pose, sp, level=0):
    s = _filled_summary(L)
    rc = L.lib().ea_solve_views(ctx._h, len(views), ctx._views(views), level, pose.ctypes.data_as(C.POINTER(C.c_double)),
                                C.byref(sp), C.byref(s))
    return rc, s.asdict()


@pytest.fixture(scope="module")
def degen(ea, ctx, frames):
    """64 x 48 frames with XYZ points (z-guard), and 640 x 480 slots: 0 = frame 0 (points), 1 = frame 2, 2 = flat image (no
    edges: its distance transform is constant), 3 = no points."""
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
    flat = np.full((1, 480, 640, 3), 128, np.uint8)
    big.preprocess_host([0, 1], frames["bgr"][[0, 2]], frames["depth"][[0, 2]], ea.ROLE_BOTH)
    big.preprocess_host([2], flat, np.full((1, 480, 640), 5000, np.uint16), ea.ROLE_BOTH)
    big.set_points(3, np.zeros((0, 4), np.float32))
    trunc = ea.FrameSet(ctx, ea.frame_params(width=64, height=48, max_points=100), 1)
    trunc.preprocess_host([0], rng.integers(0, 256, (1, 48, 64, 3)).astype(np.uint8), np.full((1, 48, 64), 1000, np.uint16), ea.ROLE_BOTH)
    yield dict(small=small, zpose=zpose, big=big, trunc=trunc)
    small.close(); big.close(); trunc.close()


START = np.array([0.99995, 0.006, -0.004, 0.005, 0.01, -0.01, 0.02])
START[:4] /= np.linalg.norm(START[:4])


def test_shard_degenerate_inputs(ea, ctx, degen, shard):
    from edge_alignment_b200 import _lib as L
    D = degen
    big, small = D["big"], D["small"]
    sp = ea.solve_params(point_stride=1, loss_type=ea.LOSS_TRIVIAL)
    # a point at |z'| < 0.01 at the start pose: FAILURE_EVAL_X0 (as the batched solver), pose untouched
    pose, s = shard.solve(small, 0, small, 0, D["zpose"], sp)
    assert s["termination_name"] == "FAILURE_EVAL_X0" and np.array_equal(pose, D["zpose"])
    _, S = ctx.solve_batch(small, [0], small, [0], [D["zpose"]], sp)
    assert S[0][0]["termination_name"] == "FAILURE_EVAL_X0"
    # a now-frame without edges: zero gradient, immediate convergence, pose bit for bit
    pose, s = shard.solve(big, 0, big, 2, START, ea.solve_params())
    assert s["termination_name"] == "CONVERGENCE_GRADIENT" and np.array_equal(pose, START) and s["evaluations"] == 1
    assert s["initial_cost"] == 0.0 and s["final_cost"] == 0.0
    # the iteration cap binds: both paths stop where the batched solver stops
    sp3 = ea.solve_params(point_stride=1, max_num_iterations=3)
    pose, s = shard.solve(big, 0, big, 1, START, sp3)
    bp, bS = ctx.solve_batch(big, [0], big, [1], [START], sp3)
    assert s["iterations"] <= 3 and s["termination_name"] == "NO_CONVERGENCE" == bS[0][0]["termination_name"]
    assert s["iterations"] == bS[0][0]["iterations"] and s["evaluations"] == bS[0][0]["evaluations"] <= 3 + 2
    _assert_pose_close(pose, bp[0], 2e-6)
    # a truncated reference list is refused (EA_ERR_CAPACITY), as ea_solve_batch refuses it
    with pytest.raises(ea.EaError) as e:
        shard.solve(D["trunc"], 0, D["trunc"], 0, None, sp)
    assert e.value.code == 4
    # bad level / slot (EA_ERR_INVALID_ARG)
    for args, level in (((big, 0, big, 1), 1), ((big, 4, big, 1), 0), ((big, 0, big, -1), 0)):
        with pytest.raises(ea.EaError) as e:
            shard.solve(*args, None, sp, level=level)
        assert e.value.code == 1
    # no residuals: skipped like the batched solver -- pose untouched, no evaluation, nothing launched
    n0 = ctx.launch_count()
    pose = START.copy()
    rc, s = _raw_shard_solve(L, shard, big, 3, big, 1, pose, sp)
    assert rc == 0 and ctx.launch_count() == n0
    assert s["termination_name"] == "SKIPPED_NO_POINTS" and s["evaluations"] == 0 and s["n_residuals"] == 0 and s["iterations"] == 0
    assert s["initial_cost"] == 0.0 and s["final_cost"] == 0.0 and s["truncated"] == 0 and s["reserved"] == 0
    assert np.array_equal(pose, START)
    _, bS = ctx.solve_batch(big, [3], big, [1], [START], sp)
    assert bS[0][0]["termination_name"] == "SKIPPED_NO_POINTS"
    # every summary field is written
    rc, s = _raw_shard_solve(L, shard, big, 0, big, 1, START.copy(), ea.solve_params(point_stride=30))
    assert rc == 0 and s["truncated"] == 0 and s["reserved"] == 0 and 1 <= s["termination"] <= 5


def test_views_degenerate_inputs(ea, ctx, degen):
    from edge_alignment_b200 import _lib as L
    D = degen
    big, small = D["big"], D["small"]
    sp = ea.solve_params(point_stride=1, loss_type=ea.LOSS_TRIVIAL)
    pose, s = ctx.solve_views([dict(ref=small, ref_slot=0, now=small, now_slot=0)], D["zpose"], sp)
    assert s["termination_name"] == "FAILURE_EVAL_X0" and np.array_equal(pose, D["zpose"])
    pose, s = ctx.solve_views([dict(ref=big, ref_slot=0, now=big, now_slot=2)], START, ea.solve_params())
    assert s["termination_name"] == "CONVERGENCE_GRADIENT" and np.array_equal(pose, START) and s["evaluations"] == 1
    sp3 = ea.solve_params(point_stride=1, max_num_iterations=3)
    pose, s = ctx.solve_views([dict(ref=big, ref_slot=0, now=big, now_slot=1)], START, sp3)
    bp, bS = ctx.solve_batch(big, [0], big, [1], [START], sp3)
    assert s["iterations"] <= 3 and s["termination_name"] == "NO_CONVERGENCE" == bS[0][0]["termination_name"]
    assert s["iterations"] == bS[0][0]["iterations"] and s["evaluations"] == bS[0][0]["evaluations"]
    _assert_pose_close(pose, bp[0], 2e-6)
    ok = dict(ref=big, ref_slot=0, now=big, now_slot=1)
    with pytest.raises(ea.EaError) as e:
        ctx.solve_views([ok, dict(ref=D["trunc"], ref_slot=0, now=D["trunc"], now_slot=0)], None, sp)
    assert e.value.code == 4
    with pytest.raises(ea.EaError) as e:
        ctx.eval_views([dict(ref=D["trunc"], ref_slot=0, now=D["trunc"], now_slot=0)], IDENTITY, sp)
    assert e.value.code == 4
    for views, level in (([ok], 1), ([ok, dict(ok, ref_slot=4)], 0), ([dict(ok, now_slot=-1), ok], 0)):
        with pytest.raises(ea.EaError) as e:
            ctx.solve_views(views, None, sp, level=level)
        assert e.value.code == 1
    # no residuals over all views: skipped like the batched solver, nothing launched
    empty = dict(ref=big, ref_slot=3, now=big, now_slot=1)
    n0 = ctx.launch_count()
    pose = START.copy()
    rc, s = _raw_solve_views(L, ctx, [empty, empty], pose, sp)
    assert rc == 0 and ctx.launch_count() == n0
    assert s["termination_name"] == "SKIPPED_NO_POINTS" and s["evaluations"] == 0 and s["n_residuals"] == 0 and s["iterations"] == 0
    assert s["initial_cost"] == 0.0 and s["final_cost"] == 0.0 and s["truncated"] == 0 and s["reserved"] == 0
    assert np.array_equal(pose, START)
    # every summary field is written (truncated and reserved included)
    rc, s = _raw_solve_views(L, ctx, [ok, empty], START.copy(), ea.solve_params(point_stride=30))
    assert rc == 0 and s["truncated"] == 0 and s["reserved"] == 0 and 1 <= s["termination"] <= 5
