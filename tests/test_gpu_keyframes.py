"""Tracker key-frame policy mode (ea_tracker_set_keyframe_policy, ea_tracker_get_trajectory, ea_tracker_wait_trajectory).

Every stream decides on the device when its own key frame changes (interval, translation, rotation, cost, lost) and keeps a
world trajectory, world_T_frame = world_T_key o inverse(key_T_frame), the world being the stream's frame 0.  The fixed-interval
tracker is the oracle for policy {max_interval = K}: the same pairs with the same warm starts, so the results are bit-identical.
Everything else is replayed on the host: the decision rule from the returned poses and summaries, the composition in numpy
fp64, and every (key, frame, warm start) pair through ctx.solve_batch.
"""
import ctypes as C
import math
import os
import sys

import numpy as np
import pytest

from conftest import ROOT

sys.path.insert(0, os.path.join(ROOT, "tools"))

W, H = 640, 480
LOST_TERMS = (6, 7, 8)   # EA_TERM_FAILURE_EVAL_X0, EA_TERM_FAILURE_INVALID_STEPS, EA_TERM_SKIPPED_NO_POINTS


def test_keyframe_struct_layouts_match_header():
    from edge_alignment_b200 import _lib as L
    assert C.sizeof(L.KeyframePolicy) == 4 + 4 + 3 * 8
    assert C.sizeof(L.TrackInfo) == 2 * 4
    assert (L.KEY_FIRST, L.KEY_INTERVAL, L.KEY_TRANSLATION, L.KEY_ROTATION, L.KEY_COST, L.KEY_LOST) == (1, 2, 4, 8, 16, 32)


@pytest.fixture(scope="module")
def ea():
    import edge_alignment_b200 as ea
    return ea


@pytest.fixture(scope="module")
def ctx(ea):
    c = ea.Context(0)
    yield c
    c.close()


# ---- numpy fp64 pose algebra (wxyz quaternions) ---------------------------------------------------------------------------
def qmul(a, b):
    return np.array([a[0] * b[0] - a[1] * b[1] - a[2] * b[2] - a[3] * b[3],
                     a[0] * b[1] + a[1] * b[0] + a[2] * b[3] - a[3] * b[2],
                     a[0] * b[2] - a[1] * b[3] + a[2] * b[0] + a[3] * b[1],
                     a[0] * b[3] + a[1] * b[2] - a[2] * b[1] + a[3] * b[0]])


def qrot(q, v):
    u = q[1:]
    c = np.cross(u, v)
    return v + 2.0 * (q[0] * c + np.cross(u, c))


def compose(world_key, pose):
    """world_T_frame = world_T_key o inverse(key_T_frame)."""
    q = qmul(world_key[:4], np.array([pose[0], -pose[1], -pose[2], -pose[3]]))
    q = q / np.linalg.norm(q)
    return np.concatenate([q, world_key[4:] - qrot(q, pose[4:])])


def rot_angle(q):
    return 2.0 * math.atan2(float(np.linalg.norm(q[1:4])), abs(float(q[0])))


def pose_err(a, b):
    d = abs(float(np.dot(a[:4] / np.linalg.norm(a[:4]), b[:4] / np.linalg.norm(b[:4]))))
    return 2.0 * math.acos(min(1.0, d)), float(np.linalg.norm(a[4:] - b[4:]))


# ---- sequences and runs -------------------------------------------------------------------------------------------------
def make_seq(speeds, T, seed):
    """One synthetic sequence per (max_rot_deg, max_trans) entry: bgr [T,S,h,w,3] u8 and depth [T,S,h,w] u16 on the GPU,
    plus the camera-to-world trajectories."""
    import torch
    import synth
    S = len(speeds)
    bgr = torch.empty((T, S, H, W, 3), dtype=torch.uint8, device="cuda")
    depth = torch.empty((T, S, H, W), dtype=torch.uint16, device="cuda")
    traj = []
    for s, (rot, trans) in enumerate(speeds):
        Rw, tw = synth.trajectory(T, seed * 1009 + s, max_rot_deg=rot, max_trans=trans)
        b, d = synth.render(Rw, tw, seed * 1009 + s, W, H, device="cuda")
        bgr[:, s] = b; depth[:, s] = d
        traj.append((Rw, tw))
    torch.cuda.synchronize()
    return bgr.contiguous(), depth.contiguous(), traj


def rows(S):
    return [tuple(getattr(s, k) for k, _ in s._fields_) for s in S]


def run(tr, img, depth, mode="device", policy=True):
    """Steps every frame; per frame (poses [S,7], summary rows, world [S,7], key_frame [S], key_reasons [S]) -- the last three
    None without a policy.  mode: "device" (stream-ordered), "ready" (set_inputs_ready) or "host" (pinned, submit t, wait t-1)."""
    import torch
    T = img.shape[0]
    fi, fd = img[0].numel(), depth[0].numel() * 2
    out = []
    if mode == "host":
        hi, hd = img.cpu().pin_memory(), depth.cpu().pin_memory()
        torch.cuda.synchronize()

        def collect(t):
            p, S = tr.wait(t)
            out.append((p, rows(S)) + (tr.wait_trajectory(t) if policy else (None, None, None)))
        for t in range(T):
            tr.step_host(hi.data_ptr() + t * fi, hd.data_ptr() + t * fd, fetch=False)
            if t > 0:
                collect(t - 1)
        collect(T - 1)
        return out
    tr.set_inputs_ready(mode == "ready")
    for t in range(T):
        tr.step_device(img.data_ptr() + t * fi, depth.data_ptr() + t * fd)
        p, S = tr.poses()
        out.append((p, rows(S)) + (tr.trajectory() if policy else (None, None, None)))
    tr.set_inputs_ready(False)
    return out


def replay_rule(res, n_levels, finest, max_interval=0, max_translation=0.0, max_rotation=0.0, max_cost=0.0):
    """The decision rule on the host from the returned poses and summaries: (key_frame [T,S], key_reasons [T,S])."""
    T, S = len(res), res[0][0].shape[0]
    kf = np.zeros((T, S), np.int32); rs = np.zeros((T, S), np.int32)
    rs[0] = 1
    cur = np.zeros(S, np.int32)
    for t in range(1, T):
        for s in range(S):
            p = res[t][0][s]; sm = res[t][1][s * n_levels + finest]
            term, n_res, cost = sm[0], sm[4], sm[7]
            r = 0
            if max_interval > 0 and t - cur[s] >= max_interval:
                r |= 2
            if term in LOST_TERMS:
                r |= 32
            else:
                if max_translation > 0 and np.linalg.norm(p[4:]) > max_translation:
                    r |= 4
                if max_rotation > 0 and rot_angle(p) > max_rotation:
                    r |= 8
                if max_cost > 0 and n_res > 0 and cost / n_res > max_cost:
                    r |= 16
            kf[t, s] = cur[s]; rs[t, s] = r
            if r:
                cur[s] = t
    return kf, rs


def check_composition(res):
    """World poses against the numpy composition of the returned poses along the returned key chain (1e-12)."""
    T, S = len(res), res[0][0].shape[0]
    for s in range(S):
        np.testing.assert_array_equal(res[0][2][s], [1, 0, 0, 0, 0, 0, 0])
        for t in range(1, T):
            k = res[t][3][s]
            if res[t][4][s] & 32:
                np.testing.assert_array_equal(res[t][2][s], res[t - 1][2][s])
                continue
            np.testing.assert_allclose(res[t][2][s], compose(res[k][2][s], res[t][0][s]), rtol=0, atol=1e-12,
                                       err_msg="stream %d frame %d" % (s, t))


def assert_bit_identical(a, b, world=True):
    for t, (x, y) in enumerate(zip(a, b)):
        np.testing.assert_array_equal(x[0], y[0], err_msg="poses, frame %d" % t)
        assert x[1] == y[1], "summaries, frame %d" % t
        if world:
            for i in (2, 3, 4):
                np.testing.assert_array_equal(x[i], y[i], err_msg="trajectory field %d, frame %d" % (i, t))


def params(ea, **sp_kw):
    kw = dict(point_stride=1, loss_type=ea.LOSS_HUBER, loss_scale=0.1)
    kw.update(sp_kw)
    return ea.frame_params(n_levels=3), ea.solve_params(**kw)


# ---- 1. equivalence with the fixed interval -------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 2, 5])
def test_interval_policy_equals_fixed_interval(ea, ctx, K):
    """Policy {max_interval = K} against a fixed-interval-K tracker, 6 streams x 14 frames: poses and summaries bit-identical
    through stream-ordered device steps, device steps with set_inputs_ready and the pipelined host path; EA_KEY_FIRST on frame 0
    and EA_KEY_INTERVAL exactly on the frames t % K == 0."""
    bgr, depth, _ = make_seq([(1.2, 0.025)] * 6, 14, seed=11)
    fp, sp = params(ea)
    fixed = ea.Tracker(ctx, fp, sp, 6, K)
    pol = ea.Tracker(ctx, fp, sp, 6, 10)
    pol.set_keyframe_policy(max_interval=K)
    try:
        for mode in ("device", "ready", "host"):
            fixed.reset(); pol.reset()
            a = run(fixed, bgr, depth, mode, policy=False)
            b = run(pol, bgr, depth, mode)
            assert_bit_identical(a, b, world=False)
            for t, r in enumerate(b):
                want = ea.KEY_FIRST if t == 0 else (ea.KEY_INTERVAL if t % K == 0 else 0)
                assert (r[4] == want).all(), (mode, t, r[4])
                assert (r[3] == (0 if t == 0 else (t - 1) // K * K)).all(), (mode, t, r[3])
            check_composition(b)
            if mode == "device":
                dev = b
            else:
                assert_bit_identical(dev, b)
    finally:
        fixed.close(); pol.close()


# ---- 2. trajectory composition ----------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_world_trajectory_composes_and_follows_ground_truth(ea, ctx):
    """30 frames, 4 streams re-keyed by motion.  World poses equal the numpy fp64 composition of the returned poses along the
    returned key chain to 1e-12, and follow synth.relative_pose(Rw, tw, t, 0) within (1 + key switches so far) x (1 deg, 3 cm),
    the per-key bound of the tracker tests chained once per alignment.  Largest error observed on a B200: 0.96 deg and 28 mm
    (27 key switches over the 4 streams), against bounds that grow by 1 deg / 3 cm per switch."""
    import synth
    T = 30
    bgr, depth, traj = make_seq([(1.2, 0.025)] * 4, T, seed=23)
    fp, sp = params(ea)
    tr = ea.Tracker(ctx, fp, sp, 4, 10)
    tr.set_keyframe_policy(max_translation=0.08, max_rotation=math.radians(4))
    try:
        res = run(tr, bgr, depth)
    finally:
        tr.close()
    check_composition(res)
    worst = [0.0, 0.0]
    n_switch = 0
    for s, (Rw, tw) in enumerate(traj):
        chain = 1
        for t in range(1, T):
            assert not res[t][4][s] & ea.KEY_LOST, (s, t)
            ang, dt = pose_err(res[t][2][s], synth.relative_pose(Rw, tw, t, 0))
            worst = [max(worst[0], ang), max(worst[1], dt)]
            assert ang < chain * math.radians(1.0) and dt < chain * 0.03, (s, t, chain, ang, dt)
            if res[t][4][s]:
                chain += 1; n_switch += 1
    assert n_switch >= 4
    print("largest world-pose error over %d frames: %.4f deg, %.2f mm (%d key switches)" % (T, math.degrees(worst[0]), worst[1] * 1e3, n_switch))


# ---- 3. per-stream motion criteria ------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_motion_criteria_per_stream(ea, ctx):
    """Slow (0.2 deg / 5 mm per frame) and fast (1.2 deg / 25 mm) streams with max_translation = 5 cm, max_rotation = 3 deg:
    the key schedule is the host replay of the rule, streams re-key on different frames, and every pose is the replay of its
    (key, frame, warm start) pair through ctx.solve_batch (cluster_size 1 in both) within 1e-6 rad / 1e-6 m."""
    T, speeds = 16, [(0.2, 0.005), (1.2, 0.025)] * 3
    S = len(speeds)
    bgr, depth, _ = make_seq(speeds, T, seed=31)
    fp, sp = params(ea, cluster_size=1)
    tr = ea.Tracker(ctx, fp, sp, S, 10)
    rule = dict(max_translation=0.05, max_rotation=math.radians(3.0))
    tr.set_keyframe_policy(**rule)
    try:
        res = run(tr, bgr, depth)
    finally:
        tr.close()
    kf, rs = replay_rule(res, fp.n_levels, sp.finest_level, **rule)
    np.testing.assert_array_equal(np.stack([r[3] for r in res]), kf)
    np.testing.assert_array_equal(np.stack([r[4] for r in res]), rs)
    sched = {tuple(np.nonzero(rs[1:, s])[0]) for s in range(S)}
    assert len(sched) >= 2, sched
    assert (rs[1:, 1::2] != 0).sum() > (rs[1:, 0::2] != 0).sum()      # the fast streams re-key more often
    check_composition(res)
    # replay every pair through the batched solve
    fs = ea.FrameSet(ctx, fp, T * S)
    try:
        fs.preprocess_host(np.arange(T * S), bgr.cpu().numpy().reshape(T * S, H, W, 3), depth.cpu().numpy().reshape(T * S, H, W),
                           ea.ROLE_BOTH)
        refs, nows, warm, got = [], [], [], []
        for t in range(1, T):
            for s in range(S):
                refs.append(kf[t, s] * S + s); nows.append(t * S + s)
                warm.append(ea.IDENTITY if rs[t - 1, s] else res[t - 1][0][s])
                got.append(res[t][0][s])
        poses, _ = ctx.solve_batch(fs, refs, fs, nows, np.array(warm), sp)
    finally:
        fs.close()
    for i, (p, g) in enumerate(zip(poses, got)):
        ang, dt = pose_err(p, g)
        assert ang < 1e-6 and dt < 1e-6, (i, ang, dt)


# ---- 4. cost criterion ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_cost_criterion_extremes(ea, ctx):
    """A tiny positive max_cost_per_residual makes every frame a key frame (EA_KEY_COST), bit-identical to a fixed interval of
    1; a huge one never fires."""
    T, S = 8, 4
    bgr, depth, _ = make_seq([(1.2, 0.025)] * S, T, seed=41)
    fp, sp = params(ea)
    fixed = ea.Tracker(ctx, fp, sp, S, 1)
    pol = ea.Tracker(ctx, fp, sp, S, 10)
    try:
        a = run(fixed, bgr, depth, policy=False)
        pol.set_keyframe_policy(max_cost_per_residual=1e-300)
        b = run(pol, bgr, depth)
        assert_bit_identical(a, b, world=False)
        for t in range(1, T):
            assert (b[t][4] == ea.KEY_COST).all() and (b[t][3] == t - 1).all(), t
        pol.reset()
        pol.set_keyframe_policy(max_cost_per_residual=1e300)
        c = run(pol, bgr, depth)
        for t in range(1, T):
            assert (c[t][4] == 0).all() and (c[t][3] == 0).all(), t
        check_composition(b); check_composition(c)
    finally:
        fixed.close(); pol.close()


# ---- 5. lost and re-anchor ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_lost_frame_reanchors_stream(ea, ctx):
    """Stream 1's frame 0 has no valid depth: its frame 1 reports EA_TERM_SKIPPED_NO_POINTS and EA_KEY_LOST, its world pose is
    held at identity and frame 1 becomes its key frame.  From frame 2 on it follows the camera motion since frame 1 (the
    re-anchored world: frame 1 held where frame 0 was) within (1 + key switches) x (1 deg, 3 cm).  The other streams match a
    run with valid depth within 1e-6 rad / 1e-6 m (their scheduling differs, so not bit for bit)."""
    import synth
    T, S, bad = 8, 4, 1
    bgr, depth, traj = make_seq([(1.2, 0.025)] * S, T, seed=53)
    broken = depth.clone()
    broken[0, bad] = 0
    fp, sp = params(ea)
    tr = ea.Tracker(ctx, fp, sp, S, 10)
    rule = dict(max_translation=0.08, max_rotation=math.radians(4))
    try:
        tr.set_keyframe_policy(**rule)
        ok = run(tr, bgr, depth)
        tr.reset()
        lost = run(tr, bgr, broken)
    finally:
        tr.close()
    assert lost[1][1][bad * fp.n_levels + sp.finest_level][0] == 8      # EA_TERM_SKIPPED_NO_POINTS
    assert lost[1][4][bad] == ea.KEY_LOST and lost[1][3][bad] == 0
    np.testing.assert_array_equal(lost[1][2][bad], ea.IDENTITY)
    assert lost[2][3][bad] == 1
    kf, rs = replay_rule(lost, fp.n_levels, sp.finest_level, **rule)
    np.testing.assert_array_equal(np.stack([r[4] for r in lost]), rs)
    check_composition(lost)
    Rw, tw = traj[bad]
    chain = 1
    for t in range(2, T):
        ang, dt = pose_err(lost[t][2][bad], synth.relative_pose(Rw, tw, t, 1))
        assert ang < chain * math.radians(1.0) and dt < chain * 0.03, (t, ang, dt)
        chain += 1 if lost[t][4][bad] else 0
    for t in range(T):
        for s in range(S):
            if s == bad:
                continue
            for i in (0, 2):
                ang, dt = pose_err(lost[t][i][s], ok[t][i][s])
                assert ang < 1e-6 and dt < 1e-6, (t, s, i, ang, dt)
            assert lost[t][4][s] == ok[t][4][s] and lost[t][3][s] == ok[t][3][s], (t, s)


# ---- 6. gray input ------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_gray_policy_equals_replicated_bgr(ea, ctx):
    """GRAY8 frames with a policy give bit-identical poses, summaries and trajectories to BGR (g, g, g) with the same policy."""
    import torch
    T, S = 12, 4
    bgr, depth, _ = make_seq([(0.2, 0.005), (1.2, 0.025)] * 2, T, seed=61)
    b = bgr.to(torch.int64)
    gray = ((b[..., 0] * 9798 + b[..., 1] * 19235 + b[..., 2] * 3735 + 16384) >> 15).to(torch.uint8).contiguous()
    rep = gray.unsqueeze(-1).expand(*gray.shape, 3).contiguous()
    torch.cuda.synchronize()
    fp, sp = params(ea)
    tg = ea.Tracker(ctx, fp, sp, S, 10, image_format=ea.IMAGE_GRAY8)
    tb = ea.Tracker(ctx, fp, sp, S, 10)
    try:
        for tr in (tg, tb):
            tr.set_keyframe_policy(max_interval=5, max_translation=0.05, max_rotation=math.radians(3))
        for mode in ("device", "host"):
            tg.reset(); tb.reset()
            assert_bit_identical(run(tg, gray, depth, mode), run(tb, rep, depth, mode))
    finally:
        tg.close(); tb.close()


# ---- 7. errors, reset, probe, capacity --------------------------------------------------------------------------------
@pytest.mark.gpu
def test_policy_errors_reset_and_probe(ea, ctx):
    """EA_ERR_STATE: a policy after the first step, a trajectory in fixed mode, wait_trajectory outside the ring.
    EA_ERR_INVALID_ARG: NULL depth in policy mode, negative / non-finite thresholds (nothing launched).  reset keeps the policy
    and restarts the world at identity; probe_gather and EA_ERR_CAPACITY keep working in policy mode."""
    T, S = 5, 2
    bgr, depth, _ = make_seq([(1.2, 0.025)] * S, T, seed=71)
    fp, sp = params(ea)
    tr = ea.Tracker(ctx, fp, sp, S, 10)
    fi, fd = bgr[0].numel(), depth[0].numel() * 2

    def code(f, *a, **k):
        with pytest.raises(ea.EaError) as e:
            f(*a, **k)
        return e.value.code
    try:
        assert code(tr.trajectory) == 5
        assert code(tr.wait_trajectory, 0) == 5
        l0 = ctx.launch_count()
        for bad in (dict(max_interval=-1), dict(max_translation=-0.1), dict(max_rotation=float("nan")),
                    dict(max_cost_per_residual=float("inf")), dict(max_translation=float("-inf"))):
            assert code(tr.set_keyframe_policy, **bad) == 1, bad
        assert code(tr.trajectory) == 5                                     # a rejected policy leaves fixed mode on
        tr.set_keyframe_policy(max_interval=3, max_translation=0.05)
        assert code(tr.step_device, bgr.data_ptr(), 0) == 1
        hb = bgr[0].cpu().numpy()
        assert code(tr.step_host, hb.ctypes.data, 0) == 1
        assert ctx.launch_count() == l0 and tr.frame_index() == 0
        first = run(tr, bgr, depth)
        assert code(tr.set_keyframe_policy, max_interval=2) == 5
        assert code(tr.set_keyframe_policy, None) == 5
        assert code(tr.wait_trajectory, 0) == 5 and code(tr.wait_trajectory, -1) == 5
        rate, ms, n = tr.probe_gather(level=0, repeats=2)
        assert rate > 0 and n > 0
        # host path: only the last two frames stay in the ring
        tr.reset()
        again = run(tr, bgr, depth, "host")
        assert_bit_identical(first, again)
        assert code(tr.wait_trajectory, T - 3) == 5
        # reset keeps the policy and restarts the world at identity
        tr.reset()
        tr.step_device(bgr.data_ptr() + fi, depth.data_ptr() + fd)
        w, k, r = tr.trajectory()
        np.testing.assert_array_equal(w, np.tile(ea.IDENTITY, (S, 1)))
        assert (k == 0).all() and (r == ea.KEY_FIRST).all()
        tr.reset()
        assert_bit_identical(first, run(tr, bgr, depth))
        # back to the fixed interval
        tr.reset(); tr.set_keyframe_policy(None)
        assert code(tr.trajectory) == 5
    finally:
        tr.close()
    # a truncated key-frame point list is still reported
    tc = ea.Tracker(ctx, ea.frame_params(n_levels=3, max_points=500), sp, S, 10)
    try:
        tc.set_keyframe_policy(max_interval=2)
        for t in range(3):
            tc.step_device(bgr.data_ptr() + t * fi, depth.data_ptr() + t * fd)
        assert code(tc.poses) == 4                                          # EA_ERR_CAPACITY
        w, k, r = tc.trajectory()
        assert r.tolist() == [ea.KEY_INTERVAL] * S
    finally:
        tc.close()
