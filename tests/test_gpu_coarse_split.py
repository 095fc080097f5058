"""Coarse / fine split of the batched solve: big batches solve the coarse pyramid levels in CTAs of EA_SOLVE_COARSE_THREADS
threads (several per SM) and the finest level in the full-width kernel. The narrower CTA evaluates as a virtual CTA of the
full width, so poses and summaries are bit-identical to the single launch. A batch below the split threshold (2 x SMs pairs)
or with one level runs the single launch, so the reference here is the same pairs solved in batches below the threshold."""
import os
import re
import subprocess
import sys
import tempfile

import numpy as np
import pytest

from conftest import ROOT

CHUNK = 100          # pairs per reference batch: below the split threshold on any GPU with more than 50 SMs


def _sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _solve_pairs(ctx, fs, pairs, starts, sp, chunk=None):
    """Poses and per-level summaries of the pairs, solved in batches of `chunk` pairs (all at once by default) through the
    device entry point (the host one refuses truncated point lists)."""
    import ctypes
    import torch
    from edge_alignment_b200 import _lib as L
    n, nl = len(pairs), fs.params.n_levels
    step = chunk or n
    ssz = ctypes.sizeof(L.Summary)
    poses = torch.tensor(np.asarray(starts, np.float64), device="cuda")
    summ = torch.zeros(n * nl * ssz, dtype=torch.uint8, device="cuda")
    rs = torch.tensor([a for a, _ in pairs], dtype=torch.int32, device="cuda")
    ns = torch.tensor([b for _, b in pairs], dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    for i in range(0, n, step):
        m = min(step, n - i)
        ctx.solve_batch_device(m, fs, rs[i:].data_ptr(), fs, ns[i:].data_ptr(), poses[i:].data_ptr(), sp,
                               d_summaries=summ[i * nl * ssz:].data_ptr())
    ctx.sync()
    raw = summ.cpu().numpy().tobytes()
    S = [[L.Summary.from_buffer_copy(raw, (i * nl + l) * ssz).asdict() for l in range(nl)] for i in range(n)]
    return poses.cpu().numpy(), S


def _pairs(n_frames, n, seed):
    rng = np.random.default_rng(seed)
    base = [(a, b) for a in range(n_frames) for b in range(n_frames)]
    pairs = [base[i % len(base)] for i in range(n)]
    starts = np.tile(np.array([1.0, 0, 0, 0, 0, 0, 0]), (n, 1))
    starts[:, 4:] = rng.normal(0.0, 0.01, (n, 3))                  # every pair its own warm start
    return pairs, starts


def _assert_identical(got, ref):
    (gp, gs), (rp, rs) = got, ref
    np.testing.assert_array_equal(gp, rp)
    assert gs == rs


@pytest.fixture(scope="module")
def ea():
    import edge_alignment_b200 as ea
    return ea


@pytest.fixture(scope="module")
def ctx(ea):
    c = ea.Context(0)
    yield c
    c.close()


def _frameset(ea, ctx, frames, n_levels, max_points=0, flat=False):
    fs = ea.FrameSet(ctx, ea.frame_params(n_levels=n_levels, max_points=max_points), 6)
    fs.preprocess_host(np.arange(5), frames["bgr"], frames["depth"], ea.ROLE_BOTH)
    if flat:     # slot 5: no edges at all, so no reference points at any level (SKIPPED_NO_POINTS)
        fs.preprocess_host([5], np.full((1, 480, 640, 3), 128, np.uint8), np.full((1, 480, 640), 5000, np.uint16), ea.ROLE_BOTH)
    return fs


@pytest.mark.gpu
@pytest.mark.parametrize("n_levels", [1, 2, 4])
@pytest.mark.parametrize("loss,stride,strategy", [("huber", 1, 0), ("cauchy", 30, 0), ("trivial", 30, 0), ("huber", 30, 1)])
def test_split_matches_single_launch(ea, ctx, frames, n_levels, loss, stride, strategy):
    losses = {"huber": (ea.LOSS_HUBER, 0.1), "cauchy": (ea.LOSS_CAUCHY, 1.0), "trivial": (ea.LOSS_TRIVIAL, 1.0)}
    lt, ls = losses[loss]
    sp = ea.solve_params(point_stride=stride, loss_type=lt, loss_scale=ls, trust_region_strategy=strategy, cluster_size=1)
    fs = _frameset(ea, ctx, frames, n_levels)
    try:
        for n in ((2 * _sm_count(), 1184) if stride > 1 else (2 * _sm_count(),)):
            pairs, starts = _pairs(5, n, seed=n)
            _assert_identical(_solve_pairs(ctx, fs, pairs, starts, sp), _solve_pairs(ctx, fs, pairs, starts, sp, CHUNK))
    finally:
        fs.close()


@pytest.mark.gpu
def test_split_skipped_levels_truncated_lists_and_xyz_points(ea, ctx, frames, oracle):
    sp = ea.solve_params(point_stride=3, loss_type=ea.LOSS_HUBER, loss_scale=0.1, cluster_size=1)
    n = 2 * _sm_count() + 7
    # a reference frame without points at any level, and point lists truncated at their capacity
    fs = _frameset(ea, ctx, frames, 3, max_points=3000, flat=True)
    try:
        pairs, starts = _pairs(6, n, seed=1)
        got = _solve_pairs(ctx, fs, pairs, starts, sp)
        assert any(s[2]["termination_name"] == "SKIPPED_NO_POINTS" for s in got[1])
        assert any(s[0]["truncated"] for s in got[1])
        _assert_identical(got, _solve_pairs(ctx, fs, pairs, starts, sp, CHUNK))
    finally:
        fs.close()
    # fp32 XYZ point streams at every level
    fs = _frameset(ea, ctx, frames, 2)
    try:
        for s in range(5):
            xyz, _ = oracle.get_aX(frames["bgr"][s], frames["depth"][s], frames["K"])
            p4 = np.ones((len(xyz), 4), np.float32); p4[:, :3] = xyz
            for level in range(2):
                fs.set_points(s, p4[::4 ** level], level=level, mode=ea.POINTS_XYZ)
        pairs, starts = _pairs(5, n, seed=2)
        _assert_identical(_solve_pairs(ctx, fs, pairs, starts, sp), _solve_pairs(ctx, fs, pairs, starts, sp, CHUNK))
    finally:
        fs.close()


@pytest.mark.gpu
@pytest.mark.parametrize("ready", [False, True])
def test_split_tracker_across_key_frame_switches(ea, ctx, ready):
    """A tracker over 2 x SMs streams (split; declared-complete inputs also turn the tail helpers off) against the same
    streams in two trackers below the split threshold, across key-frame switches."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import synth
    S, T = 2 * _sm_count(), 5
    bgr, depth, _ = synth.make_sequences(S, T, seed=3, device="cuda")
    torch.cuda.synchronize()
    fp, sp = ea.frame_params(n_levels=3), ea.solve_params(point_stride=4, loss_type=ea.LOSS_HUBER, loss_scale=0.1)

    def run(lo, hi):
        b = bgr[:, lo:hi].contiguous(); d = depth[:, lo:hi].contiguous()
        fb, fd = b[0].numel(), d[0].numel() * 2
        tr = ea.Tracker(ctx, fp, sp, hi - lo, 2)
        try:
            tr.set_inputs_ready(ready)
            out = []
            for t in range(T):
                tr.step_device(b.data_ptr() + t * fb, d.data_ptr() + t * fd)
                out.append(tr.poses()[0].copy())
            return np.stack(out)
        finally:
            tr.close()

    whole = run(0, S)
    halves = np.concatenate([run(0, S // 2), run(S // 2, S)], axis=1)
    np.testing.assert_array_equal(whole, halves)


def test_narrow_solve_kernel_evaluation_loop_has_no_local_memory():
    """The coarse-phase kernel ea_k_solve_batch<EA_SOLVE_COARSE_THREADS, false> runs the evaluation loop of the full-width
    kernel in a narrower CTA; like the full-width kernel's, that loop (the innermost loop around the staging cp.async) must
    not touch local memory."""
    from edge_alignment_b200 import build
    try:
        nvcc = build.nvcc()
    except RuntimeError:
        pytest.skip("nvcc not found")
    cuobjdump = os.path.join(os.path.dirname(nvcc), "cuobjdump") if os.path.isabs(nvcc) else "cuobjdump"
    with tempfile.TemporaryDirectory() as tmp:
        obj = os.path.join(tmp, "ea_solve.o")
        p = subprocess.run([nvcc] + build.NVCC_FLAGS + ["-c", os.path.join(build.CSRC, "ea_solve.cu"), "-o", obj],
                           stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        if p.returncode != 0 and not os.path.exists(nvcc):
            pytest.skip("nvcc not runnable")
        assert p.returncode == 0, p.stdout[-4000:]
        for threads in (256, 512):
            fn = "_Z16ea_k_solve_batchILi%dELb0EEv11EaSolveArgs" % threads
            sass = subprocess.run([cuobjdump, "-sass", "-fun", fn, obj], stdout=subprocess.PIPE, text=True, check=True).stdout
            loops = _staging_loops(sass)
            assert loops, "%s: no evaluation loop found" % fn
            for body in loops:
                bad = [t for t in body if re.match(r"(@!?P\d+\s+)?(LDL|STL)\b", t)]
                assert not bad, "%s: local memory in the evaluation loop: %s" % (fn, bad[:4])


def _staging_loops(sass):
    """Instruction lists of the innermost loops that contain a predicated LDGSTS (the per-iteration point prefetch)."""
    ins = []
    for line in sass.splitlines():
        m = re.match(r"\s*/\*([0-9a-f]{4,})\*/\s+(.*?)\s*;", line)
        if m:
            ins.append((int(m.group(1), 16), m.group(2)))
    branches = []
    for a, t in ins:
        m = re.search(r"\bBRA\b.*?(0x[0-9a-f]+)$", t)
        if m and int(m.group(1), 16) <= a:
            branches.append((int(m.group(1), 16), a))
    loops = []
    for s, t in ins:
        if "LDGSTS" not in t or not t.startswith("@"):
            continue
        enclosing = [(lo, hi) for lo, hi in branches if lo <= s < hi]
        if enclosing:
            lo, hi = min(enclosing, key=lambda b: b[1] - b[0])
            loops.append([u for a, u in ins if lo <= a <= hi])
    return loops
