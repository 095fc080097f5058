"""Multi-GPU paths (SURVEY.md 8e).  Single-GPU parts always run with -m gpu; the NCCL part needs >= 2 devices
and is skipped otherwise."""
import os
import sys

import numpy as np
import pytest

from conftest import IDENTITY, ROOT, rot_angle_between

pytestmark = pytest.mark.gpu


def test_pair_shards_are_independent(frames):
    """configs[2] at small scale: solving contiguous blocks of a batch separately (what each rank does) gives the very
    same poses as solving the whole batch at once -- no data-path collective is needed."""
    import edge_alignment_b200 as ea
    from edge_alignment_b200 import sharding
    ctx = ea.Context(0)
    fs = ea.FrameSet(ctx, ea.frame_params(), 5)
    try:
        fs.preprocess_host(np.arange(5), frames["bgr"], frames["depth"], ea.ROLE_BOTH)
        pairs = [(a, b) for a in range(5) for b in range(5) if a != b] * 3
        ref = np.array([p[0] for p in pairs]); now = np.array([p[1] for p in pairs])
        sp = ea.solve_params(point_stride=5, cluster_size=1)
        whole, _ = ctx.solve_batch(fs, ref, fs, now, None, sp)
        for world in (2, 4, 8):
            parts = []
            for r in range(world):
                rr, nn = sharding.shard_pairs(ref, now, r, world)
                parts.append(ctx.solve_batch(fs, rr, fs, nn, None, sp)[0])
            np.testing.assert_array_equal(np.concatenate(parts), whole)
    finally:
        fs.close(); ctx.close()


@pytest.mark.parametrize("mode", ["kernel", "nccl"])
def test_point_sharded_solve_single_rank(frames, solver_golden, mode, monkeypatch):
    """ea_shard_solve with world == 1: the persistent cooperative kernel (grid reduce + LM inside the kernel, 2 launches per
    solve) and the host-driven launch loop (EA_SHARD_MODE=nccl) == the batched solver; a second solve on the same shard
    reuses its control block and reproduces the first bit for bit."""
    import ctypes as C
    import edge_alignment_b200 as ea
    from edge_alignment_b200 import _lib as L
    monkeypatch.setenv("EA_SHARD_MODE", mode)
    ctx = ea.Context(0)
    fs = ea.FrameSet(ctx, ea.frame_params(), 2)
    try:
        fs.preprocess_host([0, 1], frames["bgr"][[0, 2]], frames["depth"][[0, 2]], ea.ROLE_BOTH)
        sh = C.c_void_p()
        assert L.lib().ea_shard_create(ctx._h, None, 0, 1, C.byref(sh)) == 0
        g = solver_golden["pose_1_3_cauchy_stride1"]; gs = solver_golden["summary_1_3_cauchy_stride1"]
        got = []
        for _ in range(2):
            pose = IDENTITY.copy(); s = L.Summary(); sp = ea.solve_params(point_stride=1)
            rc = L.lib().ea_shard_solve(sh, fs._h, 0, fs._h, 1, 0, pose.ctypes.data_as(C.POINTER(C.c_double)), C.byref(sp), C.byref(s))
            assert rc == 0, L.lib().ea_last_error()
            assert rot_angle_between(pose[:4], g[:4]) < 1e-4 and np.abs(pose[4:] - g[4:]).max() < 1e-4
            assert s.termination == int(gs[5]) and abs(s.iterations - int(gs[2])) <= 2 and s.n_residuals == 44458
            prof = (C.c_double * 8)()
            assert L.lib().ea_shard_profile(sh, prof) == 0
            assert prof[0] == s.evaluations and prof[1] > 0 and prof[6] == (1.0 if mode == "kernel" else 0.0)
            if mode == "kernel":
                assert prof[7] == 2 and prof[2] > 0 and prof[5] > 0        # two launches for the whole solve; timed sections ran
            got.append((pose.copy(), s.iterations, s.final_cost))
        assert np.array_equal(got[0][0], got[1][0]) and got[0][1:] == got[1][1:]
        # invalid solve parameters are refused here as everywhere else
        bad = ea.solve_params(point_stride=1); bad.loss_scale = 0.0
        assert L.lib().ea_shard_solve(sh, fs._h, 0, fs._h, 1, 0, pose.ctypes.data_as(C.POINTER(C.c_double)), C.byref(bad), C.byref(s)) == 1      # EA_ERR_INVALID_ARG
        L.lib().ea_shard_destroy(sh)
    finally:
        fs.close(); ctx.close()


def _nccl_worker(rank, world, port, q, mode="kernel"):
    import ctypes as C
    os.environ["EA_SHARD_MODE"] = mode
    import torch
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("gloo", rank=rank, world_size=world)       # only to pass the NCCL id around
    import edge_alignment_b200 as ea
    from edge_alignment_b200 import _lib as L
    z = np.load(os.path.join(ROOT, "tests", "golden", "frames.npz"))
    ctx = ea.Context(rank)
    fs = ea.FrameSet(ctx, ea.frame_params(), 2)
    fs.preprocess_host([0, 1], z["bgr"][[0, 2]], z["depth"][[0, 2]], ea.ROLE_BOTH)   # DT replicated on every rank
    ident = torch.zeros(128, dtype=torch.uint8)
    if rank == 0:
        buf = (C.c_uint8 * 128)()
        assert L.lib().ea_shard_unique_id(buf) == 0
        ident = torch.tensor(list(buf), dtype=torch.uint8)
    dist.broadcast(ident, 0)
    idbuf = (C.c_uint8 * 128)(*ident.tolist())
    sh = C.c_void_p()
    assert L.lib().ea_shard_create(ctx._h, idbuf, rank, world, C.byref(sh)) == 0, L.lib().ea_last_error()
    pose = np.array([1.0, 0, 0, 0, 0, 0, 0]); s = L.Summary(); sp = ea.solve_params(point_stride=1)
    rc = L.lib().ea_shard_solve(sh, fs._h, 0, fs._h, 1, 0, pose.ctypes.data_as(C.POINTER(C.c_double)), C.byref(sp), C.byref(s))
    prof = (C.c_double * 8)()
    L.lib().ea_shard_profile(sh, prof)
    # a second solve on the same shard (epochs continue) from a different start
    pose2 = np.array([0.9999875, 0.005, 0.0, 0.0, 0.01, 0.0, 0.0]); pose2[:4] /= np.linalg.norm(pose2[:4]); s2 = L.Summary()
    rc2 = L.lib().ea_shard_solve(sh, fs._h, 0, fs._h, 1, 0, pose2.ctypes.data_as(C.POINTER(C.c_double)), C.byref(sp), C.byref(s2))
    q.put((rank, rc | rc2, pose.tolist(), s.iterations, s.final_cost, list(prof), pose2.tolist()))
    L.lib().ea_shard_destroy(sh)
    dist.destroy_process_group()


@pytest.mark.parametrize("mode", ["kernel", "nccl"])
def test_point_sharded_solve_nccl_two_ranks(solver_golden, mode):
    """Two ranks, each with half of the ordered point list: the in-kernel all-reduce over peer-mapped NVLink memory
    ("kernel") and the ncclAllReduce-per-evaluation loop ("nccl") both land on the single-GPU result, with bit-identical
    poses and decisions on the two ranks."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29600 + (os.getpid() % 2000) + (7 if mode == "nccl" else 0)
    procs = [ctx.Process(target=_nccl_worker, args=(r, 2, port, q, mode)) for r in range(2)]
    [p.start() for p in procs]
    out = sorted(q.get(timeout=300) for _ in range(2))
    [p.join(timeout=120) for p in procs]
    g = solver_golden["pose_1_3_cauchy_stride1"]
    for rank, rc, pose, its, cost, prof, pose2 in out:
        pose = np.array(pose); pose2 = np.array(pose2)
        assert rc == 0
        assert rot_angle_between(pose[:4], g[:4]) < 1e-4 and np.abs(pose[4:] - g[4:]).max() < 1e-4
        assert rot_angle_between(pose2[:4], g[:4]) < 2e-4 and np.abs(pose2[4:] - g[4:]).max() < 2e-4    # same optimum from the other start
        assert prof[6] == (1.0 if mode == "kernel" else 0.0)
    assert out[0][2] == out[1][2] and out[0][3] == out[1][3] and out[0][6] == out[1][6]      # bit-identical decisions on every rank
    print("point-sharded 2 ranks [%s]: %d evaluations, %.3f ms per solve, per evaluation: eval %.1f us, reduce %.1f us, all-reduce %.1f us, LM %.1f us"
          % (mode, out[0][5][0], out[0][5][1], out[0][5][2], out[0][5][3], out[0][5][4], out[0][5][5]))
