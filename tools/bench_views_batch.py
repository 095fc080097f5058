#!/usr/bin/env python
"""Multi-camera problems solved in one persistent launch (ea_solve_views_batch) against the same problems one at a time
(per-level ea_solve_views calls) and against the single-camera batched solver (ea_solve_batch) on the left views alone.

Inputs: synthetic stereo rigs (tools/synth.py, rendered on the GPU).  The left camera of a rig follows `trajectory`; the right
one is the left one composed with a fixed rig (0.12 m baseline, 2 degrees of yaw, synth.stereo_rig).  A problem is the motion
a -> b of one rig with two views: left -> left plain, and right -> right through the rig transform T21.  640 x 480, 3 levels,
Huber(0.1), stride 1, Ceres-default LM, solved from the identity.  Frames are preprocessed once, before any timing.

Prints one JSON line:
  batch       problems/s and point-evaluations/s of ea_solve_views_batch (kernel time from CUDA events on the context stream,
              the median over --reps calls; point-evaluations = sum over (problem, level) of evaluations x residuals)
  loop        the same for the first --loop-problems problems, one at a time, through per-level ea_solve_views calls (host
              wall clock: these calls are synchronous)
  mono        ea_solve_batch on the left views alone (kernel time from CUDA events): the single-camera point-evaluations/s
  accuracy    fraction of the problems within 1 degree / 3 cm of the true b_T_a
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.dont_write_bytecode = True
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))


def rot_deg(qa, qb):
    d = abs(float(np.dot(qa / np.linalg.norm(qa), qb / np.linalg.norm(qb))))
    return np.degrees(2.0 * np.arccos(min(1.0, d)))


def point_evals(summaries):
    return float(sum(s["evaluations"] * s["n_residuals"] for per in summaries for s in per))


def gpu_name():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=20).stdout
        return out.strip().splitlines()[0] if out.strip() else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--problems", type=int, default=1184)
    ap.add_argument("--rigs", type=int, default=64, help="distinct rigs (each with its own scene and trajectory)")
    ap.add_argument("--frames", type=int, default=6, help="frames per rig; problems are pairs a -> b with 1 <= |b - a| <= 2")
    ap.add_argument("--loop-problems", type=int, default=64)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--seed", type=int, default=3)
    a = ap.parse_args()
    import torch
    import synth
    import edge_alignment_b200 as ea
    if not torch.cuda.is_available():
        raise SystemExit("bench_views_batch: no CUDA device (the solver has no CPU path)")
    ctx = ea.Context(0)
    fp = ea.frame_params(n_levels=3)
    R, T = a.rigs, a.frames
    left = ea.FrameSet(ctx, fp, R * T)
    right = ea.FrameSet(ctx, fp, R * T)
    traj, rigs = [], []
    t0 = time.perf_counter()
    for r in range(R):
        seed = a.seed * 100003 + r
        Rw, tw = synth.trajectory(T, seed)
        Rw2, tw2, T21 = synth.stereo_rig(Rw, tw)
        for fs, (Rc, tc) in ((left, (Rw, tw)), (right, (Rw2, tw2))):
            b, d = synth.render(Rc, tc, seed, device="cuda")
            torch.cuda.synchronize()
            fs.preprocess_device(list(range(r * T, (r + 1) * T)), b.data_ptr(), d.data_ptr(), ea.ROLE_BOTH)
            ctx.sync()
        traj.append((Rw, tw)); rigs.append(T21)
    prep_s = time.perf_counter() - t0
    pairs = [(r, i, j) for r in range(R) for i in range(T) for j in range(T) if 1 <= abs(i - j) <= 2]
    chosen = [pairs[k % len(pairs)] for k in range(a.problems)]
    problems = [[dict(ref=left, ref_slot=r * T + i, now=left, now_slot=r * T + j),
                 dict(ref=right, ref_slot=r * T + i, now=right, now_slot=r * T + j, T21=rigs[r])] for r, i, j in chosen]
    gts = [synth.relative_pose(traj[r][0], traj[r][1], i, j) for r, i, j in chosen]
    sp = ea.solve_params(point_stride=1, loss_type=ea.LOSS_HUBER, loss_scale=0.1)
    n = len(problems)

    # ---- batched: one launch for every problem ----
    ctx.solve_views_batch(problems, None, sp)                          # warm-up (modules, scratch)
    ctx.profile_enable(True)
    ctx.profile_read()
    ms, wall = [], []
    for _ in range(a.reps):
        w0 = time.perf_counter()
        poses, S = ctx.solve_views_batch(problems, None, sp)
        wall.append(time.perf_counter() - w0)
        ms.append(ctx.profile_read()["solve_ms"])
    batch_ms = float(np.median(ms))
    pe = point_evals(S)
    ok = [rot_deg(p[:4], g[:4]) < 1.0 and np.abs(p[4:] - g[4:]).max() < 0.03 for p, g in zip(poses, gts)]

    # ---- one problem at a time, level by level through ea_solve_views ----
    m = min(a.loop_problems, n)
    ctx.profile_enable(False)
    ctx.solve_views(problems[0], None, sp, level=2)                    # warm-up
    w0 = time.perf_counter()
    loop_pe = 0.0
    loop_poses = []
    for k in range(m):
        pose = np.array(ea.IDENTITY)
        for level in (2, 1, 0):
            pose, s = ctx.solve_views(problems[k], pose, sp, level=level)
            loop_pe += s["evaluations"] * s["n_residuals"]
        loop_poses.append(pose)
    loop_s = time.perf_counter() - w0
    loop_dev = max(max(rot_deg(p[:4], q[:4]), np.abs(p[4:] - q[4:]).max()) for p, q in zip(loop_poses, poses[:m]))

    # ---- mono reference: the left views alone through ea_solve_batch ----
    rs = np.array([p[0]["ref_slot"] for p in problems], np.int32)
    ns = np.array([p[0]["now_slot"] for p in problems], np.int32)
    ctx.solve_batch(left, rs, left, ns, None, sp)
    ctx.profile_enable(True)
    ctx.profile_read()
    mms = []
    for _ in range(a.reps):
        _, MS = ctx.solve_batch(left, rs, left, ns, None, sp)
        mms.append(ctx.profile_read()["solve_ms"])
    mono_ms = float(np.median(mms))
    mono_pe = point_evals(MS)

    out = {
        "metric": "multi-camera problems/sec (stereo rigs, 2 views, 640x480, 3 levels)",
        "gpu": gpu_name(),
        "problems": n, "rigs": R, "frames_per_rig": T, "preprocess_s": round(prep_s, 2),
        "batch": {"kernel_ms": round(batch_ms, 3), "kernel_ms_all": [round(x, 3) for x in ms], "call_ms": round(1e3 * float(np.median(wall)), 3),
                  "problems_per_s": round(n / (batch_ms * 1e-3), 1), "point_evals_per_s": float("%.4g" % (pe / (batch_ms * 1e-3))),
                  "point_evals": pe},
        "loop": {"problems": m, "wall_ms": round(1e3 * loop_s, 2), "problems_per_s": round(m / loop_s, 1),
                 "point_evals_per_s": float("%.4g" % (loop_pe / loop_s)), "max_pose_diff_vs_batch": float("%.3g" % loop_dev)},
        "mono": {"kernel_ms": round(mono_ms, 3), "pairs_per_s": round(n / (mono_ms * 1e-3), 1),
                 "point_evals_per_s": float("%.4g" % (mono_pe / (mono_ms * 1e-3)))},
        "speedup_batch_vs_loop": round((n / (batch_ms * 1e-3)) / (m / loop_s), 1),
        "batch_point_evals_vs_mono": round((pe / batch_ms) / (mono_pe / mono_ms), 3),
        "within_1deg_3cm": round(float(np.mean(ok)), 4),
    }
    print(json.dumps(out))
    left.close(); right.close(); ctx.close()


if __name__ == "__main__":
    main()
