#!/usr/bin/env python
"""Tracker key-frame policy mode against the fixed interval, on the default bench.py workload.

Workload: bench.py's default line -- 1 184 camera streams, 640 x 480, 3 pyramid levels, Huber(0.1), stride 1 -- on synthetic
sequences (tools/synth.make_sequences) fed as 8-bit gray frames, as tools/bench_gray.py does.  Three arms:
  fixed      ea_tracker_create's fixed schedule, a key frame every 10 frames
  interval   key-frame policy {max_interval = 10}: the same schedule decided on the device, per stream
  motion     key-frame policy with translation / rotation thresholds only, scaled before timing (a short untimed sweep) so that
             it re-keys about as often as the other two arms
The policy arms preprocess every frame for both roles and upload depth with every frame; the fixed arm does both only for
key frames.  The script fails unless the interval arm's poses, summaries and key schedule equal the fixed arm's bit for bit,
step by step (resident path) and frame by frame (host path).  At 1 184 streams this also covers the two-lane preprocessing.

The arms alternate within one call, --runs times each.  Per arm it reports the median over runs of
  resident     alignments/s with frames resident in HBM (ea_tracker_step_device, stream-ordered as bench.py's value)
  e2e          alignments/s with every step's frames uploaded from pinned host memory (ea_tracker_step_host, pipelined with
               ea_tracker_wait as bench.py's e2e leg)
  preprocess   device ms per step of the preprocessing pipeline in the resident run (ea_profile_read)
  launches     kernel launches per step (ea_launch_count)
  h2d          bytes uploaded per step by the host path
  key_rate     key frames per stream and step
plus the card's name, power limit and SM clocks, read in the same call.
"""
import argparse
import json
import math
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.dont_write_bytecode = True
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_gray import gpu_info, ring_index   # noqa: E402

W, H, N_LEVELS, HUBER_A, INTERVAL = 640, 480, 3, 0.1, 10   # bench.py's default line


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--streams", type=int, default=1184)
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--frames", type=int, default=6, help="distinct frames per stream (walked forwards and backwards)")
    ap.add_argument("--seed", type=int, default=1234)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_keyframes.py: no CUDA device; the product path has no CPU fallback")
    import edge_alignment_b200 as ea
    import synth

    S, K, Wm, NF = a.streams, a.steps, max(a.warmup, 3), a.frames
    T = Wm + K + 1
    dev = torch.device("cuda", 0)
    bgr_src, depth_d, _ = synth.make_sequences(S, NF, seed=a.seed, device=dev)
    b = bgr_src.to(torch.int32)
    gray_d = ((b[..., 0] * 9798 + b[..., 1] * 19235 + b[..., 2] * 3735 + 16384) >> 15).to(torch.uint8).contiguous()
    del b, bgr_src
    depth_d = depth_d.contiguous()
    gray_h, depth_h = gray_d.cpu().pin_memory(), depth_d.cpu().pin_memory()
    fb, fd = W * H * S, W * H * 2 * S
    torch.cuda.synchronize()

    ctx = ea.Context(0)
    stream = torch.cuda.current_stream()
    ctx.set_stream(stream.cuda_stream)
    fp = ea.frame_params(n_levels=N_LEVELS)
    sp = ea.solve_params(point_stride=1, loss_type=ea.LOSS_HUBER, loss_scale=HUBER_A)
    mk = lambda: ea.Tracker(ctx, fp, sp, S, INTERVAL, image_format=ea.IMAGE_GRAY8)
    arms = {"fixed": dict(tracker=mk(), policy=None), "interval": dict(tracker=mk(), policy=dict(max_interval=INTERVAL)),
            "motion": dict(tracker=mk(), policy=None)}
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    dev_frame = lambda t: (gray_d.data_ptr() + ring_index(t, NF) * fb, depth_d.data_ptr() + ring_index(t, NF) * fd)

    def start(arm):
        tr = arm["tracker"]
        tr.reset()
        if arm["policy"]:
            tr.set_keyframe_policy(**arm["policy"])
        else:
            tr.set_keyframe_policy(None)

    def key_rate(arm, steps):
        """Key frames per stream and step over frames 1..steps (resident, untimed)."""
        start(arm)
        tr, n = arm["tracker"], 0
        for t in range(steps + 1):
            tr.step_device(*dev_frame(t))
            if t > 0:
                n += int((tr.trajectory()[2] != 0).sum())
        return n / (S * steps)

    # motion arm: thresholds (s * 2 cm, s * 1 deg), s chosen by a geometric sweep for the key rate closest to 1 / INTERVAL
    best = None
    for s in (3.0, 4.0, 5.0, 6.0, 8.0, 10.0, 12.0):
        arms["motion"]["policy"] = dict(max_translation=0.02 * s, max_rotation=math.radians(1.0) * s)
        r = key_rate(arms["motion"], 30)
        if best is None or abs(r - 1.0 / INTERVAL) < abs(best[1] - 1.0 / INTERVAL):
            best = (s, r)
    arms["motion"]["policy"] = dict(max_translation=0.02 * best[0], max_rotation=math.radians(1.0) * best[0])

    # correctness first: the interval arm against the fixed arm, every step of the resident path
    for name in ("fixed", "interval"):
        start(arms[name])
        arms[name]["check"] = []
        for t in range(T):
            tr = arms[name]["tracker"]
            tr.step_device(*dev_frame(t))
            p, Ss = tr.poses()
            arms[name]["check"].append((p, bytes(Ss), tr.trajectory()[2].copy() if name == "interval" else None))
    for t, (x, y) in enumerate(zip(arms["fixed"]["check"], arms["interval"]["check"])):
        want = ea.KEY_FIRST if t == 0 else (ea.KEY_INTERVAL if t % INTERVAL == 0 else 0)
        if not (np.array_equal(x[0], y[0]) and x[1] == y[1] and (y[2] == want).all()):
            raise SystemExit("bench_keyframes.py: interval arm differs from the fixed arm at step %d" % t)

    def run_arm(name):
        arm = arms[name]
        tr, pol = arm["tracker"], arm["policy"] is not None
        start(arm)
        for t in range(Wm + 1):
            tr.step_device(*dev_frame(t))
        torch.cuda.synchronize()
        ctx.profile_enable(True); ctx.profile_read()
        l0 = ctx.launch_count()
        e0.record(stream)
        for t in range(Wm + 1, T):
            tr.step_device(*dev_frame(t))
        e1.record(stream)
        torch.cuda.synchronize()
        ms_res = e0.elapsed_time(e1)
        launches = (ctx.launch_count() - l0) / K
        prof = ctx.profile_read(); ctx.profile_enable(False)
        # e2e: pinned host frames through the host entry point, frame t submitted before frame t-1's results are read
        start(arm)
        hframe = lambda t: (gray_h.data_ptr() + ring_index(t, NF) * fb, depth_h.data_ptr() + ring_index(t, NF) * fd)
        for t in range(Wm + 1):
            tr.step_host(*hframe(t), fetch=True)
        torch.cuda.synchronize()
        e2e = []
        keys = 0
        e0.record(stream)
        for t in range(Wm + 1, T):
            tr.step_host(*hframe(t), fetch=False)
            if t > Wm + 1:
                p, Ss = tr.wait(t - 1)
                e2e.append((p, bytes(Ss)))
                if pol:
                    keys += int((tr.wait_trajectory(t - 1)[2] != 0).sum())
        p, Ss = tr.wait(T - 1)
        e1.record(stream)
        torch.cuda.synchronize()
        e2e.append((p, bytes(Ss)))
        if pol:
            keys += int((tr.wait_trajectory(T - 1)[2] != 0).sum())
        else:
            keys = S * sum(1 for t in range(Wm + 1, T) if t % INTERVAL == 0)
        ms_e2e = e0.elapsed_time(e1)
        n_depth = K if pol else sum(1 for t in range(Wm + 1, T) if t % INTERVAL == 0)
        arm.setdefault("runs", []).append(dict(
            resident=S * K / (ms_res * 1e-3), e2e=S * K / (ms_e2e * 1e-3),
            preprocess_ms_per_step=prof["preprocess_ms"] / K, launches_per_step=launches,
            h2d_bytes_per_step=(fb * K + fd * n_depth) / K, key_rate=keys / (S * K), _e2e=e2e))

    for _ in range(a.runs):
        for name in arms:
            run_arm(name)
    clocks = gpu_info()
    for i, (x, y) in enumerate(zip(arms["fixed"]["runs"], arms["interval"]["runs"])):
        for f, (u, v) in enumerate(zip(x["_e2e"], y["_e2e"])):
            if not (np.array_equal(u[0], v[0]) and u[1] == v[1]):
                raise SystemExit("bench_keyframes.py: run %d host-path frame %d of the interval arm differs from the fixed arm" % (i, f))

    out = {"workload": "tracker, %d streams, %dx%d gray, %d levels, Huber(%g), stride 1; %d timed steps after %d warm-up, %d distinct "
                       "frames per stream" % (S, W, H, N_LEVELS, HUBER_A, K, Wm, NF),
           "gpu": "name, power.limit, clocks.sm, clocks.max.sm = " + clocks, "runs": a.runs, "interval_equals_fixed": True,
           "motion_policy": dict(arms["motion"]["policy"], sweep_scale=best[0], sweep_key_rate=best[1])}
    for name, arm in arms.items():
        keys_ = [k for k in arm["runs"][0] if not k.startswith("_")]
        out[name] = {k: float(np.median([r[k] for r in arm["runs"]])) for k in keys_}
        out[name]["resident_runs"] = [round(r["resident"]) for r in arm["runs"]]
        out[name]["e2e_runs"] = [round(r["e2e"]) for r in arm["runs"]]
        arm["tracker"].close()
    for name in ("interval", "motion"):
        out[name + "_over_fixed"] = {k: out[name][k] / out["fixed"][k] for k in ("resident", "e2e", "preprocess_ms_per_step")}
    ctx.close()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
