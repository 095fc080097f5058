#!/usr/bin/env python
"""8-bit gray input against BGR input through the tracker, on the default bench.py workload.

Workload: bench.py's default line -- 1 184 camera streams, 640 x 480, 3 pyramid levels, Huber(0.1), stride 1, a key frame every
10 frames -- on synthetic sequences (tools/synth.make_sequences) converted to gray with OpenCV's 15-bit RGB2GRAY formula.  The
gray arm feeds those frames as EA_IMAGE_GRAY8; the BGR arm feeds the same frames replicated to three channels.  The two arms
therefore compute the same thing, and the script fails unless their poses and summaries are bit-identical.

The arms alternate within one call, --runs times each.  Per arm it reports the median over runs of
  resident     alignments/s with frames resident in HBM (ea_tracker_step_device, stream-ordered as bench.py's value)
  e2e          alignments/s with every step's frames uploaded from pinned host memory (ea_tracker_step_host, pipelined with
               ea_tracker_wait as bench.py's e2e leg)
  preprocess   device ms per step of the preprocessing pipeline in the resident run (ea_profile_read)
  h2d          bytes uploaded per step (images every step, depth on key frames), and the ceiling: the same uploads from the
               same pinned buffers with no kernels running, as GB/s and as the alignments/s they would allow
plus the card's name, power limit and SM clocks, read in the same call.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.dont_write_bytecode = True
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

W, H, N_LEVELS, HUBER_A, KEYFRAME_INTERVAL = 640, 480, 3, 0.1, 10   # bench.py's default line


def ring_index(t, n):
    """bench.py's walk over n distinct frames: 0, 1, .., n-1, n-2, .., 1, 0, 1, .."""
    if n <= 1:
        return 0
    p = t % (2 * n - 2)
    return p if p < n else 2 * n - 2 - p


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=20).stdout
        return out.strip().splitlines()[0] if out.strip() else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


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
        raise SystemExit("bench_gray.py: no CUDA device; the product path has no CPU fallback")
    import edge_alignment_b200 as ea
    import synth

    S, K, Wm, NF = a.streams, a.steps, max(a.warmup, 3), a.frames
    T = Wm + K + 1
    dev = torch.device("cuda", 0)
    bgr_src, depth_d, _ = synth.make_sequences(S, NF, seed=a.seed, device=dev)
    b = bgr_src.to(torch.int32)
    gray_d = ((b[..., 0] * 9798 + b[..., 1] * 19235 + b[..., 2] * 3735 + 16384) >> 15).to(torch.uint8).contiguous()
    del b, bgr_src
    rep_d = gray_d.unsqueeze(-1).expand(*gray_d.shape, 3).contiguous()
    depth_d = depth_d.contiguous()
    frame_d = W * H * 2 * S
    keys = sorted({ring_index(t, NF) for t in range(T) if t % KEYFRAME_INTERVAL == 0})
    hd = {f: depth_d[f].cpu().pin_memory() for f in keys}
    arms = {
        "bgr": dict(fmt=ea.IMAGE_BGR8, dev=rep_d, host=rep_d.cpu().pin_memory(), frame_b=W * H * 3 * S),
        "gray": dict(fmt=ea.IMAGE_GRAY8, dev=gray_d, host=gray_d.cpu().pin_memory(), frame_b=W * H * S),
    }
    torch.cuda.synchronize()

    ctx = ea.Context(0)
    stream = torch.cuda.current_stream()
    ctx.set_stream(stream.cuda_stream)
    fp = ea.frame_params(n_levels=N_LEVELS)
    sp = ea.solve_params(point_stride=1, loss_type=ea.LOSS_HUBER, loss_scale=HUBER_A)
    for arm in arms.values():
        arm["tracker"] = ea.Tracker(ctx, fp, sp, S, KEYFRAME_INTERVAL, image_format=arm["fmt"])
        arm["runs"] = []
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    n_key = sum(1 for t in range(Wm + 1, T) if t % KEYFRAME_INTERVAL == 0)

    def run_arm(arm):
        tr, fb = arm["tracker"], arm["frame_b"]
        dptr = lambda t: hd[ring_index(t, NF)].data_ptr() if t % KEYFRAME_INTERVAL == 0 else 0
        # resident
        tr.reset()
        for t in range(Wm + 1):
            tr.step_device(arm["dev"].data_ptr() + ring_index(t, NF) * fb, depth_d.data_ptr() + ring_index(t, NF) * frame_d)
        torch.cuda.synchronize()
        ctx.profile_enable(True); ctx.profile_read()
        e0.record(stream)
        for t in range(Wm + 1, T):
            tr.step_device(arm["dev"].data_ptr() + ring_index(t, NF) * fb, depth_d.data_ptr() + ring_index(t, NF) * frame_d)
        e1.record(stream)
        torch.cuda.synchronize()
        ms_res = e0.elapsed_time(e1)
        prof = ctx.profile_read(); ctx.profile_enable(False)
        res_out = tr.poses()
        # e2e: pinned host frames through the host entry point, frame t submitted before frame t-1's results are read
        hb = arm["host"]
        tr.reset()
        for t in range(Wm + 1):
            tr.step_host(hb.data_ptr() + ring_index(t, NF) * fb, dptr(t), fetch=True)
        torch.cuda.synchronize()
        e0.record(stream)
        for t in range(Wm + 1, T):
            tr.step_host(hb.data_ptr() + ring_index(t, NF) * fb, dptr(t), fetch=False)
            if t > Wm + 1:
                tr.wait(t - 1)
        e2e_out = tr.wait(T - 1)
        e1.record(stream)
        torch.cuda.synchronize()
        ms_e2e = e0.elapsed_time(e1)
        # ceiling: the same uploads from the same pinned buffers, nothing else running
        stage_b = torch.empty(hb.shape[1:], dtype=torch.uint8, device=dev)
        stage_d = torch.empty((S, H, W), dtype=torch.uint16, device=dev)
        stage_b.copy_(hb[0], non_blocking=True)
        torch.cuda.synchronize()
        e0.record(stream)
        for t in range(Wm + 1, T):
            stage_b.copy_(hb[ring_index(t, NF)], non_blocking=True)
            if t % KEYFRAME_INTERVAL == 0:
                stage_d.copy_(hd[ring_index(t, NF)], non_blocking=True)
        e1.record(stream)
        torch.cuda.synchronize()
        ms_c = e0.elapsed_time(e1)
        del stage_b, stage_d
        h2d = (fb * K + frame_d * n_key) / K
        summ = lambda Ss: [tuple(getattr(s, k) for k, _ in s._fields_) for s in Ss]
        arm["runs"].append(dict(resident=S * K / (ms_res * 1e-3), e2e=S * K / (ms_e2e * 1e-3),
                                preprocess_ms_per_step=prof["preprocess_ms"] / max(1, prof["n_preprocess"]),
                                h2d_bytes_per_step=int(h2d), h2d_ceiling_gbs=h2d * K / (ms_c * 1e-3) / 1e9,
                                h2d_ceiling_alignments_s=S * K / (ms_c * 1e-3), frac_of_h2d_ceiling=ms_c / ms_e2e,
                                _res=(res_out[0].copy(), summ(res_out[1])), _e2e=(e2e_out[0].copy(), summ(e2e_out[1]))))

    for _ in range(a.runs):
        for name in ("bgr", "gray"):
            run_arm(arms[name])
    clocks = gpu_info()

    # correctness first: every run of both arms returns the same poses and summaries, bit for bit
    ref = arms["bgr"]["runs"][0]
    for name, arm in arms.items():
        for i, r in enumerate(arm["runs"]):
            for leg in ("_res", "_e2e"):
                if not (np.array_equal(r[leg][0], ref[leg][0]) and r[leg][1] == ref[leg][1]):
                    raise SystemExit("bench_gray.py: %s run %d %s results differ from the BGR arm's" % (name, i, leg[1:]))

    out = {"workload": "tracker, %d streams, %dx%d, %d levels, Huber(%g), stride 1, key frame every %d; %d timed steps after %d warm-up, "
                       "%d distinct frames per stream" % (S, W, H, N_LEVELS, HUBER_A, KEYFRAME_INTERVAL, K, Wm, NF),
           "gpu": "name, power.limit, clocks.sm, clocks.max.sm = " + clocks, "runs": a.runs, "results_identical": True}
    for name, arm in arms.items():
        keys_ = [k for k in arm["runs"][0] if not k.startswith("_")]
        out[name] = {k: float(np.median([r[k] for r in arm["runs"]])) for k in keys_}
        out[name]["e2e_runs"] = [round(r["e2e"]) for r in arm["runs"]]
        out[name]["resident_runs"] = [round(r["resident"]) for r in arm["runs"]]
        arm["tracker"].close()
    out["gray_over_bgr"] = {k: out["gray"][k] / out["bgr"][k] for k in ("resident", "e2e", "preprocess_ms_per_step", "h2d_bytes_per_step")}
    out["estimates"] = {"h2d_bytes_ratio": 1.2 / 3.2, "e2e_ceiling_alignments_s": 150e3,
                        "note": "set before measuring: 2.7x fewer upload bytes, an upload ceiling near 150 k alignments/s, and a shorter "
                                "preprocessing step (the gray edge kernel skips the 3-channel blur and the colour conversion)"}
    ctx.close()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
