#!/usr/bin/env python
"""Milliseconds per frame of Canny-mode preprocessing, on two workloads.

  bundled     the five bundled 640x480 frames, repeated to the batch size: short edge chains, every weak edge near a strong
              one (the common case)
  serpentine  640x480 serpentine frames (tests/test_gpu_canny_edt.serpentine, gray-l1 ramp): one edge chain of ~75 k pixels
              whose farthest pixel is ~26 k 8-connected steps from the nearest strong one, and its mirror images

Settings: the standalone Canny variant (box blur -> gray -> Canny 30/90 L1), exact DT normalised to [0, 1], both roles, one
level.  Frames and depth are resident on the device (ea_frameset_preprocess_device); a timed run is --iters back-to-back calls
ending in a device synchronise, timed by the host clock, after --warmup untimed calls.  The workloads alternate, --runs times
each; the median run is reported, with the spread, the card's name, power limit and SM clocks, read in the same call.
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
sys.path.insert(0, os.path.join(ROOT, "tests"))

W, H = 640, 480


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=20).stdout
        return out.strip().splitlines()[0] if out.strip() else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--batch", type=str, default="5,296", help="comma-separated batch sizes (frames per call)")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--runs", type=int, default=5)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_canny.py: no CUDA device; the product path has no CPU fallback")
    import edge_alignment_b200 as ea
    from test_gpu_canny_edt import LONG_CHAINS, serpentine

    z = np.load(os.path.join(ROOT, "tests", "golden", "frames.npz"))
    s = serpentine(W, H, LONG_CHAINS["gray-l1"][4])
    serp = [s, s[:, ::-1], s[::-1], s[::-1, ::-1]]
    sources = {"bundled": (z["bgr"], z["depth"]),
               "serpentine": (np.stack([np.repeat(v[..., None], 3, -1) for v in serp]), np.stack([z["depth"][0]] * len(serp)))}
    ctx = ea.Context(0)
    fp = ea.frame_params(edge_detector=ea.EDGE_CANNY_GRAY, canny_low=30.0, canny_high=90.0, canny_l2=0, dt_kind=ea.DT_EXACT,
                         dt_normalize=ea.NORM_01, max_points=W * H)
    out = {"gpu": gpu_info(), "width": W, "height": H, "iters": a.iters, "runs": a.runs, "ms_per_frame": {}}
    for n in (int(v) for v in a.batch.split(",")):
        fs = ea.FrameSet(ctx, fp, n)
        dev = {}
        for name, (bgr, dep) in sources.items():
            idx = np.arange(n) % len(bgr)
            dev[name] = (torch.from_numpy(np.ascontiguousarray(bgr[idx])).cuda(), torch.from_numpy(np.ascontiguousarray(dep[idx])).cuda())
        torch.cuda.synchronize()
        slots = np.arange(n)
        call = lambda name: fs.preprocess_device(slots, dev[name][0].data_ptr(), dev[name][1].data_ptr(), ea.ROLE_BOTH)
        runs = {name: [] for name in sources}
        for name in sources:
            for _ in range(a.warmup):
                call(name)
        ctx.sync()
        for _ in range(a.runs):
            for name in sources:
                t0 = time.perf_counter()
                for _ in range(a.iters):
                    call(name)
                ctx.sync()
                runs[name].append((time.perf_counter() - t0) * 1e3 / (a.iters * n))
        for name, r in runs.items():
            out["ms_per_frame"]["%s/batch%d" % (name, n)] = {"median": round(float(np.median(r)), 5),
                                                             "min": round(min(r), 5), "max": round(max(r), 5)}
        fs.close()
    ctx.close()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
