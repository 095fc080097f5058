#!/usr/bin/env python
"""Camera / decoder frame layouts against dense gray through the tracker, on the default bench.py workload.

Workload: bench.py's default line -- 1 184 camera streams, 640 x 480, 3 pyramid levels, Huber(0.1), stride 1, a key frame every
10 frames -- on synthetic sequences (tools/synth.make_sequences) converted to gray with OpenCV's 15-bit RGB2GRAY formula.  Arms:
  gray   EA_IMAGE_GRAY8, dense
  nv12   EA_IMAGE_NV12 with an NVDEC-like row pitch of 768 bytes, the chroma plane after the luma (random bytes)
  yuyv   EA_IMAGE_YUYV, dense (random chroma bytes)
All arms carry the same luma, so the script fails unless their poses and summaries are bit-identical.

The arms alternate within one call, --runs times each.  Per arm it reports the median over runs of
  resident     alignments/s with frames resident in HBM (ea_tracker_step_device, stream-ordered as bench.py's value)
  e2e          alignments/s with every step's frames uploaded from pinned host memory (ea_tracker_step_host, pipelined with
               ea_tracker_wait as bench.py's e2e leg)
  preprocess   device ms per step of the preprocessing pipeline in the resident run (ea_profile_read)
  h2d          bytes uploaded per step (the rows the kernels read every step, depth on key frames); the achieved rate of the
               image upload alone (the library's own copy, timed with nothing else running), against a dense copy of the same
               number of bytes from the same pinned memory in the same run
plus the card's name, power limit and SM clocks, read in the same call.
"""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.dont_write_bytecode = True
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_gray import H, HUBER_A, KEYFRAME_INTERVAL, N_LEVELS, W, gpu_info, ring_index  # noqa: E402

NV12_PITCH = 768


class _Pitched(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("pitch", C.c_size_t), ("xsize", C.c_size_t), ("ysize", C.c_size_t)]


class _Triple(C.Structure):
    _fields_ = [("x", C.c_size_t), ("y", C.c_size_t), ("z", C.c_size_t)]


class _Memcpy3DParms(C.Structure):   # cudaMemcpy3DParms
    _fields_ = [("srcArray", C.c_void_p), ("srcPos", _Triple), ("srcPtr", _Pitched), ("dstArray", C.c_void_p), ("dstPos", _Triple),
                ("dstPtr", _Pitched), ("extent", _Triple), ("kind", C.c_int)]


def cuda_runtime():
    path = "/usr/local/cuda/lib64/libcudart.so"
    rt = C.CDLL(path if os.path.exists(path) else "libcudart.so")
    rt.cudaMemcpyAsync.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]
    rt.cudaMemcpy2DAsync.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int, C.c_void_p]
    rt.cudaMemcpy3DAsync.argtypes = [C.POINTER(_Memcpy3DParms), C.c_void_p]
    return rt


def check(rc):
    if rc != 0:
        raise SystemExit("bench_yuv.py: CUDA runtime error %d" % rc)


def upload_frames(rt, dst, src, lay, n, stream):
    """The copy ea_upload_frames issues for n frames of layout lay (H2D): the rows the kernels read, packed dense."""
    row = {0: 3 * W, 1: W, 2: W, 3: 2 * W, 4: 2 * W}[lay.format]
    pitch = lay.row_pitch or row
    rows = (lay.frame_stride or (3 * H // 2 if lay.format == 2 else H) * pitch) // pitch
    if pitch == row and rows == H:
        return check(rt.cudaMemcpyAsync(dst, src, row * H * n, 1, stream))
    if rows == H:
        return check(rt.cudaMemcpy2DAsync(dst, row, src, pitch, row, H * n, 1, stream))
    p = _Memcpy3DParms(srcPtr=_Pitched(src, pitch, row, rows), dstPtr=_Pitched(dst, row, row, H), extent=_Triple(row, H, n), kind=1)
    return check(rt.cudaMemcpy3DAsync(C.byref(p), stream))


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
        raise SystemExit("bench_yuv.py: no CUDA device; the product path has no CPU fallback")
    import edge_alignment_b200 as ea
    import synth

    S, K, Wm, NF = a.streams, a.steps, max(a.warmup, 3), a.frames
    T = Wm + K + 1
    dev = torch.device("cuda", 0)
    bgr_src, depth_d, _ = synth.make_sequences(S, NF, seed=a.seed, device=dev)
    b = bgr_src.to(torch.int32)
    gray_d = ((b[..., 0] * 9798 + b[..., 1] * 19235 + b[..., 2] * 3735 + 16384) >> 15).to(torch.uint8).contiguous()
    del b, bgr_src
    g = torch.Generator(device=dev); g.manual_seed(a.seed)
    nv12_d = torch.randint(0, 256, (NF, S, 3 * H // 2, NV12_PITCH), dtype=torch.uint8, device=dev, generator=g)
    nv12_d[:, :, :H, :W] = gray_d
    yuyv_d = torch.randint(0, 256, (NF, S, H, 2 * W), dtype=torch.uint8, device=dev, generator=g)
    yuyv_d[..., 0::2] = gray_d
    depth_d = depth_d.contiguous()
    frame_d = W * H * 2 * S
    keys = sorted({ring_index(t, NF) for t in range(T) if t % KEYFRAME_INTERVAL == 0})
    hd = {f: depth_d[f].cpu().pin_memory() for f in keys}
    arms = {
        "gray": dict(layout=ea.image_layout(ea.IMAGE_GRAY8), dev=gray_d, up_b=W * H * S),
        "nv12": dict(layout=ea.image_layout(ea.IMAGE_NV12, NV12_PITCH, 3 * H // 2 * NV12_PITCH), dev=nv12_d, up_b=W * H * S),
        "yuyv": dict(layout=ea.image_layout(ea.IMAGE_YUYV), dev=yuyv_d, up_b=2 * W * H * S),
    }
    for arm in arms.values():
        arm["host"] = arm["dev"].cpu().pin_memory()
        arm["frame_b"] = arm["dev"][0].numel()
    torch.cuda.synchronize()

    ctx = ea.Context(0)
    stream = torch.cuda.current_stream()
    ctx.set_stream(stream.cuda_stream)
    fp = ea.frame_params(n_levels=N_LEVELS)
    sp = ea.solve_params(point_stride=1, loss_type=ea.LOSS_HUBER, loss_scale=HUBER_A)
    for arm in arms.values():
        arm["tracker"] = ea.Tracker(ctx, fp, sp, S, KEYFRAME_INTERVAL)
        arm["tracker"].set_image_layout(arm["layout"])
        arm["runs"] = []
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    n_key = sum(1 for t in range(Wm + 1, T) if t % KEYFRAME_INTERVAL == 0)
    rt = cuda_runtime()

    def timed_copies(fn, reps):
        fn(0)
        torch.cuda.synchronize()
        e0.record(stream)
        for t in range(reps):
            fn(t)
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

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
        # upload rates, nothing else running: the rows the kernels read, with the copy the library issues (ea_upload_frames),
        # against a dense copy of as many bytes from the same pinned memory
        up = arm["up_b"]
        dst = torch.empty(up, dtype=torch.uint8, device=dev)
        s_ = stream.cuda_stream
        ms_up = timed_copies(lambda t: upload_frames(rt, dst.data_ptr(), hb.data_ptr() + ring_index(t, NF) * fb, arm["layout"], S, s_), 10)
        ms_dense = timed_copies(lambda t: check(rt.cudaMemcpyAsync(dst.data_ptr(), hb.data_ptr(), up, 1, s_)), 10)
        del dst
        h2d = (up * K + frame_d * n_key) / K
        summ = lambda Ss: [tuple(getattr(s, k) for k, _ in s._fields_) for s in Ss]
        arm["runs"].append(dict(resident=S * K / (ms_res * 1e-3), e2e=S * K / (ms_e2e * 1e-3),
                                preprocess_ms_per_step=prof["preprocess_ms"] / max(1, prof["n_preprocess"]),
                                h2d_gb_per_step=h2d / 1e9, image_upload_gbs=up / (ms_up * 1e-3) / 1e9,
                                dense_copy_gbs=up / (ms_dense * 1e-3) / 1e9,
                                _res=(res_out[0].copy(), summ(res_out[1])), _e2e=(e2e_out[0].copy(), summ(e2e_out[1]))))

    for _ in range(a.runs):
        for name in ("gray", "nv12", "yuyv"):
            run_arm(arms[name])
    clocks = gpu_info()

    # correctness first: every run of every arm returns the same poses and summaries, bit for bit
    ref = arms["gray"]["runs"][0]
    for name, arm in arms.items():
        for i, r in enumerate(arm["runs"]):
            for leg in ("_res", "_e2e"):
                if not (np.array_equal(r[leg][0], ref[leg][0]) and r[leg][1] == ref[leg][1]):
                    raise SystemExit("bench_yuv.py: %s run %d %s results differ from the gray arm's" % (name, i, leg[1:]))

    out = {"workload": "tracker, %d streams, %dx%d, %d levels, Huber(%g), stride 1, key frame every %d; %d timed steps after %d warm-up, "
                       "%d distinct frames per stream; NV12 row pitch %d" % (S, W, H, N_LEVELS, HUBER_A, KEYFRAME_INTERVAL, K, Wm, NF, NV12_PITCH),
           "gpu": "name, power.limit, clocks.sm, clocks.max.sm = " + clocks, "runs": a.runs, "poses_identical": True}
    for name, arm in arms.items():
        keys_ = [k for k in arm["runs"][0] if not k.startswith("_")]
        out[name] = {k: float(np.median([r[k] for r in arm["runs"]])) for k in keys_}
        out[name]["e2e_runs"] = [round(r["e2e"]) for r in arm["runs"]]
        out[name]["resident_runs"] = [round(r["resident"]) for r in arm["runs"]]
        arm["tracker"].close()
    out["estimates"] = {"nv12_e2e_alignments_s": 126e3, "yuyv_e2e_ceiling_alignments_s": 82e3, "gray_preprocess_ms_per_step": 2.35,
                        "note": "set before measuring: NV12 e2e as gray's if the pitched copy reaches the dense rate; YUYV e2e at most "
                                "about 82 k (0.73 GB image + 0.07 GB depth per step at 55.5 GB/s); device preprocessing of NV12 "
                                "within noise of gray's, YUYV a little above"}
    ctx.close()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
