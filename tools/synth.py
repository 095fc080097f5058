"""Synthetic TUM-fr1-shaped RGB-D sequences (BASELINE.json configs[1..4]): a textured box room ray-cast from a
smoothly moving pinhole camera, so both views of every pair are exact and the ground-truth relative pose is known.
Data synthesis only -- not part of the measured path.  Runs on CPU (tests) or GPU (bench) through torch.

Frame format == the reference's inputs (standalone_edge_align.cpp:118-122): BGR u8 [h][w][3], depth u16 = metres *
5000 with ~25 % invalid (zero) pixels like the bundled TUM grabs.
"""
import numpy as np
import torch

TUM_K = (525.0, 525.0, 319.5, 239.5)   # standalone_edge_align.cpp:152


def _hash32(x):
    # 32-bit integer mix inside int64 (identical on CPU and CUDA, no overflow): Wang-style xorshift-multiply
    M = 0xFFFFFFFF
    x = x & M
    x = ((x ^ (x >> 16)) * 0x45D9F3B) & M
    x = ((x ^ (x >> 16)) * 0x45D9F3B) & M
    return (x ^ (x >> 16)) & M


def trajectory(n_frames, seed, max_rot_deg=1.2, max_trans=0.025):
    """Camera-to-world poses (R [n,3,3], t [n,3]) of a smooth random walk; per-frame motion stays within the
    magnitude the bundled fixtures show (<= ~2.5 deg / 5 cm)."""
    rng = np.random.default_rng(seed)
    R = np.eye(3); t = np.zeros(3)
    w = rng.normal(0, 1, 3); v = rng.normal(0, 1, 3)
    Rs, ts = [], []
    for _ in range(n_frames):
        Rs.append(R.copy()); ts.append(t.copy())
        w = 0.85 * w + 0.5 * rng.normal(0, 1, 3); v = 0.85 * v + 0.5 * rng.normal(0, 1, 3)
        wv = w / max(1.0, np.linalg.norm(w)) * np.radians(max_rot_deg)
        vv = v / max(1.0, np.linalg.norm(v)) * max_trans
        th = np.linalg.norm(wv)
        k = wv / th if th > 0 else np.array([1.0, 0, 0])
        Kx = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
        dR = np.eye(3) + np.sin(th) * Kx + (1 - np.cos(th)) * Kx @ Kx
        R = R @ dR
        t = np.clip(t + R @ vv, -0.6, 0.6)     # stay well inside the room
    return np.stack(Rs), np.stack(ts)


def relative_pose(Rw, tw, a, b):
    """b_T_a as (q wxyz, t): X_b = R X_a + t for camera-to-world poses of frames a and b."""
    R = Rw[b].T @ Rw[a]
    t = Rw[b].T @ (tw[a] - tw[b])
    qw = np.sqrt(max(0.0, 1 + R[0, 0] + R[1, 1] + R[2, 2])) / 2
    q = np.array([qw, (R[2, 1] - R[1, 2]) / (4 * qw), (R[0, 2] - R[2, 0]) / (4 * qw), (R[1, 0] - R[0, 1]) / (4 * qw)])
    return np.concatenate([q, t])


def render(Rw, tw, seed, width=640, height=480, K=TUM_K, device="cpu", cell=0.2, hole_frac=0.25, room=(1.7, 1.25, 2.6),
           n_boxes=5, chunk=8):
    """Render len(Rw) frames (batched over frames).  Returns (bgr u8 [n,h,w,3], depth u16 [n,h,w]) on `device`."""
    dev = torch.device(device)
    n = len(Rw)
    fx, fy, cx, cy = K
    f64 = torch.float64
    Rw_t = torch.as_tensor(np.asarray(Rw), dtype=f64, device=dev)
    tw_t = torch.as_tensor(np.asarray(tw), dtype=f64, device=dev)
    v, u = torch.meshgrid(torch.arange(height, device=dev, dtype=f64), torch.arange(width, device=dev, dtype=f64), indexing="ij")
    d_cam = torch.stack([(u - cx) / fx, (v - cy) / fy, torch.ones_like(u)], -1)            # [h,w,3], z = 1
    half = torch.tensor(room, dtype=f64, device=dev)
    brng = np.random.default_rng(int(seed) * 31 + 7)
    boxes = np.stack([np.concatenate([[brng.uniform(-1.1, 1.1), brng.uniform(-0.7, 0.9), brng.uniform(1.2, 2.3)],
                                      brng.uniform(0.12, 0.38, 3)]) for _ in range(max(n_boxes, 1))])
    boxes_t = torch.as_tensor(boxes, dtype=f64, device=dev)
    bgr = torch.empty((n, height, width, 3), dtype=torch.uint8, device=dev)
    depth = torch.empty((n, height, width), dtype=torch.int32, device=dev)
    for c0 in range(0, n, chunk):
        c1 = min(n, c0 + chunk)
        d = torch.einsum("hwj,nij->nhwi", d_cam, Rw_t[c0:c1])                            # world ray directions [m,h,w,3]
        o = tw_t[c0:c1, None, None, :]
        # slab exit of an axis-aligned room containing the camera: per axis the wall the ray heads to
        tpos = torch.where(d > 0, (half - o) / d.clamp_min(1e-12), (-half - o) / d.clamp_max(-1e-12))
        tpos = torch.where(d == 0, torch.full_like(tpos, 1e30), tpos)
        t_hit, axis = tpos.min(-1)
        side = (torch.gather(d, -1, axis.unsqueeze(-1)).squeeze(-1) > 0).long()
        obj = torch.zeros_like(axis)
        dsafe = torch.where(d.abs() < 1e-12, torch.full_like(d, 1e-12), d)
        # furniture: axis-aligned boxes in front of the camera (slab entry test) => depth discontinuities
        for bi in range(n_boxes):
            c = boxes_t[bi, :3]; hs = boxes_t[bi, 3:]
            t1 = (c - hs - o) / dsafe; t2 = (c + hs - o) / dsafe
            tn = torch.minimum(t1, t2); tf = torch.maximum(t1, t2)
            t_near, ax_b = tn.max(-1); t_far = tf.min(-1).values
            hit = (t_near < t_far) & (t_near > 0.05) & (t_near < t_hit)
            t_hit = torch.where(hit, t_near, t_hit); axis = torch.where(hit, ax_b, axis)
            side = torch.where(hit, (torch.gather(d, -1, ax_b.unsqueeze(-1)).squeeze(-1) < 0).long(), side)
            obj = torch.where(hit, torch.full_like(obj, bi + 1), obj)
        p = o + d * t_hit.unsqueeze(-1)
        # plane coordinates = the two non-hit axes; surface id = object*8 + axis*2 + side
        a_ax = (axis + 1) % 3; b_ax = (axis + 2) % 3
        pa = torch.gather(p, -1, a_ax.unsqueeze(-1)).squeeze(-1); pb = torch.gather(p, -1, b_ax.unsqueeze(-1)).squeeze(-1)
        wall = obj * 8 + axis * 2 + side
        ca = torch.floor(pa / cell).long() + 4096; cb = torch.floor(pb / cell).long() + 4096
        h0 = _hash32(ca * 73856093 + cb * 19349663 + wall * 83492791 + (seed * 2654435761))
        fa = torch.floor(pa / (cell * 0.37)).long() + 4096; fb = torch.floor(pb / (cell * 0.37)).long() + 4096
        h1 = _hash32(fa * 73856093 + fb * 19349663 + wall * 83492791 + (seed * 2654435761 + 40503))
        # the fine layer only exists in ~half of the coarse cells (keeps the edge density TUM-like)
        on = (_hash32(ca * 2246822519 + cb * 3266489917 + wall * 668265263 + seed) & 1).to(f64).unsqueeze(-1)
        rgb0 = torch.stack([(h0 & 255), ((h0 >> 8) & 255), ((h0 >> 16) & 255)], -1).to(f64)
        rgb1 = torch.stack([(h1 & 255), ((h1 >> 8) & 255), ((h1 >> 16) & 255)], -1).to(f64)
        col = 0.65 * rgb0 + 0.35 * (rgb1 * on + (1 - on) * 128.0)
        shade = (1.15 - 0.12 * t_hit).clamp(0.6, 1.1).unsqueeze(-1)                      # mild distance shading
        bgr[c0:c1] = (col * shade).clamp(0, 255).to(torch.uint8)
        depth[c0:c1] = torch.round(t_hit * 5000.0).clamp(0, 65535).to(torch.int32)         # d_cam has z = 1 => depth == t
    # invalid-depth blobs: low-frequency noise, ~hole_frac of the pixels (the bundled TUM grabs have 24-25 %)
    if hole_frac > 0:
        g = torch.Generator(device="cpu"); g.manual_seed(int(seed) * 7919 + 13)
        lo = torch.rand((n, 1, height // 16 + 2, width // 16 + 2), generator=g).to(dev)
        noise = torch.nn.functional.interpolate(lo, size=(height, width), mode="bilinear", align_corners=False).squeeze(1)
        thr = torch.quantile(noise[0].flatten().float(), hole_frac)
        depth = torch.where(noise < thr, torch.zeros_like(depth), depth)
    return bgr, depth.to(torch.uint16)


def make_sequences(n_streams, n_frames, seed=0, width=640, height=480, K=TUM_K, device="cpu"):
    """n_streams independent sequences.  Returns bgr [T,S,h,w,3] u8, depth [T,S,h,w] u16 (frame-major so that one
    tracker step reads one contiguous block), and the list of (Rw, tw) trajectories."""
    bgr = torch.empty((n_frames, n_streams, height, width, 3), dtype=torch.uint8, device=device)
    depth = torch.empty((n_frames, n_streams, height, width), dtype=torch.uint16, device=device)
    traj = []
    for s in range(n_streams):
        Rw, tw = trajectory(n_frames, seed * 100003 + s)
        b, d = render(Rw, tw, seed * 100003 + s, width, height, K, device)
        bgr[:, s] = b; depth[:, s] = d
        traj.append((Rw, tw))
    return bgr, depth, traj


def stereo_rig(Rw, tw, baseline=0.12, yaw_deg=2.0):
    """A second camera rigidly mounted beside the one that follows (Rw, tw): `baseline` metres along its x axis, turned by
    `yaw_deg` about its y axis.  Returns the second camera's camera-to-world poses (R [n,3,3], t [n,3]) and T21, the 4x4
    transform from first-camera to second-camera coordinates (ea_view.cam_T_first; X_2 = R21 X_1 + t21)."""
    a = np.radians(yaw_deg)
    R12 = np.array([[np.cos(a), 0, np.sin(a)], [0, 1, 0], [-np.sin(a), 0, np.cos(a)]])   # second camera's axes in the first's
    t12 = np.array([baseline, 0.0, 0.0])
    Rw2 = np.einsum("nij,jk->nik", np.asarray(Rw), R12)
    tw2 = np.asarray(tw) + np.einsum("nij,j->ni", np.asarray(Rw), t12)
    T21 = np.eye(4)
    T21[:3, :3] = R12.T
    T21[:3, 3] = -R12.T @ t12
    return Rw2, tw2, T21
