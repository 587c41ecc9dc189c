"""Synthetic rigs and detections for the throughput configs of BASELINE.json (SURVEY.md 8(d)).

Everything is keyed by the GLOBAL frame index through a counter-based hash (splitmix64), so any
sharding of the frame range over GPUs sees the same data.  Runs in torch on whatever device the
caller names (the bench generates on the GPU; the parity tests copy the same tensors to the host for
the oracle).
"""
from __future__ import annotations

import math

import numpy as np

from . import Camera

SEED = 20240607


def look_at_quat(pos, target=(0.0, 0.0, 0.0)):
    """(w,x,y,z) of the camera-to-world rotation whose +z axis points from pos to target, x to the
    right and y down -- the convention of the reference's ray model (Triangulator.cpp:15-55) and of
    Camera::createExtricsicMat (Camera.h:133-153: extrinsic R = toRotMatrix(q)^-1)."""
    p, t = np.asarray(pos, float), np.asarray(target, float)
    z = (t - p) / np.linalg.norm(t - p)
    up = np.array([0.0, 0.0, 1.0])
    x = np.cross(z, up)
    x /= np.linalg.norm(x)
    y = np.cross(z, x)
    R = np.stack([x, y, z], axis=1)  # columns = camera axes in world coordinates
    t_ = R[0, 0] + R[1, 1] + R[2, 2]
    if t_ > 0:
        s = math.sqrt(t_ + 1.0) * 2
        q = (0.25 * s, (R[2, 1] - R[1, 2]) / s, (R[0, 2] - R[2, 0]) / s, (R[1, 0] - R[0, 1]) / s)
    elif R[0, 0] > R[1, 1] and R[0, 0] > R[2, 2]:
        s = math.sqrt(1.0 + R[0, 0] - R[1, 1] - R[2, 2]) * 2
        q = ((R[2, 1] - R[1, 2]) / s, 0.25 * s, (R[0, 1] + R[1, 0]) / s, (R[0, 2] + R[2, 0]) / s)
    elif R[1, 1] > R[2, 2]:
        s = math.sqrt(1.0 + R[1, 1] - R[0, 0] - R[2, 2]) * 2
        q = ((R[0, 2] - R[2, 0]) / s, (R[0, 1] + R[1, 0]) / s, 0.25 * s, (R[1, 2] + R[2, 1]) / s)
    else:
        s = math.sqrt(1.0 + R[2, 2] - R[0, 0] - R[1, 1]) * 2
        q = ((R[1, 0] - R[0, 1]) / s, (R[0, 2] + R[2, 0]) / s, (R[1, 2] + R[2, 1]) / s, 0.25 * s)
    return tuple(float(v) for v in q)


def ring_rig(n_cams=8, rings=((6000.0, 3000.0),), width=1920, height=1080, focal=1081.0810546875):
    """Cameras evenly spaced on ring(s) (radius, z) in mm, looking at the origin; built through the
    same Camera arithmetic as the real rigs.  BASELINE config 4: 8 cameras, one ring; config 5: 32
    cameras on two rings ((6000,3000),(9000,5000))."""
    cams = []
    per = n_cams // len(rings)
    for r_i, (radius, z) in enumerate(rings):
        n = per if r_i < len(rings) - 1 else n_cams - per * (len(rings) - 1)
        for k in range(n):
            a = 2 * math.pi * (k + 0.5 * r_i) / n
            pos = (radius * math.cos(a), radius * math.sin(a), z)
            cams.append(Camera(len(cams) + 1, width, height, focal, pos, look_at_quat(pos, (0.0, 0.0, 1000.0))))
    return cams


def _hash01(torch, idx, stream):
    """splitmix64(idx, stream) -> float64 uniform in (0,1); idx int64 tensor."""
    M34, M37, M33 = (1 << 34) - 1, (1 << 37) - 1, (1 << 33) - 1
    z = idx + (SEED + 0x632BE59BD9B4E019 * (stream + 1)) % (1 << 63)
    z = z * -7046029254386353131  # 0x9E3779B97F4A7C15 as int64
    z = (z ^ ((z >> 30) & M34)) * -4658895280553007687  # 0xBF58476D1CE4E5B9
    z = (z ^ ((z >> 27) & M37)) * -7723592293110705685  # 0x94D049BB133111EB
    z = z ^ ((z >> 31) & M33)
    return (((z >> 11) & ((1 << 53) - 1)).to(torch.float64) + 0.5) * (1.0 / (1 << 53))


def generate_frames(cams, n_frames, frame0=0, device="cpu", p_missing=0.2, noise_px=1.0, out=None, chunk=1 << 22,
                    volume=((-2000.0, 2000.0), (-2000.0, 2000.0), (200.0, 2500.0)), want_truth=False, dtype=None,
                    p_outlier=0.0):
    """-> xy [n_cams, n_frames, 2] float32 (integer-valued pixels, (-1,-1) = missing) on `device`
    (+ truth [n_frames, 3] float64 if asked).  Pixels: project with the reference's own P, add
    N(0, noise_px), round to the nearest integer (real detections are integers,
    DetectionsContainer.cpp:36), then drop each (camera, frame) with probability p_missing.
    p_outlier > 0: a present view is replaced, with that probability, by a uniform random pixel of the image (a false
    detection), drawn from hash streams of its own, so the inlier views are the same as with p_outlier = 0."""
    import torch
    dtype = dtype or torch.float32
    nc = len(cams)
    if out is None:
        out = torch.empty((nc, n_frames, 2), dtype=dtype, device=device)
    truth = torch.empty((n_frames, 3), dtype=torch.float64, device=device) if want_truth else None
    P = torch.tensor(np.stack([c.P for c in cams]), dtype=torch.float64, device=device)  # [nc,3,4]
    for a in range(0, n_frames, chunk):
        n = min(chunk, n_frames - a)
        idx = torch.arange(frame0 + a, frame0 + a + n, dtype=torch.int64, device=device)
        X = torch.stack([lo + (hi - lo) * _hash01(torch, idx, k) for k, (lo, hi) in enumerate(volume)], dim=1)
        if truth is not None:
            truth[a:a + n] = X
        Xh = torch.cat([X, torch.ones((n, 1), dtype=torch.float64, device=device)], dim=1)  # [n,4]
        for c in range(nc):
            h = Xh @ P[c].T  # [n,3]
            u1, u2 = _hash01(torch, idx, 16 + 4 * c), _hash01(torch, idx, 17 + 4 * c)
            rad = torch.sqrt(-2.0 * torch.log(u1)) * noise_px
            px = torch.round(h[:, 0] / h[:, 2] + rad * torch.cos(2 * math.pi * u2))
            py = torch.round(h[:, 1] / h[:, 2] + rad * torch.sin(2 * math.pi * u2))
            miss = _hash01(torch, idx, 18 + 4 * c) < p_missing
            if p_outlier > 0:
                bad = _hash01(torch, idx, 1024 + 4 * c) < p_outlier
                px = torch.where(bad, torch.floor(_hash01(torch, idx, 1025 + 4 * c) * cams[c].width), px)
                py = torch.where(bad, torch.floor(_hash01(torch, idx, 1026 + 4 * c) * cams[c].height), py)
            if dtype == torch.uint16:
                px = torch.where(miss, torch.full_like(px, 65535.0), px.clamp(0, 65534))
                py = torch.where(miss, torch.full_like(py, 65535.0), py.clamp(0, 65534))
                out[c, a:a + n, 0] = px.to(torch.int32).to(torch.uint16)
                out[c, a:a + n, 1] = py.to(torch.int32).to(torch.uint16)
            else:
                px = torch.where(miss, torch.full_like(px, -1.0), px)
                py = torch.where(miss, torch.full_like(py, -1.0), py)
                out[c, a:a + n, 0] = px.to(dtype)
                out[c, a:a + n, 1] = py.to(dtype)
    return (out, truth) if want_truth else out


def drone_positions(torch, idx, n_drones, volume=((-2000.0, 2000.0), (-2000.0, 2000.0), (200.0, 2500.0))):
    """World positions [n_drones, n, 3] (mm) at the global frame indices `idx`: drone d circles a centre on a hexagon
    of radius 1500 mm (1500 mm between neighbours) with a Lissajous figure of at most 450 mm amplitude, so any two
    drones stay >= 600 mm apart, and it moves < 60 mm per frame -- inside the classifier's MAX_STEP = 200 mm gate
    (DroneClassifier.h:13).  A closed-form function of the frame index: any sharding sees the same flight."""
    t = idx.to(torch.float64)
    (x0, x1), (y0, y1), (z0, z1) = volume
    cx, cy = 0.5 * (x0 + x1), 0.5 * (y0 + y1)
    out = []
    for d in range(n_drones):
        a = 2 * math.pi * d / max(n_drones, 1)
        wx, wy, wz = 0.031 + 0.0037 * d, 0.043 - 0.0029 * d, 0.017 + 0.0021 * d  # rad per frame
        px = cx + 1500.0 * math.cos(a) + 450.0 * torch.sin(wx * t + 0.9 * d)
        py = cy + 1500.0 * math.sin(a) + 450.0 * torch.sin(wy * t + 1.7 * d)
        pz = z0 + (z1 - z0) * (d + 0.5) / n_drones + 150.0 * torch.sin(wz * t + 0.3 * d)
        out.append(torch.stack([px, py, pz], dim=1))
    return torch.stack(out)


def generate_multi_drone(cams, n_frames, n_drones=6, frame0=0, device="cpu", p_drop=0.2, noise_px=1.0, chunk=1 << 20):
    """BASELINE config 5's classifier input (SURVEY.md 8d): n_drones drones per frame, every camera sees each with
    probability 1 - p_drop, and stores its detections in a per-(camera, frame) random order, so the assignment is not
    trivial.  Pixels are projected with the reference's own P, N(0, noise_px) noise, rounded to integers.
    -> (det_offsets int32 [n_cams * (n_frames + 1)], dets_xy float64 [n, 2], truth float64 [n_drones, n_frames, 3]):
    the CSR layout of tri_classify / orc_classify ([cam][frame][det], offsets absolute).  Everything is keyed by the
    global frame index (counter-based hash), so shards and sequences cut from the same index range agree."""
    import torch
    nc = len(cams)
    P = torch.tensor(np.stack([c.P for c in cams]), dtype=torch.float64, device=device)
    counts = torch.zeros((nc, n_frames), dtype=torch.int32, device=device)
    xs, truth = [[] for _ in range(nc)], []
    for a in range(0, n_frames, chunk):
        n = min(chunk, n_frames - a)
        idx = torch.arange(frame0 + a, frame0 + a + n, dtype=torch.int64, device=device)
        X = drone_positions(torch, idx, n_drones)  # [D, n, 3]
        truth.append(X)
        Xh = torch.cat([X, torch.ones((n_drones, n, 1), dtype=torch.float64, device=device)], dim=2)
        for c in range(nc):
            h = Xh @ P[c].T  # [D, n, 3]
            px, py, keep, key = [], [], [], []
            for d in range(n_drones):
                s0 = 64 + 8 * (c * n_drones + d)
                u1, u2 = _hash01(torch, idx, s0), _hash01(torch, idx, s0 + 1)
                rad = torch.sqrt(-2.0 * torch.log(u1)) * noise_px
                x = torch.round(h[d, :, 0] / h[d, :, 2] + rad * torch.cos(2 * math.pi * u2))
                y = torch.round(h[d, :, 1] / h[d, :, 2] + rad * torch.sin(2 * math.pi * u2))
                inside = (x >= 0) & (x < cams[c].width) & (y >= 0) & (y < cams[c].height) & (h[d, :, 2] > 0)
                px.append(x); py.append(y)
                keep.append((_hash01(torch, idx, s0 + 2) >= p_drop) & inside)
                key.append(_hash01(torch, idx, s0 + 3))
            px, py, keep, key = torch.stack(px, 1), torch.stack(py, 1), torch.stack(keep, 1), torch.stack(key, 1)  # [n, D]
            order = torch.argsort(torch.where(keep, key, key + 2.0), dim=1)  # kept detections first, in hashed order
            px, py, keep = torch.gather(px, 1, order), torch.gather(py, 1, order), torch.gather(keep, 1, order)
            counts[c, a:a + n] = keep.sum(1).to(torch.int32)
            xs[c].append(torch.stack([px[keep], py[keep]], dim=1))  # row-major boolean mask keeps [frame][det] order
    cnt = counts.to(torch.int64)
    per_cam = cnt.sum(1)
    base = torch.cumsum(per_cam, 0) - per_cam
    offs = torch.zeros((nc, n_frames + 1), dtype=torch.int64, device=device)
    offs[:, 1:] = torch.cumsum(cnt, 1)
    offs += base[:, None]
    dets = torch.cat([torch.cat(x, 0) for x in xs], 0)
    return (offs.to(torch.int32).reshape(-1).cpu().numpy(), dets.cpu().numpy().astype(np.float64),
            torch.cat(truth, 1).cpu().numpy())
