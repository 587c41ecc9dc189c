"""Throughput of the outlier-robust batch (tri_triangulate_points_robust_device) on one GPU.

Configs: 8 cameras x 100 M frames and 32 cameras x 20 M frames, device-resident, 20 % missing views, p_outlier 0.1, in FP64
and FP32; float3 points + inlier masks out.  Reports CUDA-event kernel time per call and points/s, the algorithmic flops
per frame counted from the valid-view counts actually drawn (formula below, from the kernel's own operation counts), the
share of the FP64 / FP32 pipe peak and of HBM, and which bound applies.  A seeded sample of frames is checked against the
FP64 CPU oracle at the timed size.  Prints one JSON line; --out also writes it to a file.

    python tools/bench_robust.py [--frames8 100000000] [--frames32 20000000] [--reps 5] [--out profiles/robust_bench.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle")]

# NVIDIA data sheet, HGX B200, per GPU (the 8-GPU figures / 8): FP64 37 TFLOP/s, FP32 75 TFLOP/s, HBM3e 7.7 TB/s
PEAK = {"fp64_flops": 37e12, "fp32_flops": 75e12, "hbm_bytes": 7.7e12}

# flops of the kernel's building blocks (an FMA counts 2): one view's two DLT rows into the normal equations, the
# adjugate solve, one projection with its squared pixel residual
F_ADD_VIEW = 2 * (2 * (4 + 9))  # 2 rows x (4 row FMAs + 9 accumulation FMAs)
F_SOLVE = 42  # cofactors 18, determinant 5, reciprocal 1, three dot products 18
F_PROJECT = 26  # w 6, reciprocal 1, du 8, dv 8, r^2 3
F_PAIR = 2 * F_ADD_VIEW + F_SOLVE


def flops_per_frame(views, inliers):
    """Algorithmic flops of one frame: pairs x (2-view solve + |V| projections) + refit over |I| views."""
    v = views.astype(np.float64)
    i = inliers.astype(np.float64)
    ok = v >= 2
    pairs = v * (v - 1) / 2
    refit = np.where(i >= 2, i * F_ADD_VIEW + F_SOLVE + i * F_PROJECT, 0.0)
    return np.where(ok, pairs * (F_PAIR + v * F_PROJECT) + refit, 0.0)


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def run_config(torch, T, S, O, R, nc, n_frames, p_outlier, flags, reps, warmup, sample):
    cams = S.ring_rig(32, rings=((6000.0, 3000.0), (9000.0, 5000.0))) if nc == 32 else S.ring_rig(nc)
    eng = T.Engine(cams, 0)
    xy = S.generate_frames(cams, n_frames, device="cuda:0", p_outlier=p_outlier)
    out = {"xyz_f32": torch.empty((n_frames, 3), dtype=torch.float32, device="cuda:0"),
           "mask": torch.empty((n_frames,), dtype=torch.int32, device="cuda:0")}
    tau = 10.0
    for _ in range(warmup):
        eng.triangulate_points_robust_device(xy, tau, flags | T.ALLOW_TOO_FEW, out=out)
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in ev:
        a.record()
        eng.triangulate_points_robust_device(xy, tau, flags | T.ALLOW_TOO_FEW, out=out)
        b.record()
    torch.cuda.synchronize()
    eng.device_status()
    ms = sorted(a.elapsed_time(b) for a, b in ev)
    t = ms[len(ms) // 2] * 1e-3
    # algorithmic work from the views actually drawn (valid views from the input, inliers from the output)
    valid = torch.zeros(n_frames, dtype=torch.int32, device="cuda:0")
    for c in range(nc):
        valid += ((xy[c, :, 0] != -1) & (xy[c, :, 1] != -1)).to(torch.int32)
    inl = torch.zeros(n_frames, dtype=torch.int32, device="cuda:0")
    m = out["mask"]
    for c in range(nc):
        inl += (m >> c) & 1
    v, i = valid.cpu().numpy(), inl.cpu().numpy()
    fl = flops_per_frame(v, i)
    flops = float(fl.sum())
    bytes_ = float(n_frames) * (8 * nc + 12 + 4)
    f64 = not (flags & T.F32)
    t_flop = flops / (PEAK["fp64_flops"] if f64 else PEAK["fp32_flops"])
    t_mem = bytes_ / PEAK["hbm_bytes"]
    # oracle check on a seeded sample of frames of the timed batch
    rng = np.random.default_rng(12345 + nc)
    idx = np.sort(rng.choice(n_frames, size=min(sample, n_frames), replace=False))
    it = torch.from_numpy(idx).to("cuda:0")
    sub = xy[:, it].cpu().numpy()
    ref = R.triangulate_points_robust([O.make_camera(c.cam_id, c.width, c.height, c.focal, c.position, c.quat) for c in cams], sub, tau,
                                      allow_too_few=True)
    got_m = out["mask"][it].cpu().numpy().view(np.uint32)
    got_x = out["xyz_f32"][it].cpu().numpy().astype(np.float64)
    thin = ref["margin"] < (1e-9 if f64 else 1e-3)
    same = got_m == ref["mask"]
    both = same & (ref["mask"] != 0)
    tol = 1e-3 + 1e-6 * np.abs(ref["xyz"][both]) if f64 else 1.0  # float3 rounding of the FP64 point / the FP32 tier (1e-4 of 10 m)
    xyz_ok = bool(np.all(np.abs(got_x[both] - ref["xyz"][both]) <= tol))
    return {"cams": nc, "frames": n_frames, "p_missing": 0.2, "p_outlier": p_outlier, "precision": "fp64" if f64 else "fp32",
            "max_reproj_px": tau, "kernel_ms": round(ms[len(ms) // 2], 4), "kernel_ms_min": round(ms[0], 4),
            "points_per_s": n_frames / t, "mean_valid_views": float(v.mean()), "mean_inliers": float(i.mean()),
            "flops_per_frame": flops / n_frames, "achieved_flops": flops / t, "hbm_bytes_per_frame": bytes_ / n_frames,
            "achieved_hbm_bytes_per_s": bytes_ / t, "share_of_pipe_peak": t_flop / t, "share_of_hbm_peak": t_mem / t,
            "bound": "compute (%s pipe)" % ("FP64" if f64 else "FP32") if t_flop > t_mem else "memory (HBM)",
            "consensus_frames": float((i >= 2).mean()),
            "oracle_sample": int(len(idx)), "oracle_masks_equal": int(same.sum()), "oracle_thin_margin": int(thin.sum()),
            "oracle_ok": bool(np.all(same | thin)) and xyz_ok}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames8", type=int, default=100_000_000)
    ap.add_argument("--frames32", type=int, default=20_000_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--sample", type=int, default=2000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_robust.py measures the GPU kernels: no CUDA device")
    import oracle_py as O
    import robust_oracle_py as R
    import tri_b200 as T
    from tri_b200 import synthetic as S
    info = gpu_info()
    res = []
    for nc, nf in ((8, a.frames8), (32, a.frames32)):
        for fl in (0, T.F32):
            res.append(run_config(torch, T, S, O, R, nc, nf, 0.1, fl, a.reps, a.warmup, a.sample))
            torch.cuda.empty_cache()
    line = json.dumps({"bench": "robust", "gpu": info, "peak_datasheet": PEAK, "configs": res,
                       "all_oracle_ok": all(r["oracle_ok"] for r in res)})
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
