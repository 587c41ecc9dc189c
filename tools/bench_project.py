"""Throughput of the forward projection (tri_project_points_device) on one GPU.

Configs, device-resident: 8 cameras x 100 M points in FP64 and FP32 with float2 and ushort2 pixel rows, and 32 cameras x
20 M points in FP64 and FP32 with float2 rows; input points float64 [n][3] (24 B) in FP64, float32 [n][3] (12 B) in
FP32 -- the point outputs of the batch calls of the same precision; visibility masks on.  Reports the
CUDA-event time per call and points/s, the algorithmic bytes (input + n_cams x pixel bytes + 4 B mask per point) and
their share of the measured copy roofline (6550 GB/s, DESIGN.md section 3), the FP64 instructions per point and their
share of the FP64 pipe (FP64 configs), and the bound: the modelled one (HBM or FP64 pipe) the measured time reaches to
0.8 or more, otherwise "not determined".  A seeded sample of points of every timed batch is
checked against numpy FP64 (h = Xh @ P.T).  The card's name, power limit and max SM clock are read in the same run.
Prints one JSON line; --out also writes it to a file.

    python tools/bench_project.py [--points8 100000000] [--points32 20000000] [--reps 5] [--out profiles/project_bench.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT]

COPY_ROOFLINE = 6550.1e9  # B/s, measured device-to-device copy peak of a B200 (DESIGN.md section 3)
# NVIDIA data sheet, HGX B200, per GPU: FP64 37 TFLOP/s = 18.5e12 FP64 FMA-instructions/s (one FMA counts 2 flops)
FP64_INSTR_PEAK = 18.5e12
# FP64 pipe instructions per view in the kernel (tri_project.cu): w, x, y three DFMA each (9), the reciprocal
# (MUFU.RCP64H seed + four DFMA, 4 on the pipe), u and v (2), four bound compares (DSETP, 4) and w > 0 (1) = 20
FP64_PER_VIEW = 20
PIX_BYTES = {"float2": 8, "ushort2": 4}
BOUND_SHARE = 0.8


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def points(torch, n, seed):
    """Points around and beyond the synthetic volume (some views invisible), generated on the GPU from a seed."""
    g = torch.Generator(device="cuda:0")
    g.manual_seed(seed)
    lo = torch.tensor([-9000.0, -9000.0, -3000.0], dtype=torch.float64, device="cuda:0")
    hi = torch.tensor([9000.0, 9000.0, 9000.0], dtype=torch.float64, device="cuda:0")
    X = torch.rand((n, 3), dtype=torch.float64, device="cuda:0", generator=g)
    return lo + (hi - lo) * X


def numpy_check(cams, X, xy, mask, f64, pix):
    """The sample against numpy FP64: masks equal away from image borders, pixels within the precision's tolerance."""
    nc = len(cams)
    Xh = np.c_[X, np.ones(len(X))]
    band, tol = (1e-6, 1e-9) if f64 else (1e-2, 1e-3)
    ok_mask, ok_pix, thin = True, True, np.zeros(len(X), bool)
    for c, cam in enumerate(cams):
        h = Xh @ np.asarray(cam.P).T
        with np.errstate(all="ignore"):
            u, v = h[:, 0] / h[:, 2], h[:, 1] / h[:, 2]
        W, H = cam.width - 0.5, cam.height - 0.5
        vis = (h[:, 2] > 0) & (u >= -0.5) & (u < W) & (v >= -0.5) & (v < H)
        # FP32: the error grows as 1 / depth; the bounds hold from 2 m on and scale by 2 m / depth closer in
        scale = 1.0 if f64 else np.maximum(2000.0 / np.where(h[:, 2] > 0, h[:, 2], np.inf), 1.0)
        near = np.min(np.abs(np.stack([u + 0.5, u - W, v + 0.5, v - H])), axis=0) < band * scale
        thin |= near
        got = (mask >> c & 1).astype(bool)
        ok_mask &= bool(np.all((got == vis) | near))
        both = got & vis
        if pix == "float2":
            d = np.maximum(np.abs(xy[c, :, 0] - u), np.abs(xy[c, :, 1] - v))
            ok_pix &= bool(np.all((d < tol * scale + 2.5e-4)[both]))
        else:
            t = tol * scale
            tie = (np.abs(np.abs(u - np.floor(u)) - 0.5) < t) | (np.abs(np.abs(v - np.floor(v)) - 0.5) < t)
            sel = both & ~tie
            ok_pix &= bool(np.array_equal(xy[c, sel, 0], np.rint(u[sel])) and np.array_equal(xy[c, sel, 1], np.rint(v[sel])))
        ok_pix &= bool(np.all(xy[c, ~got] == (-1 if pix == "float2" else 0xFFFF)))
    return ok_mask, ok_pix, int(thin.sum())


def run_config(torch, T, S, nc, n, f64, pix, reps, warmup, sample):
    cams = S.ring_rig(32, rings=((6000.0, 3000.0), (9000.0, 5000.0))) if nc == 32 else S.ring_rig(nc)
    eng = T.Engine(cams, 0)
    X = points(torch, n, 1000 + nc)
    if not f64:
        X = X.float()
    tdt = torch.float32 if pix == "float2" else torch.uint16
    out = {"xy": torch.empty((nc, n, 2), dtype=tdt, device="cuda:0"), "mask": torch.empty((n,), dtype=torch.int32, device="cuda:0")}
    fl = 0 if f64 else T.F32
    for _ in range(warmup):
        eng.project_points_device(X, fl, out=out)
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in ev:
        a.record()
        eng.project_points_device(X, fl, out=out)
        b.record()
    torch.cuda.synchronize()
    ms = sorted(a.elapsed_time(b) for a, b in ev)
    t = ms[len(ms) // 2] * 1e-3
    bytes_pp = (24 if f64 else 12) + nc * PIX_BYTES[pix] + 4
    t_mem = n * bytes_pp / COPY_ROOFLINE
    res = {"cams": nc, "points": n, "precision": "fp64" if f64 else "fp32", "input": "float64 [n][3]" if f64 else "float32 [n][3]",
           "pixels": pix, "mask": True, "ms": round(ms[len(ms) // 2], 4), "ms_min": round(ms[0], 4), "points_per_s": n / t,
           "bytes_per_point": bytes_pp, "achieved_bytes_per_s": n * bytes_pp / t, "share_of_copy_roofline": t_mem / t}
    model = {"HBM": t_mem}
    if f64:
        model["FP64 pipe"] = n * nc * FP64_PER_VIEW / FP64_INSTR_PEAK
        res.update({"fp64_instr_per_point": nc * FP64_PER_VIEW, "share_of_fp64_pipe": model["FP64 pipe"] / t})
    # a modelled bound is named only when the measured time comes close to it (>= BOUND_SHARE of it); otherwise the
    # time is set by something neither model counts and the bound is left undetermined
    top = max(model, key=model.get)
    res["bound"] = top if model[top] / t >= BOUND_SHARE else "not determined (largest modelled share %.2f, %s)" % (model[top] / t, top)
    res["visible_fraction"] = float(sum(((out["mask"] >> c) & 1).sum().item() for c in range(nc)) / (n * nc))
    # numpy FP64 on a seeded ~2 M-point sample of the timed batch (drawn with replacement, duplicates collapsed)
    rng = np.random.default_rng(12345 + nc)
    idx = np.unique(rng.integers(0, n, size=min(sample, n)))
    it = torch.from_numpy(idx).to("cuda:0")
    Xs = X[it].double().cpu().numpy()
    xy = (out["xy"][:, it] if pix == "float2" else out["xy"].view(torch.int16)[:, it]).cpu().numpy()  # no uint16 gather
    if pix == "ushort2":
        xy = xy.view(np.uint16)
    mask = out["mask"][it].cpu().numpy().view(np.uint32)
    ok_mask, ok_pix, thin = numpy_check(cams, Xs, xy.astype(np.float64) if pix == "float2" else xy, mask, f64, pix)
    res.update({"check_sample": int(len(idx)), "check_border_points": thin, "check_masks_ok": ok_mask, "check_pixels_ok": ok_pix})
    del out, X
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--points8", type=int, default=100_000_000)
    ap.add_argument("--points32", type=int, default=20_000_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--sample", type=int, default=2_000_000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_project.py measures the GPU kernel: no CUDA device")
    import tri_b200 as T
    from tri_b200 import synthetic as S
    info = gpu_info()
    res = []
    for f64 in (True, False):
        for pix in ("float2", "ushort2"):
            res.append(run_config(torch, T, S, 8, a.points8, f64, pix, a.reps, a.warmup, a.sample))
    for f64 in (True, False):
        res.append(run_config(torch, T, S, 32, a.points32, f64, "float2", a.reps, a.warmup, a.sample))
    line = json.dumps({"bench": "project", "gpu": info, "copy_roofline_bytes_per_s": COPY_ROOFLINE,
                       "fp64_instr_peak_per_s": FP64_INSTR_PEAK, "configs": res,
                       "all_checks_ok": all(r["check_masks_ok"] and r["check_pixels_ok"] for r in res)})
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
