"""Launch each batch kernel variant a few times on device-resident synthetic frames (for ncu).
  python tools/profile_kernels.py [--frames N] [--reps R] [--only dlt_f64,dlt_f32,ray_f64,ray_f32,ray_ref]
Prints CUDA-event times per variant (never quote numbers taken under ncu)."""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
import tri_b200 as T  # noqa: E402
from tri_b200 import synthetic as S  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--frames", type=int, default=32_000_000)
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--cams", type=int, default=8)
ap.add_argument("--only", default="dlt_f64,dlt_f32,ray_f64,ray_f32")
a = ap.parse_args()
rings = ((6000.0, 3000.0),) if a.cams <= 8 else ((6000.0, 3000.0), (9000.0, 5000.0))
cams = S.ring_rig(a.cams, rings=rings)
eng = T.Engine(cams, 0)
xy = S.generate_frames(cams, a.frames, device="cuda:0")
out = {"xyz_f32": torch.empty((a.frames, 3), dtype=torch.float32, device="cuda:0")}
variants = {"dlt_f64": (T.MATRIX, 0), "dlt_f32": (T.MATRIX, T.F32), "ray_f64": (T.RAY, T.RAY_ANALYTIC_LM), "ray_f32": (T.RAY, T.F32),
            "ray_closed_f64": (T.RAY, 0), "ray_ref": (T.RAY, T.RAY_REFERENCE_LM)}
for name in a.only.split(","):
    mode, fl = variants[name]
    n = a.frames if name != "ray_ref" else min(a.frames, 200_000)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(a.reps + 1)]
    eng.triangulate_points_device(mode, xy, fl | T.ALLOW_TOO_FEW, out=out, n_frames=n)
    ev[0].record()
    for i in range(a.reps):
        eng.triangulate_points_device(mode, xy, fl | T.ALLOW_TOO_FEW, out=out, n_frames=n)
        ev[i + 1].record()
    torch.cuda.synchronize()
    ms = min([ev[i].elapsed_time(ev[i + 1]) for i in range(a.reps)] or [float('nan')])
    gb = (8 * a.cams + 12) * n / 1e9
    print("%-14s %9.3f ms  %8.1f GB/s  %.3e frames/s" % (name, ms, gb / (ms * 1e-3), n / (ms * 1e-3)), flush=True)
