"""End-to-end (pinned host buffers -> tri_triangulate_points -> pinned host result) timing."""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import tri_b200 as T
from tri_b200 import synthetic as S
F = int(sys.argv[1]) if len(sys.argv) > 1 else 100_000_000
cams = S.ring_rig(8)
eng = T.Engine(cams, 0)
xy = S.generate_frames(cams, F, device="cuda:0")
h_xy = torch.empty((8, F, 2), dtype=torch.float32, pin_memory=True); h_xy.copy_(xy)
h_out = torch.empty((F, 3), dtype=torch.float32, pin_memory=True)
torch.cuda.synchronize()
for rep in range(4):
    t0 = time.perf_counter()
    eng.triangulate_points_raw(T.MATRIX, T.ALLOW_TOO_FEW, h_xy.data_ptr(), 8, F, F, xyz_f32_ptr=h_out.data_ptr())
    dt = time.perf_counter() - t0
    print("%.1f ms  %.2e frames/s  %.1f GB/s" % (dt * 1e3, F / dt, 76 * F / dt / 1e9), flush=True)
