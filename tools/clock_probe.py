"""Sustained-run probe: time N back-to-back launches of one kernel variant while sampling SM clock / power."""
import os, subprocess, sys, threading, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import tri_b200 as T
from tri_b200 import synthetic as S
name = sys.argv[1] if len(sys.argv) > 1 else "dlt_f32"
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 400
frames = int(sys.argv[3]) if len(sys.argv) > 3 else 100_000_000
variants = {"dlt_f64": (T.MATRIX, 0), "dlt_f32": (T.MATRIX, T.F32), "ray_f64": (T.RAY, 0)}
mode, fl = variants[name]
cams = S.ring_rig(8)
eng = T.Engine(cams, 0)
xy = S.generate_frames(cams, frames, device="cuda:0")
out = {"xyz_f32": torch.empty((frames, 3), dtype=torch.float32, device="cuda:0")}
rows = []
p = subprocess.Popen(["nvidia-smi", "--query-gpu=clocks.sm,clocks.mem,power.draw,clocks_event_reasons.active", "--format=csv,noheader,nounits", "-lms", "20"],
                     stdout=subprocess.PIPE, text=True)
threading.Thread(target=lambda: [rows.append((time.time(), l.strip())) for l in p.stdout], daemon=True).start()
time.sleep(0.3)
for _ in range(3):
    eng.triangulate_points_device(mode, xy, fl | T.ALLOW_TOO_FEW, out=out)
torch.cuda.synchronize()
ev = [torch.cuda.Event(enable_timing=True) for _ in range(reps + 1)]
t0 = time.time()
ev[0].record()
for i in range(reps):
    eng.triangulate_points_device(mode, xy, fl | T.ALLOW_TOO_FEW, out=out)
    ev[i + 1].record()
torch.cuda.synchronize()
t1 = time.time()
time.sleep(0.1)
p.terminate()
ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(reps)]
print(name, "first5 %.3f  mid %.3f  last5 %.3f ms" % (sum(ms[:5]) / 5, sum(ms[reps // 2:reps // 2 + 5]) / 5, sum(ms[-5:]) / 5))
inr = [r for t, r in rows if t0 <= t <= t1]
print("samples during run:", len(inr))
for r in inr[:: max(1, len(inr) // 12)]:
    print("   ", r)
print("idle before:", rows[0][1] if rows else None)
