"""Linking-pass timing loop: S09_D6 (3000 frames x 6 drones) and a synthetic 6-drone sequence, link_us from the call's own events.
  python tools/link_iter.py [--frames N]"""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "oracle"))
import numpy as np  # noqa: E402
import oracle_py as O  # noqa: E402  (fixture loader only)
import tri_b200 as T  # noqa: E402
from tri_b200 import synthetic as S  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--frames", type=int, default=20000)
a = ap.parse_args()
G = os.path.join(ROOT, "tests", "golden")
cams = T.load_cameras_xml(G + "/S09_D6_cameras.xml")
offs, xy, nc, nf = O.load_dets(G + "/S09_D6_dets.npz")
eng = T.Engine(cams, 0)
ref = None
for rep in range(4):
    r = eng.classify(T.MATRIX, 6, offs, xy, nf, 0)
    if ref is None:
        ref = r
    assert np.array_equal(ref["assign"], r["assign"]) and np.array_equal(ref["paths"], r["paths"])
    print("S09_D6 link_us %d (%.2f us/frame) enumerate_us %d phase1 %d phase2 %d" % (
        r["stats"]["link_us"], r["stats"]["link_us"] / nf, r["stats"]["enumerate_us"], r["stats"]["phase1"], r["stats"]["phase2"]), flush=True)
gold = os.path.join(G, "golden_S09_D6_classify_matrix.npz")
if os.path.exists(gold):
    g = np.load(gold)
    n = min(g["assign"].shape[1], nf)
    print("S09_D6 assignments equal to the golden file on %d frames:" % n, bool(np.array_equal(g["assign"][:, :n], ref["assign"][:, :n])))
rig = S.ring_rig(8)
so, sx, truth = S.generate_multi_drone(rig, a.frames, 6)
e2 = T.Engine(rig, 0)
for rep in range(3):
    r = e2.classify(T.MATRIX, 6, so, sx, a.frames, 0)
    print("synthetic 6 drones x %d frames: link_us %d (%.2f us/frame) enumerate_us %d phase1 %d phase2 %d" % (
        a.frames, r["stats"]["link_us"], r["stats"]["link_us"] / a.frames, r["stats"]["enumerate_us"], r["stats"]["phase1"], r["stats"]["phase2"]), flush=True)
