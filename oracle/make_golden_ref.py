"""Golden vectors of what tests/test_gpu_ref.py compares the CUDA path with: the outputs of the reference's own code
(oracle/_ref) on the fixtures, as the C oracle reproduces them bit for bit.  tests/test_ref_parity.py checks every
array stored here against oracle/_ref wherever that is built, so a GPU machine needs neither the reference's sources
nor its build to run the comparison.
  golden_ref_<dataset>.npz
    matrix_assign / matrix_phase / matrix_paths   DroneClassifier::classifyDrones, --triangulator matrix, every frame
    matrix_err                                    the triangulatePoint error of every accepted combination (0 elsewhere)
    matrix_margin_error / matrix_margin_gate      the decision margins of that run (orc_last_margins)
    ray_assign / ray_phase / ray_paths            --triangulator ray (cv::LMSolver trajectory), first RAY_FRAMES frames
    batch_matrix_xyz / batch_ray_xyz              Triangulator::triangulatePoints (R02_D1: one drone, one detection each)
Run: python oracle/make_golden_ref.py"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import oracle_py as O  # noqa: E402

G = os.path.join(os.path.dirname(HERE), "tests", "golden")
DATASETS = {"R02_D1": 1, "R04_D2": 2, "S01_D2_A": 2, "S09_D6": 6}
RAY_FRAMES = {"R02_D1": None, "S09_D6": 300}


def accepted_errors(cams, res, offs, xy, nc, nf):
    o = offs.reshape(nc, nf + 1)
    err = np.zeros(res["phase"].shape)
    for p, f in zip(*np.nonzero(res["phase"])):
        sub = [c for c in range(nc) if res["assign"][p, f, c] > 0]
        err[p, f] = O.matrix_point(cams, sub, [xy[o[c, f] + res["assign"][p, f, c] - 1] for c in sub])[1]
    return err


def main():
    for ds, nd in DATASETS.items():
        cams = O.load_cameras("%s/%s_cameras.xml" % (G, ds))
        offs, xy, nc, nf = O.load_dets("%s/%s_dets.npz" % (G, ds))
        m = O.classify(cams, O.MATRIX, nd, offs, xy, nc, nf)
        out = dict(matrix_assign=m["assign"], matrix_phase=m["phase"], matrix_paths=m["paths"],
                   matrix_err=accepted_errors(cams, m, offs, xy, nc, nf),
                   matrix_margin_error=m["margins"]["error"], matrix_margin_gate=m["margins"]["gate"])
        if ds in RAY_FRAMES:
            fr = RAY_FRAMES[ds] or nf
            o, x, _, _ = O.slice_frames(offs, xy, nc, nf, 0, fr)
            r = O.classify(cams, O.RAY, nd, o, x, nc, fr)
            out.update(ray_assign=r["assign"], ray_phase=r["phase"], ray_paths=r["paths"])
        if ds == "R02_D1":
            pts = O.dets_to_points(offs, xy, nc, nf)
            out.update(batch_matrix_xyz=O.triangulate_points(cams, pts, O.MATRIX)["xyz"],
                       batch_ray_xyz=O.triangulate_points(cams, pts, O.RAY)["xyz"])
        path = "%s/golden_ref_%s.npz" % (G, ds)
        np.savez_compressed(path, **out)
        print(path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
