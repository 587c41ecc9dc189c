"""Pins the plain-C oracle and the golden vectors to the REFERENCE'S OWN CODE: oracle/_ref/libref.so is the
reference's Triangulator / MatrixTriangulator / RayTriangulator / DroneClassifier / DetectionsContainer / utils
sources and Camera.h compiled UNMODIFIED against oracle/shim (OpenCV C++ is not installed; the shim's third-party
arithmetic forwards to the cv2-pinned primitives of tri_oracle.c).  What these tests establish is that the control
flow the oracle restates -- Iterator DFS, fillCombinationQueue pruning, std::priority_queue / std::sort order,
tracking and re-initialisation -- is the reference's.  CPU only; skipped where oracle/_ref has not been built
(it needs /root/reference at build time)."""
import os

import numpy as np
import pytest

import oracle_py as O
import ref_py as R

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
pytestmark = pytest.mark.skipif(not R.available(), reason="oracle/_ref/libref.so not built (needs /root/reference)")

DATASETS = {"R02_D1": 1, "R04_D2": 2, "S01_D2_A": 2, "S09_D6": 6}


def load(ds, frames=None):
    xml = "%s/%s_cameras.xml" % (G, ds)
    offs, xy, nc, nf = O.load_dets("%s/%s_dets.npz" % (G, ds))
    if frames is not None and frames < nf:
        offs, xy, nc, nf = O.slice_frames(offs, xy, nc, nf, 0, frames)
    return xml, O.load_cameras(xml), offs, xy, nc, nf


def test_cameras_are_bit_identical_to_the_reference_loader():
    """loadCamerasXML + createCamera + Camera::compCamParams (utils.cpp:46-107, Camera.h:177-187), pugixml included."""
    for ds in DATASETS:
        xml, cams, *_ = load(ds)
        ref = R.Reference(xml=xml, mode=R.MATRIX)
        assert ref.n_cams == len(cams)
        for i, c in enumerate(cams):
            rc = ref.camera(i)
            assert np.array_equal(rc["P"].reshape(-1), np.array(c.P))
            assert np.array_equal(rc["K"].reshape(-1), np.array(c.K)) and np.array_equal(rc["E"].reshape(-1), np.array(c.E))
            assert (rc["fovx"], rc["fovy"], rc["fx"], rc["fy"], rc["cx"], rc["cy"]) == (c.fovx, c.fovy, c.fx, c.fy, c.cx, c.cy)
        # the same cameras through createCamera directly (what the engine's hosts feed)
        ref2 = R.Reference(cams=O.parse_cameras_xml(xml), mode=R.MATRIX)
        assert all(np.array_equal(ref2.camera(i)["P"], ref.camera(i)["P"]) for i in range(ref.n_cams))


@pytest.mark.parametrize("mode", [O.MATRIX, O.RAY])
def test_triangulate_points_and_its_errors(mode):
    xml, cams, offs, xy, nc, nf = load("R02_D1")
    pts = O.dets_to_points(offs, xy, nc, nf)
    ref = R.Reference(xml=xml, mode=mode)
    got = ref.triangulate_points(pts)
    orc = O.triangulate_points(cams, pts, mode)
    assert np.array_equal(got, orc["xyz"])  # MatrixTriangulator.cpp:70-100 / RayTriangulator.cpp:51-81
    g = np.load(G + "/golden_R02_D1_batch.npz")  # the cv2 twin's vectors
    key = "matrix_xyz" if mode == O.MATRIX else "ray_xyz"
    assert np.abs(got - g[key]).max() < (1e-8 if mode == O.MATRIX else 1e-3)
    bad = pts.copy()
    bad[1:, 7] = -1
    with pytest.raises(RuntimeError, match="Too few rays are found" if mode == O.MATRIX else "Too few detections are found"):
        ref.triangulate_points(bad)
    assert O.triangulate_points(cams, bad, mode)["status"] == O.ERR_TOO_FEW


def test_triangulate_point_subsets_and_dist_from_ray():
    xml, cams, offs, xy, nc, nf = load("R02_D1")
    pts = O.dets_to_points(offs, xy, nc, nf)
    rm, rr = R.Reference(xml=xml, mode=R.MATRIX), R.Reference(xml=xml, mode=R.RAY)
    rng = np.random.default_rng(5)
    for f in rng.integers(0, nf, 40):
        for sub in ([0, 1], [1, 3], [0, 2, 3], [0, 1, 2, 3]):
            X, e, _ = rm.triangulate_point(sub, pts[sub, f])
            Xo, eo = O.matrix_point(cams, sub, pts[sub, f])
            assert np.array_equal(X, Xo) and e == eo
            X, e, it = rr.triangulate_point(sub, pts[sub, f])
            Xo, eo, ito = O.ray_point(cams, sub, pts[sub, f])
            assert np.array_equal(X, Xo) and e == eo and it == ito
        p = rng.normal(0, 1500, 3)
        for c in range(nc):
            assert rm.dist_from_ray(c, pts[c, f, 0], pts[c, f, 1], p) == O.lib().orc_dist_from_ray(
                O.C.byref(cams[c]), O.C.c_double(pts[c, f, 0]), O.C.c_double(pts[c, f, 1]), O._p(np.ascontiguousarray(p)))


@pytest.mark.parametrize("ds,frames", [("R02_D1", None), ("R04_D2", None), ("S01_D2_A", None), ("S09_D6", 1000)])
def test_classifier_matrix_is_the_references(ds, frames):
    """classifyDrones run by the reference's own DroneClassifier.cpp: assignments (tapped at :130 and :315-321),
    phases and points equal the oracle's bit for bit, and the golden vectors' indices."""
    xml, cams, offs, xy, nc, nf = load(ds, frames)
    nd = DATASETS[ds]
    ref = R.Reference(xml=xml, mode=R.MATRIX).classify(nd, offs, xy, nf)
    orc = O.classify(cams, O.MATRIX, nd, offs, xy, nc, nf)
    assert np.array_equal(ref["assign"], orc["assign"]) and np.array_equal(ref["phase"], orc["phase"])
    assert np.array_equal(ref["paths"], orc["paths"])
    assert ref["stats"]["solves"] == orc["stats"]["solves"]
    assert (ref["stats"]["phase1"], ref["stats"]["phase2"]) == (orc["stats"]["phase1"], orc["stats"]["phase2"])
    for k in ("error", "step", "gate"):  # the two margin audits agree
        assert ref["margins"][k] == orc["margins"][k]
    g = np.load("%s/golden_%s_classify_matrix.npz" % (G, ds))
    n = min(ref["assign"].shape[1], g["assign"].shape[1])  # some goldens hold a prefix of the sequence
    assert np.array_equal(ref["assign"][:, :n], g["assign"][:, :n]) and np.array_equal(ref["phase"][:, :n], g["phase"][:, :n])
    np.testing.assert_allclose(ref["paths"][:, :n], g["paths"][:, :n], rtol=1e-9, atol=1e-6)


@pytest.mark.parametrize("ds,frames", [("R02_D1", 400), ("R04_D2", 150), ("S09_D6", 40)])
def test_classifier_ray_is_the_references(ds, frames):
    """--triangulator ray: cv::LMSolver's trajectory (shim LMSolverImpl::run over the reference's own
    RayClosestPoint::compute) reproduces the oracle's points, errors and total LM iterations exactly."""
    xml, cams, offs, xy, nc, nf = load(ds, frames)
    nd = DATASETS[ds]
    ref = R.Reference(xml=xml, mode=R.RAY).classify(nd, offs, xy, nf)
    orc = O.classify(cams, O.RAY, nd, offs, xy, nc, nf)
    assert np.array_equal(ref["assign"], orc["assign"]) and np.array_equal(ref["phase"], orc["phase"])
    assert np.array_equal(ref["paths"], orc["paths"])
    assert ref["stats"]["lm_iters"] == orc["stats"]["lm_iters"] and ref["stats"]["solves"] == orc["stats"]["solves"]


@pytest.mark.parametrize("ds", list(DATASETS))
def test_stored_reference_outputs_are_the_references(ds):
    """tests/golden/golden_ref_<ds>.npz (oracle/make_golden_ref.py), what tests/test_gpu_ref.py compares the CUDA path
    with, is what the reference's own code computes: classifier runs, accepted errors, margins, batch points."""
    z = np.load("%s/golden_ref_%s.npz" % (G, ds))
    xml, cams, offs, xy, nc, nf = load(ds)
    ref = R.Reference(xml=xml, mode=R.MATRIX).classify(DATASETS[ds], offs, xy, nf)
    for k in ("assign", "phase", "paths", "err"):
        assert np.array_equal(ref[k], z["matrix_" + k]), k
    assert ref["margins"]["error"] == z["matrix_margin_error"] and ref["margins"]["gate"] == z["matrix_margin_gate"]
    if "ray_paths" in z.files:
        xml, cams, offs, xy, nc, nf = load(ds, z["ray_paths"].shape[1])
        ref = R.Reference(xml=xml, mode=R.RAY).classify(DATASETS[ds], offs, xy, nf)
        for k in ("assign", "phase", "paths"):
            assert np.array_equal(ref[k], z["ray_" + k]), k
    if "batch_matrix_xyz" in z.files:
        pts = O.dets_to_points(offs, xy, nc, nf)
        for mode, k in ((R.MATRIX, "batch_matrix_xyz"), (R.RAY, "batch_ray_xyz")):
            assert np.array_equal(R.Reference(xml=xml, mode=mode).triangulate_points(pts), z[k]), k


def test_reference_cli_runs_end_to_end(tmp_path):
    """oracle/_ref/ref_main is the reference's main.cpp: same flags, ./results/drone<i>.ply, 'Execution time' line."""
    import subprocess
    if not os.path.exists(R.MAIN):
        pytest.skip("ref_main not built")
    d = np.load(G + "/R02_D1_dets.npz")
    data = tmp_path / "dl_data"
    data.mkdir()
    counts, xy = d["counts"], d["xy"]
    k = 0
    for c in range(counts.shape[0]):  # the 8-column rows of dataset/R02_D1/dl_data (frame, x, y, w, h, cx, cy, conf)
        with open(data / ("cam%d.csv" % c), "w") as f:
            for fr in range(60):
                row = [str(fr)]
                for _ in range(counts[c, fr]):
                    row += ["0", "0", "0", "0", str(int(xy[k, 0])), str(int(xy[k, 1])), "0.9"]
                    k += 1
                f.write(",".join(row) + "\n")
            k += int(counts[c, 60:].sum())
    out = subprocess.run([R.MAIN, G + "/R02_D1_cameras.xml", str(data)], cwd=tmp_path, capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr
    assert "0 / 60" in out.stdout and "Execution time:" in out.stdout
    ply = (tmp_path / "results" / "drone1.ply").read_text().split("end_header\n")[1].split("\n")
    pts = np.array([[float(v) for v in l.split()] for l in ply if l])
    g = np.load(G + "/golden_R02_D1_classify_matrix.npz")["paths"][0, :60]
    assert pts.shape == (60, 3) and np.abs(pts - g).max() < 2e-2 * np.abs(g).max() / 1e2 + 0.5  # 6 significant digits in the PLY
