"""GPU parity against the REFERENCE'S OWN CODE plus the margin audit of SURVEY.md H7: the engine computes the
matrix-mode `error` from the normal equations while the reference takes an SVD pseudo-inverse, so index parity holds
exactly as long as no threshold / ordering compare is closer than that arithmetic difference -- measured here, with a
factor 1e3 in hand.  What the reference computes on the fixtures is stored under tests/golden/golden_ref_<dataset>.npz
(oracle/make_golden_ref.py); tests/test_ref_parity.py checks those vectors against the reference's sources compiled
unmodified against oracle/shim (oracle/_ref/libref.so) wherever that is built."""
import os

import numpy as np
import pytest

import oracle_py as O
import tri_b200 as T

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
DATASETS = {"R02_D1": 1, "R04_D2": 2, "S01_D2_A": 2, "S09_D6": 6}


def load(ds, frames=None):
    xml = "%s/%s_cameras.xml" % (G, ds)
    offs, xy, nc, nf = O.load_dets("%s/%s_dets.npz" % (G, ds))
    if frames is not None and frames < nf:
        offs, xy, nc, nf = O.slice_frames(offs, xy, nc, nf, 0, frames)
    return xml, T.load_cameras_xml(xml), offs, xy, nc, nf


def reference(ds, kind):
    """The reference's output stored for `ds`: kind 'matrix' | 'ray' (classifier) or 'batch'."""
    z = np.load("%s/golden_ref_%s.npz" % (G, ds))
    return {k[len(kind) + 1:]: z[k] for k in z.files if k.startswith(kind + "_")}


def accepted_items(res, offs, xy, nc, nf):
    """(camera subset, pixels) of every accepted combination, for tri_triangulate_subsets."""
    o = offs.reshape(nc, nf + 1)
    items, where = [], []
    for p, f in zip(*np.nonzero(res["phase"])):
        cams = [c for c in range(nc) if res["assign"][p, f, c] > 0]
        pix = [xy[o[c, f] + res["assign"][p, f, c] - 1] for c in cams]
        items.append((cams, np.array(pix)))
        where.append((p, f))
    return items, where


@pytest.mark.parametrize("ds", list(DATASETS))
def test_matrix_classifier_equals_the_reference_and_margins_hold(ds):
    xml, cams, offs, xy, nc, nf = load(ds)
    nd = DATASETS[ds]
    ref = reference(ds, "matrix")
    eng = T.Engine(cams, 0)
    got = eng.classify(T.MATRIX, nd, offs, xy, nf)
    assert np.array_equal(got["assign"], ref["assign"])  # bit-exact indices (DroneClassifier.cpp:130, :315-321)
    assert np.array_equal(got["phase"], ref["phase"])
    scale = np.maximum(np.abs(ref["paths"]).max(axis=2, keepdims=True), 1.0)
    assert (np.abs(got["paths"] - ref["paths"]) / scale).max() < 1e-6
    # margin audit: the engine's error / point of every accepted combination against the reference's
    items, where = accepted_items(ref, offs, xy, nc, nf)
    sub_xyz, sub_err, _ = eng.triangulate_subsets(T.MATRIX, items)
    ref_err = np.array([ref["err"][p, f] for p, f in where])
    ref_pts = np.array([ref["paths"][p, f] for p, f in where])
    d_err = np.abs(sub_err - ref_err).max()
    d_pt = np.abs(sub_xyz - ref_pts).max()
    orc = O.classify(O.load_cameras(xml), O.MATRIX, nd, offs, xy, nc, nf)  # same decisions (test_ref_parity), all five margins
    m = orc["margins"]
    assert m["error"] == ref["margin_error"] and m["gate"] == ref["margin_gate"]
    print("%s: |d error| %.3e, |d point| %.3e mm; margins %s" % (ds, d_err, d_pt, {k: float("%.3g" % v) for k, v in m.items()}))
    assert min(m["error"], m["order"]) >= 1e3 * d_err   # error_ threshold and priority order (on the error)
    assert min(m["step"], m["tail"]) >= 1e3 * d_pt      # MAX_STEP and tail distances (on the point)
    assert m["gate"] > 1e-7                             # the ray gate runs the reference's own operation order (bit-identical, test_gpu_batch)


@pytest.mark.parametrize("ds,frames", [("R02_D1", None), ("S09_D6", 300)])
def test_ray_classifier_reference_lm_equals_the_reference(ds, frames):
    """--triangulator ray with cv::LMSolver's trajectory: points bit-identical to the reference's, incl. its
    non-converged 2-view solves (SURVEY F5)."""
    xml, cams, offs, xy, nc, nf = load(ds, frames)
    nd = DATASETS[ds]
    ref = reference(ds, "ray")
    assert ref["paths"].shape[1] == nf
    got = T.Engine(cams, 0).classify(T.RAY, nd, offs, xy, nf, T.RAY_REFERENCE_LM)
    assert np.array_equal(got["assign"], ref["assign"]) and np.array_equal(got["phase"], ref["phase"])
    assert np.array_equal(got["paths"], ref["paths"])


@pytest.mark.parametrize("mode", [T.MATRIX, T.RAY])
def test_batch_points_against_the_reference(mode):
    xml, cams, offs, xy, nc, nf = load("R02_D1")
    pts = O.dets_to_points(offs, xy, nc, nf)
    want = reference("R02_D1", "batch")["matrix_xyz" if mode == T.MATRIX else "ray_xyz"]
    eng = T.Engine(cams, 0)
    got = eng.triangulate_points(mode, pts, want=("xyz_f64",))["xyz_f64"]  # matrix: normal equations; ray: the batch default
    scale = np.maximum(np.abs(want).max(axis=1, keepdims=True), 1.0)
    tol = 1e-6 if mode == T.MATRIX else 2e-6  # ray: the reference's LM stops within ~1e-3 mm of the minimiser the engine returns
    assert (np.abs(got - want) / scale).max() < tol
    if mode == T.RAY:
        ex = eng.triangulate_points(mode, pts, T.RAY_REFERENCE_LM, want=("xyz_f64",))["xyz_f64"]
        assert np.array_equal(ex, want)
