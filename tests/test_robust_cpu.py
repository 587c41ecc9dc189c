"""CPU checks of the outlier-robust batch's contract on the FP64 oracle (orc_triangulate_points_robust), of the
projective-depth premise it rests on, and of the synthetic false detections that exercise it."""
import os

import numpy as np
import pytest

import oracle_py as O
import robust_oracle_py as R
import tri_b200 as T
from tri_b200 import synthetic as S

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
TAU = 10.0


def ocams(cams):
    return [O.make_camera(c.cam_id, c.width, c.height, c.focal, c.position, c.quat) for c in cams]


def project(cam, X):
    P = np.array(cam.P).reshape(3, 4)
    h = P @ np.append(X, 1.0)
    return h[:2] / h[2], h[2]


def frame(cams, pix):
    """one frame: pix[c] = (x, y) or None -> xy [n_cams][1][2]"""
    xy = np.full((len(cams), 1, 2), -1.0)
    for c, p in enumerate(pix):
        if p is not None:
            xy[c, 0] = p
    return xy


@pytest.fixture(scope="module")
def ring8():
    return ocams(S.ring_rig(8))


def test_one_gross_outlier_is_excluded(ring8):
    X = np.array([300.0, -200.0, 1200.0])
    pix = [project(c, X)[0] + 0.3 * np.cos(k) for k, c in enumerate(ring8)]
    pix[3] = pix[3] + np.array([250.0, -180.0])
    r = R.triangulate_points_robust(ring8, frame(ring8, pix), TAU)
    assert r["mask"][0] == 0xFF & ~(1 << 3)
    assert np.linalg.norm(r["xyz"][0] - X) < 5.0
    assert 0 < r["err"][0] < 1.0
    plain = O.triangulate_points(ring8, frame(ring8, pix), O.MATRIX)
    assert np.linalg.norm(plain["xyz"][0] - X) > 20 * np.linalg.norm(r["xyz"][0] - X)


def test_two_inconsistent_views_give_no_consensus(ring8):
    a, _ = project(ring8[0], np.array([0.0, 0.0, 1000.0]))
    b, _ = project(ring8[2], np.array([0.0, 1500.0, 2200.0]))
    r = R.triangulate_points_robust(ring8, frame(ring8, [a, None, b] + [None] * 5), TAU)
    assert r["status"] == O.OK and r["mask"][0] == 0 and np.isnan(r["err"][0]) and np.all(r["xyz"][0] == 0)


def test_hypothesis_behind_the_cameras_is_never_chosen(ring8):
    # a point outside the ring behind cameras 0 and 1 (they look inwards): its pixels reproject exactly, w < 0 on both
    X = 4.0 * (np.array(ring8[0].pos) + np.array(ring8[1].pos)) / 2
    (a, wa), (b, wb) = project(ring8[0], X), project(ring8[1], X)
    assert wa < 0 and wb < 0
    r = R.triangulate_points_robust(ring8, frame(ring8, [a, b] + [None] * 6), TAU)
    assert r["mask"][0] == 0 and np.isnan(r["err"][0])
    # with three consistent views in front, the front hypothesis wins
    Y = np.array([100.0, 100.0, 1000.0])
    pix = [project(ring8[c], Y)[0] if c in (2, 4, 6) else None for c in range(8)]
    pix[0], pix[1] = a, b
    r = R.triangulate_points_robust(ring8, frame(ring8, pix), TAU)
    assert r["mask"][0] == (1 << 2) | (1 << 4) | (1 << 6)


def test_tie_rules(ring8):
    A, B = np.array([-500.0, 400.0, 900.0]), np.array([600.0, -300.0, 1800.0])
    # count first: three noisy views of A beat two exact views of B
    pix = [None] * 8
    for c, d in ((0, 2.0), (2, -2.5), (4, 1.5)):
        pix[c] = project(ring8[c], A)[0] + d
    for c in (1, 5):
        pix[c] = project(ring8[c], B)[0]
    r = R.triangulate_points_robust(ring8, frame(ring8, pix), TAU)
    assert r["mask"][0] == (1 << 0) | (1 << 2) | (1 << 4)
    # equal counts: the smaller sum of squares wins although its pair comes later in (i, j) order
    pix = [None] * 8
    pix[0], pix[2] = project(ring8[0], A)[0] + 3.0, project(ring8[2], A)[0] - 3.0
    pix[5], pix[7] = project(ring8[5], B)[0], project(ring8[7], B)[0]
    r = R.triangulate_points_robust(ring8, frame(ring8, pix), TAU)
    assert r["mask"][0] == (1 << 5) | (1 << 7)
    # every pair of a consistent frame finds the same inlier set: the result does not depend on which pair it came from
    pix = [project(c, A)[0] for c in ring8]
    r = R.triangulate_points_robust(ring8, frame(ring8, pix), TAU)
    assert r["mask"][0] == 0xFF and r["err"][0] < 1e-6


def test_clean_data_gives_the_plain_dlt():
    cams = S.ring_rig(8)
    oc = ocams(cams)
    xy = S.generate_frames(cams, 3000).numpy()
    plain = O.triangulate_points(oc, xy, O.MATRIX, allow_too_few=True)
    r = R.triangulate_points_robust(oc, xy, TAU, allow_too_few=True)
    assert np.array_equal(r["mask"], plain["mask"])
    scale = np.maximum(np.abs(plain["xyz"]).max(axis=1, keepdims=True), 1.0)
    assert (np.abs(r["xyz"] - plain["xyz"]) / scale).max() < 1e-12


def test_too_few_views():
    cams = S.ring_rig(4)
    oc = ocams(cams)
    xy = S.generate_frames(cams, 50, p_missing=0.0).numpy()
    xy[1:, 7] = -1
    r = R.triangulate_points_robust(oc, xy, TAU)
    assert r["status"] == O.ERR_TOO_FEW and r["first_bad_frame"] == 7
    r = R.triangulate_points_robust(oc, xy, TAU, allow_too_few=True)
    assert r["status"] == O.OK and r["first_bad_frame"] == 7 and r["mask"][7] == 1 and r["err"][7] == 0


@pytest.mark.parametrize("name", ["R02_D1", "S09_D6"])
def test_visible_points_have_positive_projective_depth(name):
    cams = O.load_cameras(G + "/%s_cameras.xml" % name)
    if name == "R02_D1":  # one drone: the DLT point of every frame's detections is in front of every detecting camera
        offs, xy, nc, nf = O.load_dets(G + "/R02_D1_dets.npz")
        pts = O.dets_to_points(offs, xy, nc, nf)
        res = O.triangulate_points(cams, pts, O.MATRIX, allow_too_few=True)
        n = 0
        for f in range(nf):
            for c in range(nc):
                if res["mask"][f] >> c & 1 and bin(int(res["mask"][f])).count("1") >= 2:
                    P = np.array(cams[c].P).reshape(3, 4)
                    assert P[2] @ np.append(res["xyz"][f], 1.0) > 0
                    n += 1
        assert n > 1000
    else:  # six drones: the classifier's points (the DLT of each combination of detections) are in front of its cameras
        z = np.load(G + "/golden_S09_D6_classify_matrix.npz")
        n = 0
        for d in range(z["paths"].shape[0]):
            for f in range(z["paths"].shape[1]):
                for c in range(len(cams)):
                    if z["assign"][d, f, c] > 0:
                        P = np.array(cams[c].P).reshape(3, 4)
                        assert P[2] @ np.append(z["paths"][d, f], 1.0) > 0
                        n += 1
        assert n > 1000


def test_ring_rig_points_are_in_front():
    cams = S.ring_rig(8)
    _, truth = S.generate_frames(cams, 2000, want_truth=True)
    Xh = np.c_[truth.numpy(), np.ones(2000)]
    for c in cams:
        assert np.all(Xh @ np.array(c.P)[2] > 0)


def test_synthetic_outliers_replace_present_views_only():
    import torch
    cams = S.ring_rig(8)
    base = S.generate_frames(cams, 20000)
    assert torch.equal(S.generate_frames(cams, 20000, p_outlier=0.0), base)
    out = S.generate_frames(cams, 20000, p_outlier=0.1)
    missing = base[..., 0] == -1
    assert torch.equal(out[..., 0] == -1, missing)  # no view appears or disappears
    changed = (out != base).any(dim=2)
    assert 0.07 < changed.sum().item() / (~missing).sum().item() < 0.11
    for c, cam in enumerate(cams):
        x, y = out[c, changed[c], 0], out[c, changed[c], 1]
        assert (x >= 0).all() and (x < cam.width).all() and (y >= 0).all() and (y < cam.height).all()
    # keyed by the global frame index like the rest
    assert torch.equal(S.generate_frames(cams, 5000, frame0=12000, p_outlier=0.1), out[:, 12000:17000])
