"""GPU checks of the outlier-robust batch (tri_triangulate_points_robust / _device) against the FP64 CPU restatement of
its contract (oracle orc_triangulate_points_robust) and against the plain DLT on clean data."""
import os
import subprocess

import numpy as np
import pytest

import oracle_py as O
import robust_oracle_py as R
import tri_b200 as T
from tri_b200 import synthetic as S

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = os.path.join(ROOT, "tests", "golden")
EXTENT = 1e4  # mm: the synthetic rigs span ~10 m
TAU = 10.0


def ocams(cams):
    return [O.make_camera(c.cam_id, c.width, c.height, c.focal, c.position, c.quat) for c in cams]


def rig(nc):
    return S.ring_rig(32, rings=((6000.0, 3000.0), (9000.0, 5000.0))) if nc == 32 else S.ring_rig(nc)


@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available()
    return torch


@pytest.mark.parametrize("nc", [3, 8, 12, 32])
def test_clean_data_equals_plain_dlt(torch, nc):
    cams = rig(nc)
    eng = T.Engine(cams, 0)
    xy = S.generate_frames(cams, 40001).numpy()
    plain = eng.triangulate_points(T.MATRIX, xy, T.ALLOW_TOO_FEW, want=("xyz_f64", "mask"))
    rob = eng.triangulate_points_robust(xy, TAU, T.ALLOW_TOO_FEW)
    assert np.array_equal(rob["mask"], plain["mask"])
    ok = np.array([bin(int(m)).count("1") >= 2 for m in plain["mask"]])
    scale = np.maximum(np.abs(plain["xyz_f64"]).max(axis=1, keepdims=True), 1.0)
    assert (np.abs(rob["xyz_f64"] - plain["xyz_f64"]) / scale).max() < 1e-12
    assert np.all(rob["err"][ok] < TAU) and np.all(rob["err"][~ok] == 0)
    r32 = eng.triangulate_points_robust(xy, TAU, T.ALLOW_TOO_FEW | T.F32, want=("xyz_f32", "mask"))
    assert np.array_equal(r32["mask"], plain["mask"])
    assert np.abs(r32["xyz_f32"] - plain["xyz_f64"]).max() < 1e-4 * EXTENT


@pytest.mark.parametrize("p_out", [0.1, 0.3])
@pytest.mark.parametrize("nc", [3, 5, 8, 12, 32])
def test_outliers_against_oracle(torch, nc, p_out):
    cams = rig(nc)
    eng = T.Engine(cams, 0)
    n = 20000 if nc < 32 else 4000
    xy0, truth = S.generate_frames(cams, n, want_truth=True)
    xy = S.generate_frames(cams, n, p_outlier=p_out).numpy()
    xy0, truth = xy0.numpy(), truth.numpy()
    ref = R.triangulate_points_robust(ocams(cams), xy, TAU, allow_too_few=True)
    got = eng.triangulate_points_robust(xy, TAU, T.ALLOW_TOO_FEW)
    thin = ref["margin"] < 1e-9
    assert thin.mean() < 1e-3
    same = got["mask"] == ref["mask"]
    assert np.all(same | thin), np.nonzero(~(same | thin))[0][:10]
    both = same & (ref["mask"] != 0)
    scale = np.maximum(np.abs(ref["xyz"][both]).max(axis=1, keepdims=True), 1.0)
    assert (np.abs(got["xyz_f64"][both] - ref["xyz"][both]) / scale).max() < 1e-9
    assert np.allclose(got["err"][both], ref["err"][both], rtol=1e-9, atol=1e-9)
    assert np.all(np.isnan(got["err"][same & (ref["mask"] == 0) & (ref["err"] != 0)]))
    # FP32: the same decisions wherever the FP64 oracle's margin exceeds the FP32 tier
    g32 = eng.triangulate_points_robust(xy, TAU, T.ALLOW_TOO_FEW | T.F32, want=("xyz_f32", "mask"))
    ok32 = (g32["mask"] == ref["mask"]) | (ref["margin"] < 1e-3)
    assert np.all(ok32), np.nonzero(~ok32)[0][:10]
    # accuracy: the plain DLT is wrecked by the outliers, the robust one stays within 2x of the clean DLT
    clean = eng.triangulate_points(T.MATRIX, xy0, T.ALLOW_TOO_FEW, want=("xyz_f64", "mask"))
    okc = np.array([bin(int(m)).count("1") >= 2 for m in clean["mask"]])
    d_clean = np.median(np.linalg.norm(clean["xyz_f64"][okc] - truth[okc], axis=1))
    okr = got["mask"] != 0
    d_rob = np.median(np.linalg.norm(got["xyz_f64"][okr] - truth[okr], axis=1))
    assert d_rob < 2 * d_clean, (d_rob, d_clean)


def test_pixel_formats_tails_and_unaligned_stride(torch):
    cams = rig(8)
    eng = T.Engine(cams, 0)
    n = 2 * 256 * 7 + 36  # not a multiple of the tile
    xy = S.generate_frames(cams, n, p_outlier=0.2).numpy()
    ref = R.triangulate_points_robust(ocams(cams), xy, TAU, allow_too_few=True)
    thick = ref["margin"] >= 1e-9
    u16 = S.generate_frames(cams, n, p_outlier=0.2, dtype=torch.uint16).numpy()
    assert np.array_equal(R.triangulate_points_robust(ocams(cams), u16, TAU, allow_too_few=True)["mask"], ref["mask"])
    for arr in (xy, xy.astype(np.float64), u16):
        got = eng.triangulate_points_robust(arr, TAU, T.ALLOW_TOO_FEW)
        assert np.array_equal(got["mask"][thick], ref["mask"][thick])
        both = thick & (ref["mask"] != 0)
        assert np.abs(got["xyz_f64"][both] - ref["xyz"][both]).max() < 1e-9 * EXTENT
    # device entry point with a camera stride that is not a multiple of the vector width (odd, not 16-byte aligned rows)
    base = torch.from_numpy(xy).cuda()
    wide = torch.full((8, n + 1, 2), -1.0, dtype=torch.float32, device="cuda:0")
    wide[:, :n] = base
    view = wide[:, :n]
    assert view.stride(0) // 2 == n + 1 and (n + 1) % 2 == 1
    got = eng.triangulate_points_robust_device(view, TAU, T.ALLOW_TOO_FEW)
    st, bad = eng.device_status()
    assert st == T.OK and bad == -1
    assert np.array_equal(got["mask"].cpu().numpy().view(np.uint32)[thick], ref["mask"][thick])


def test_too_few_status_matches_plain(torch):
    cams = rig(5)
    eng = T.Engine(cams, 0)
    xy = S.generate_frames(cams, 5000, p_missing=0.0, p_outlier=0.1).numpy()
    xy[1:, 1234] = -1.0  # one view left
    xy[:, 3000] = -1.0  # none
    with pytest.raises(T.TriError) as e1:
        eng.triangulate_points(T.MATRIX, xy)
    with pytest.raises(T.TriError) as e2:
        eng.triangulate_points_robust(xy, TAU)
    assert e1.value.status == e2.value.status == T.ERR_TOO_FEW and str(e2.value) == str(e1.value) == "Too few rays are found"
    plain = eng.triangulate_points(T.MATRIX, xy, T.ALLOW_TOO_FEW, want=("xyz_f64", "mask", "err"))
    rob = eng.triangulate_points_robust(xy, TAU, T.ALLOW_TOO_FEW)
    assert plain["first_bad_frame"] == rob["first_bad_frame"] == 1234
    for f in (1234, 3000):
        assert rob["mask"][f] == plain["mask"][f] and np.all(rob["xyz_f64"][f] == 0) and rob["err"][f] == 0
    ref = R.triangulate_points_robust(ocams(cams), xy, TAU)
    assert ref["status"] == O.ERR_TOO_FEW and ref["first_bad_frame"] == 1234


def test_device_entry_point_matches_host(torch):
    cams = rig(8)
    eng = T.Engine(cams, 0)
    n = 300001
    xy = S.generate_frames(cams, n, p_outlier=0.1, device="cuda:0")
    xy[:, 77777] = -1.0
    first = eng.triangulate_points(T.MATRIX, xy.cpu().numpy(), T.ALLOW_TOO_FEW, want=("xyz_f32", "mask"))["first_bad_frame"]
    assert 0 <= first <= 77777
    for fl in (0, T.F32):
        dev = eng.triangulate_points_robust_device(xy, TAU, T.ALLOW_TOO_FEW | fl, want=("xyz_f64", "xyz_f32", "mask", "err"))
        st, bad = eng.device_status()
        assert st == T.ERR_TOO_FEW and bad == first
        host = eng.triangulate_points_robust(xy.cpu().numpy(), TAU, T.ALLOW_TOO_FEW | fl, want=("xyz_f64", "xyz_f32", "mask", "err"))
        assert host["first_bad_frame"] == first
        for k in ("xyz_f64", "xyz_f32", "err"):
            assert np.array_equal(dev[k].cpu().numpy(), host[k], equal_nan=True), k
        assert np.array_equal(dev["mask"].cpu().numpy().view(np.uint32), host["mask"])


def test_argument_checks(torch):
    import ctypes as C
    cams = rig(4)
    eng = T.Engine(cams, 0)
    xy = S.generate_frames(cams, 100).numpy()
    for fl in (T.RAY_REFERENCE_LM, T.RAY_CLOSED_FORM, T.RAY_ANALYTIC_LM, T.CLS_LAZY, 1 << 12):
        with pytest.raises(T.TriError) as e:
            eng.triangulate_points_robust(xy, TAU, fl)
        assert e.value.status == T.ERR_ARG
    for tau in (0.0, -1.0, float("nan")):
        with pytest.raises(T.TriError) as e:
            eng.triangulate_points_robust(xy, tau)
        assert e.value.status == T.ERR_ARG
    xyz, it = np.zeros((100, 3)), np.zeros(100, np.int32)
    bo = T._BatchOut(None, xyz.ctypes.data, None, None, it.ctypes.data)
    st = T.lib().tri_triangulate_points_robust(eng._h, 0, TAU, C.c_void_p(xy.ctypes.data), 4, 100, 100, C.byref(bo), None)
    assert st == T.ERR_ARG
    d = torch.from_numpy(xy).cuda()
    itd = torch.zeros(100, dtype=torch.int32, device="cuda:0")
    xd = torch.zeros((100, 3), dtype=torch.float64, device="cuda:0")
    bo = T._BatchOut(None, xd.data_ptr(), None, None, itd.data_ptr())
    st = T.lib().tri_triangulate_points_robust_device(eng._h, 0, TAU, C.c_void_p(d.data_ptr()), 4, 100, 100, C.byref(bo), None)
    assert st == T.ERR_ARG


def test_cpp_adapter_matches_python(torch, tmp_path):
    host = os.path.join(ROOT, "3d-reconstruction-triangulation_b200", "host")
    subprocess.check_call(["make", "-s", "-C", host])
    cams = T.load_cameras_xml(G + "/R02_D1_cameras.xml")
    offs, dxy, nc, nf = O.load_dets(G + "/R02_D1_dets.npz")
    pts = O.dets_to_points(offs, dxy, nc, nf)
    pts = pts[:, (pts[:, :, 0] != -1).sum(axis=0) >= 2]  # the adapter throws on a frame with < 2 views, like triangulatePoints
    nf = pts.shape[1]
    # a false detection on camera 0 in every 7th frame that has one
    pts = pts.copy()
    rows = [f for f in range(0, nf, 7) if pts[0, f, 0] != -1]
    pts[0, rows] = [[17.0, 23.0]]
    np.save(tmp_path / "pts.npy", pts)
    with open(tmp_path / "pts.txt", "w") as fh:
        fh.write("%d %d\n" % (nc, nf))
        for c in range(nc):
            fh.write(" ".join("%.17g %.17g" % (x, y) for x, y in pts[c]) + "\n")
    out = subprocess.check_output([os.path.join(host, "host_robust_selftest"), G + "/R02_D1_cameras.xml", str(tmp_path / "pts.txt"),
                                   str(TAU)], text=True).splitlines()
    eng = T.Engine(cams, 0)
    ref = eng.triangulate_points_robust(pts, TAU, T.ALLOW_TOO_FEW)
    pl = [l.split() for l in out if l.startswith("robust ")]
    assert len(pl) == nf
    xyz = np.array([[float(v) for v in p[2:5]] for p in pl])
    mask = np.array([int(p[5]) for p in pl], np.uint32)
    rms = np.array([float(p[6]) for p in pl])
    assert np.array_equal(mask, ref["mask"])
    assert np.array_equal(xyz, ref["xyz_f64"])
    assert np.array_equal(rms, ref["err"], equal_nan=True)
    lines = dict(l.split(" ", 1) for l in out if l.startswith("throw_"))
    assert lines["throw_dim"] == "Every camera should have the same number of points"
    assert lines["throw_few"] == "Too few rays are found"
