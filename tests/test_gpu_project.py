"""GPU checks of the forward projection (tri_project_points / _device): parity with numpy FP64 (h = Xh @ P.T, true
division, the visibility rule of include/tri_b200.h), invisible views, the round trip through the batch triangulation,
the batch layout (strides, odd sizes, unaligned bases, host vs device) and the argument checks."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import tri_b200 as T
from tri_b200 import synthetic as S

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PIX = {"f32": np.float32, "f64": np.float64, "u16": np.uint16}
MARK = {"f32": -1.0, "f64": -1.0, "u16": 0xFFFF}
TOL = {0: 1e-9, T.F32: 1e-3}  # px: FP64 / FP32 compute
BORDER = {0: 1e-6, T.F32: 1e-2}  # px: masks may differ this close to an image border
# The FP32 error of a pixel grows as 1 / depth (the rounding of the centred point and constants over the depth): the FP32
# bounds hold from a depth of 2 m on and scale by 2 m / depth closer in (worst on the 32-camera rig, estimated on the CPU
# with FP32 FMA chains: 1.4e-3 px at 0.85 m from an outer-ring camera, 13 m from the rig centre)
NEAR_MM = 2000.0


@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available()
    return torch


def rig(nc):
    return S.ring_rig(32, rings=((6000.0, 3000.0), (9000.0, 5000.0))) if nc == 32 else S.ring_rig(nc)


def ref_project(cams, X):
    """numpy FP64: u, v [nc, n], visibility [nc, n], mask [n], distance of (u, v) to the nearest image border [nc, n],
    depth w [nc, n]."""
    X = np.asarray(X, np.float64)
    n = len(X)
    Xh = np.c_[X, np.ones(n)]
    fin = np.isfinite(X).all(axis=1)
    u, v, vis, dist, w = (np.empty((len(cams), n)) for _ in range(5))
    vis = vis.astype(bool)
    with np.errstate(all="ignore"):
        for c, cam in enumerate(cams):
            h = Xh @ np.asarray(cam.P).T
            u[c], v[c], w[c] = h[:, 0] / h[:, 2], h[:, 1] / h[:, 2], h[:, 2]
            W, H = cam.width - 0.5, cam.height - 0.5
            vis[c] = fin & (h[:, 2] > 0) & (u[c] >= -0.5) & (u[c] < W) & (v[c] >= -0.5) & (v[c] < H)
            dist[c] = np.min(np.abs(np.stack([u[c] + 0.5, u[c] - W, v[c] + 0.5, v[c] - H])), axis=0)
    mask = (vis.astype(np.uint64) << np.arange(len(cams), dtype=np.uint64)[:, None]).sum(axis=0).astype(np.uint32)
    return u, v, vis, mask, np.where(np.isfinite(dist), dist, np.inf), w


def wide_points(n, seed=7):
    """Points around and beyond the synthetic volume: many views behind a camera or outside its image."""
    r = np.random.default_rng(seed)
    return np.stack([r.uniform(-9000, 9000, n), r.uniform(-9000, 9000, n), r.uniform(-3000, 9000, n)], axis=1)


def bits(mask, nc):
    return ((mask.astype(np.uint64)[None, :] >> np.arange(nc, dtype=np.uint64)[:, None]) & 1).astype(bool)


def check_against_ref(cams, X, out, fmt, fl):
    """out: {"xy", "mask"} of one projection in format `fmt` under flags `fl`, against numpy FP64."""
    nc = len(cams)
    u, v, vis, mask, dist, w = ref_project(cams, X)
    scale = 1.0 if fl == 0 else np.maximum(NEAR_MM / np.where(w > 0, w, np.inf), 1.0)  # FP32: 1 / depth closer than 2 m
    near = dist < BORDER[fl] * scale
    thin = near.any(axis=0)
    assert thin.mean() < 1e-3
    assert np.array_equal(out["mask"][~thin], mask[~thin])
    got = bits(out["mask"], nc)
    xy = out["xy"]
    # every invisible view holds the marker
    assert np.all(xy[~got] == MARK[fmt])
    both = got & vis
    if fmt == "u16":
        eps = 1e-6 if fl == 0 else TOL[fl] * scale
        for a, ref in ((xy[..., 0], u), (xy[..., 1], v)):
            tie = np.abs(np.abs(ref - np.floor(ref)) - 0.5) < eps
            ok = both & ~tie
            assert np.array_equal(a[ok].astype(np.float64), np.rint(ref[ok]))
    else:
        tol = (TOL[fl] * scale + (2.5e-4 if fmt == "f32" else 0.0)) * np.ones_like(u)  # float2: a pixel's float rounding
        assert np.all(np.abs(xy[..., 0][both].astype(np.float64) - u[both]) < tol[both])
        assert np.all(np.abs(xy[..., 1][both].astype(np.float64) - v[both]) < tol[both])


@pytest.mark.parametrize("in_dtype", [np.float32, np.float64])
@pytest.mark.parametrize("fl", [0, T.F32])
@pytest.mark.parametrize("nc", [1, 3, 8, 12, 32])
def test_parity_with_numpy(torch, nc, fl, in_dtype):
    cams = rig(nc)
    eng = T.Engine(cams, 0)
    X = wide_points(100003).astype(in_dtype)
    _, _, vis, _, _, _ = ref_project(cams, X)
    assert 0.05 < vis.mean() < 0.95  # both visible and invisible views are exercised
    for fmt, dt in PIX.items():
        out = eng.project_points(X, fl, pix_dtype=dt)
        assert out["xy"].shape == (nc, len(X), 2) and out["xy"].dtype == dt
        check_against_ref(cams, X, out, fmt, fl)


def edge_points(cam, eps=1e-3, depth=6000.0):
    """Points that project 1e-3 px inside / outside each of the four image edges of `cam` (FP64 back-projection);
    -> (points [8, 3], expected visibility [8])."""
    P = np.asarray(cam.P)
    M, p4 = P[:, :3], P[:, 3]
    Mi = np.linalg.inv(M)
    centre = -Mi @ p4
    W, H = cam.width, cam.height
    cu, cv = W / 2.0, H / 2.0
    pix, exp = [], []
    for inside in (True, False):
        s = eps if inside else -eps
        pix += [(-0.5 + s, cv), (W - 0.5 - s, cv), (cu, -0.5 + s), (cu, H - 0.5 - s)]
        exp += [inside] * 4
    pts = np.array([centre + depth * (Mi @ np.array([a, b, 1.0])) for a, b in pix])
    return pts, np.array(exp)


def test_invisible_views(torch):
    cams = rig(8)
    nc = len(cams)
    eng = T.Engine(cams, 0)
    pos = np.array([c.position for c in cams])
    behind = pos * np.array([1.5, 1.5, 1.0])  # outside the ring, on each camera's own side: behind it
    above = np.array([[0.0, 0.0, 1e6], [3000.0, -2000.0, 2e5]])  # far above the frustums
    edges, exp = edge_points(cams[0])
    nonfin = np.array([[np.nan, 0, 1000], [0, np.nan, 1000], [0, 0, np.nan], [np.inf, 0, 1000], [0, -np.inf, 1000],
                       [0, 0, np.inf], [np.nan, np.inf, -np.inf]])
    X = np.concatenate([behind, above, edges, nonfin])
    u, v, vis, mask, dist, _ = ref_project(cams, X)
    nb, na, ne = len(behind), len(above), len(edges)
    assert not vis[np.arange(nb), np.arange(nb)].any()  # each camera misses the point behind it
    assert not vis[:, nb:nb + na].any() and not vis[:, nb + na + ne:].any()
    assert np.array_equal(vis[0, nb + na:nb + na + ne], exp)
    for xyz_dt in (np.float64, np.float32):
        for fl in (0, T.F32):
            Xi = X.astype(xyz_dt)
            for fmt, dt in PIX.items():
                out = eng.project_points(Xi, fl, pix_dtype=dt)
                got = bits(out["mask"], nc)
                assert np.all(out["xy"][~got] == MARK[fmt])  # the marker in every format
                assert not got[np.arange(nb), np.arange(nb)].any()
                assert np.all(out["mask"][nb:nb + na] == 0) and np.all(out["mask"][nb + na + ne:] == 0)
                if fl == 0 and xyz_dt == np.float64:  # FP64: the rule holds 1e-3 px from each edge
                    assert np.array_equal(got[0, nb + na:nb + na + ne], exp)
                    assert np.array_equal(out["mask"], mask)


def test_round_trip_through_triangulation(torch):
    cams = rig(8)
    eng = T.Engine(cams, 0)
    r = np.random.default_rng(3)
    n = 200001
    X = np.stack([r.uniform(-4500, 4500, n), r.uniform(-4500, 4500, n), r.uniform(-500, 4000, n)], axis=1)
    pr = eng.project_points(X, 0, pix_dtype=np.float64)
    k = np.array([bin(int(m)).count("1") for m in pr["mask"]])
    ok = k >= 2
    assert ok.mean() > 0.5 and (k < len(cams)).mean() > 0.1  # partial visibility is exercised
    tri = eng.triangulate_points(T.MATRIX, pr["xy"], T.ALLOW_TOO_FEW, want=("xyz_f64", "mask"))
    assert np.array_equal(tri["mask"][ok], pr["mask"][ok])
    scale = np.maximum(np.abs(X[ok]).max(axis=1), 1.0)
    assert (np.linalg.norm(tri["xyz_f64"][ok] - X[ok], axis=1) / scale).max() < 1e-9
    rob = eng.triangulate_points_robust(pr["xy"], 10.0, T.ALLOW_TOO_FEW)
    assert np.array_equal(rob["mask"][ok], pr["mask"][ok])
    assert rob["err"][ok].max() < 1e-6


def test_u16_matches_synthetic_generator(torch):
    for nc in (8, 32):
        cams = rig(nc)
        eng = T.Engine(cams, 0)
        n = 100000
        gen, truth = S.generate_frames(cams, n, noise_px=0.0, p_missing=0.0, dtype=torch.uint16, want_truth=True)
        gen, truth = gen.numpy(), truth.numpy()
        out = eng.project_points(truth, 0, pix_dtype=np.uint16)
        assert np.all(out["mask"] == np.uint32((1 << nc) - 1))  # the synthetic volume is visible in every camera
        u, v, _, _, _, _ = ref_project(cams, truth)
        tie = (np.abs(np.abs(u - np.floor(u)) - 0.5) < 1e-6) | (np.abs(np.abs(v - np.floor(v)) - 0.5) < 1e-6)
        assert tie.mean() < 1e-3
        assert np.array_equal(out["xy"][~tie], gen[~tie])


@pytest.mark.parametrize("nc", [8, 32])
def test_host_and_device_bit_identical(torch, nc):
    cams = rig(nc)
    eng = T.Engine(cams, 0)
    X = wide_points(300007, seed=11)
    for xyz_dt, tdt in ((np.float32, torch.float32), (np.float64, torch.float64)):
        Xd = torch.from_numpy(X.astype(xyz_dt)).cuda()
        for fl in (0, T.F32):
            for fmt, dt in PIX.items():
                tp = {"f32": torch.float32, "f64": torch.float64, "u16": torch.uint16}[fmt]
                host = eng.project_points(X.astype(xyz_dt), fl, pix_dtype=dt)
                dev = eng.project_points_device(Xd, fl, pix_dtype=tp)
                torch.cuda.synchronize()
                assert np.array_equal(dev["xy"].cpu().numpy(), host["xy"])
                assert np.array_equal(dev["mask"].cpu().numpy().view(np.uint32), host["mask"])


def test_stride_gap_untouched(torch):
    cams = rig(8)
    nc = len(cams)
    eng = T.Engine(cams, 0)
    n, pad = 10001, 37
    X = wide_points(n, seed=5)
    full = eng.project_points(X, 0)
    # device: rows cam_stride = n + pad apart, the gap filled with a canary
    canvas = torch.full((nc, n + pad, 2), 12345.0, dtype=torch.float32, device="cuda:0")
    out = {"xy": canvas[:, :n], "mask": torch.empty(n, dtype=torch.int32, device="cuda:0")}
    eng.project_points_device(torch.from_numpy(X).cuda(), 0, out=out)
    c = canvas.cpu().numpy()
    assert np.all(c[:, n:] == 12345.0)
    assert np.array_equal(c[:, :n], full["xy"])
    # host: the same through the C call
    h = np.full((nc, n + pad, 2), 12345.0, np.float32)
    mask = np.empty(n, np.uint32)
    st = T.lib().tri_project_points(eng._h, 0, None, C.c_void_p(X.ctypes.data), n, C.c_void_p(h.ctypes.data), n + pad,
                                    C.c_void_p(mask.ctypes.data))
    assert st == T.OK
    assert np.all(h[:, n:] == 12345.0) and np.array_equal(h[:, :n], full["xy"]) and np.array_equal(mask, full["mask"])


def test_odd_sizes_and_batch_offsets(torch):
    cams = rig(12)
    eng = T.Engine(cams, 0)
    X = wide_points(1000003, seed=9)  # spans several grid strides of the persistent kernel
    Xd = torch.from_numpy(X).cuda()
    for fl in (0, T.F32):
        for fmt, tp in (("f32", torch.float32), ("u16", torch.uint16), ("f64", torch.float64)):
            full = eng.project_points_device(Xd, fl, pix_dtype=tp)
            fx, fm = full["xy"].cpu().numpy(), full["mask"].cpu().numpy()
            for a, b in ((0, 1), (0, 31), (5, 38), (100, 611), (1001, 1514), (3, 1000003), (999490, 1000003)):
                part = eng.project_points_device(Xd[a:b], fl, pix_dtype=tp)  # odd sizes, bases one point off
                assert np.array_equal(part["xy"].cpu().numpy(), fx[:, a:b]), (a, b)
                assert np.array_equal(part["mask"].cpu().numpy(), fm[a:b]), (a, b)
    check_against_ref(cams, X[:200000], {"xy": fx[:, :200000], "mask": fm[:200000].view(np.uint32)}, "f64", T.F32)


def test_unaligned_bases(torch):
    cams = rig(8)
    nc = len(cams)
    eng = T.Engine(cams, 0)
    n = 4099
    X = wide_points(n, seed=13)
    for fl in (0, T.F32):
        for xdt in (torch.float32, torch.float64):
            Xbuf = torch.empty(3 * n + 1, dtype=xdt, device="cuda:0")
            Xbuf[1:] = torch.from_numpy(X).to(xdt).reshape(-1).cuda()
            Xv = Xbuf[1:].view(n, 3)  # one element off: only element-aligned
            ref = eng.project_points_device(torch.from_numpy(X).to(xdt).cuda(), fl)
            for tp in (torch.float32, torch.float64, torch.uint16):
                aligned = eng.project_points_device(Xv, fl, pix_dtype=tp)
                flat = torch.empty(2 * nc * n + 1, dtype=tp, device="cuda:0")
                xy = flat[1:].view(nc, n, 2)  # rows aligned only to the component: the scalar-store kernel
                assert xy.data_ptr() % (2 * xy.element_size()) != 0
                mflat = torch.empty(n + 1, dtype=torch.int32, device="cuda:0")
                out = eng.project_points_device(Xv, fl, out={"xy": xy, "mask": mflat[1:]})
                assert torch.equal(out["xy"], aligned["xy"]) and torch.equal(out["mask"], aligned["mask"])
                assert torch.equal(aligned["mask"], ref["mask"])


def test_argument_checks_and_launch_count(torch):
    cams = rig(4)
    eng = T.Engine(cams, 0)
    L, h = T.lib(), eng._h
    n = 100
    X = wide_points(n)
    X32 = X.astype(np.float32)
    xy = np.empty((4, n, 2), np.float32)
    m = np.empty(n, np.uint32)
    px, pm, p64, p32 = (C.c_void_p(a.ctypes.data) for a in (xy, m, X, X32))

    def host(fl=0, f32=None, f64=p64, nn=n, xyp=px, stride=n, mp=pm):
        return L.tri_project_points(h, fl, f32, f64, nn, xyp, stride, mp)

    l0 = eng.kernel_launches
    for fl in (T.ALLOW_TOO_FEW, T.RAY_REFERENCE_LM, T.RAY_CLOSED_FORM, T.RAY_ANALYTIC_LM, T.CLS_LAZY, 1 << 12, 1 << 30):
        assert host(fl) == T.ERR_ARG
    assert host(T.PIX_F64 | T.PIX_U16) == T.ERR_ARG
    assert host(f32=p32, f64=p64) == T.ERR_ARG
    assert host(f32=None, f64=None) == T.ERR_ARG
    assert host(xyp=None, mp=None) == T.ERR_ARG
    assert host(nn=-1) == T.ERR_ARG
    assert host(stride=n - 1) == T.ERR_DIM
    assert L.tri_project_points(None, 0, None, p64, n, px, n, pm) == T.ERR_ARG
    assert eng.kernel_launches == l0
    assert host(nn=0, f64=None, xyp=None, mp=None, stride=0) == T.OK  # empty: a no-op
    assert eng.kernel_launches == l0
    assert host() == T.OK and eng.kernel_launches == l0 + 1
    assert host(f32=p32, f64=None, xyp=None) == T.OK and eng.kernel_launches == l0 + 2  # masks only
    assert host(T.F32 | T.PIX_F64, xyp=C.c_void_p(np.empty((4, n, 2)).ctypes.data), mp=None) == T.OK
    assert eng.kernel_launches == l0 + 3
    # the device entry point: the same checks, one launch per call
    Xd = torch.from_numpy(X).cuda()
    xd = torch.empty((4, n, 2), dtype=torch.float32, device="cuda:0")
    md = torch.empty(n, dtype=torch.int32, device="cuda:0")
    dp = lambda t: C.c_void_p(t.data_ptr())
    assert L.tri_project_points_device(h, T.ALLOW_TOO_FEW, None, dp(Xd), n, dp(xd), n, dp(md), None) == T.ERR_ARG
    assert L.tri_project_points_device(h, T.PIX_F64 | T.PIX_U16, None, dp(Xd), n, dp(xd), n, dp(md), None) == T.ERR_ARG
    assert L.tri_project_points_device(h, 0, dp(Xd), dp(Xd), n, dp(xd), n, dp(md), None) == T.ERR_ARG
    assert L.tri_project_points_device(h, 0, None, None, n, dp(xd), n, dp(md), None) == T.ERR_ARG
    assert L.tri_project_points_device(h, 0, None, dp(Xd), n, None, n, None, None) == T.ERR_ARG
    assert L.tri_project_points_device(h, 0, None, dp(Xd), n, dp(xd), n - 1, dp(md), None) == T.ERR_DIM
    assert L.tri_project_points_device(h, 0, None, None, 0, None, 0, None, None) == T.OK
    assert eng.kernel_launches == l0 + 3
    assert L.tri_project_points_device(h, 0, None, dp(Xd), n, dp(xd), n, dp(md), None) == T.OK
    torch.cuda.synchronize()
    assert eng.kernel_launches == l0 + 4
    assert np.array_equal(xd.cpu().numpy(), eng.project_points(X)["xy"])
    # the torch wrapper refuses buffers the kernel would read or write past: it writes n_cams rows of n pixels
    for bad in (Xd.half(), Xd.to(torch.int32), Xd.bfloat16()):
        with pytest.raises(T.TriError) as e:
            eng.project_points_device(bad)
        assert e.value.status == T.ERR_ARG
    for o in ({"xy": torch.empty((3, n, 2), dtype=torch.float32, device="cuda:0")},
              {"xy": torch.empty((1, n, 2), dtype=torch.float32, device="cuda:0")},
              {"xy": torch.empty((4, n - 1, 2), dtype=torch.float32, device="cuda:0")},
              {"xy": torch.empty((4, n, 2), dtype=torch.int32, device="cuda:0")},
              {"mask": torch.empty(n - 1, dtype=torch.int32, device="cuda:0")},
              {"mask": torch.empty(n, dtype=torch.int64, device="cuda:0")},
              {"mask": torch.empty(2 * n, dtype=torch.int32, device="cuda:0")[::2]}):
        with pytest.raises(T.TriError) as e:
            eng.project_points_device(Xd, out=o)
        assert e.value.status == T.ERR_ARG
    assert eng.kernel_launches == l0 + 5  # the refused calls launch nothing (the 5th is the host check above)
    # TRI_PIX_U16 on a camera wider than 65535: its pixels could equal the marker
    big = T.Engine(cams[:1] + [T.Camera(9, 70000, 1080, 1081.0810546875, (6000.0, 0.0, 3000.0),
                                        S.look_at_quat((6000.0, 0.0, 3000.0), (0.0, 0.0, 1000.0)))], 0)
    u16 = np.empty((2, n, 2), np.uint16)
    assert L.tri_project_points(big._h, T.PIX_U16, None, p64, n, C.c_void_p(u16.ctypes.data), n, pm) == T.ERR_ARG
    assert L.tri_project_points(big._h, 0, None, p64, n, px, n, pm) == T.OK


def test_cpp_driver_round_trip(torch):
    host = os.path.join(ROOT, "3d-reconstruction-triangulation_b200", "host")
    subprocess.check_call(["make", "-s", "-C", host])
    nc, n = 8, 2000
    out = subprocess.check_output([os.path.join(host, "host_project_selftest"), str(nc), str(n)], text=True).splitlines()
    pts = [l.split() for l in out if l.startswith("point ")]
    X = np.array([[float(v) for v in p[2:5]] for p in pts])
    mask = np.array([int(p[5]) for p in pts], np.uint32)
    pix = np.array([[float(v) for v in l.split()[3:5]] for l in out if l.startswith("pix ")]).reshape(len(X), nc, 2)
    assert len(X) == n + 2
    cams = rig(nc)
    eng = T.Engine(cams, 0)
    ref = eng.project_points(X, 0, pix_dtype=np.float64)
    _, _, vis, rmask, dist, _ = ref_project(cams, X)
    thin = (dist < 1e-6).any(axis=0)
    assert np.array_equal(mask[~thin], ref["mask"][~thin]) and np.array_equal(mask[~thin], rmask[~thin])
    both = bits(mask, nc) & bits(ref["mask"], nc)
    got = pix.transpose(1, 0, 2)
    assert np.abs(got[both] - ref["xy"][both]).max() < 1e-9
    assert np.all(got[~bits(mask, nc)] == -1.0)
    assert mask[n] & 1 == 0 and mask[n + 1] == 0  # behind camera 0; above every frustum
    rt = [l.split() for l in out if l.startswith("roundtrip ")][0]
    assert int(rt[1]) == int((np.array([bin(int(v)).count("1") for v in mask]) >= 2).sum()) and float(rt[2]) < 1e-9
    assert [l for l in out if l.startswith("empty ")] == ["empty %d 0" % nc]
