"""A frame gets bit-identical outputs whichever batch kernel runs it.

The same frames go through each mode three ways: aligned rows with the lean outputs (the streaming tile or the
generic two-frame kernel), aligned rows with the wide outputs (the tile's WIDE instantiation, or the generic
kernel when the tile cannot give the error), and rows and outputs offset by one frame, so nothing is vector-aligned
and the scalar or tail kernels take the frames.  Every output two runs share must match bit for bit.  The engine's
launch counter shows which shape ran: the aligned runs take a vector or tile kernel plus a tail kernel, the offset
run one kernel for all its frames (where a mode has only the one-frame-per-thread generic kernel, every run takes
that one kernel)."""
import numpy as np
import pytest

import tri_b200 as T
from tri_b200 import synthetic as S

pytestmark = pytest.mark.gpu

N = 3 * 512 + 77  # whole tiles of both frame-per-thread shapes plus a tail
MODES = {  # name: (robust, mode, flags, wide outputs besides xyz_f32 / mask)
    "matrix_f64": (False, T.MATRIX, 0, ("xyz_f64", "err", "iters")),
    "matrix_f32": (False, T.MATRIX, T.F32, ("xyz_f64", "err", "iters")),
    "ray_closed_f64": (False, T.RAY, T.RAY_CLOSED_FORM, ("xyz_f64", "err", "iters")),
    "ray_closed_f32": (False, T.RAY, T.RAY_CLOSED_FORM | T.F32, ("xyz_f64", "err", "iters")),
    "ray_lm_f64": (False, T.RAY, T.RAY_ANALYTIC_LM, ("xyz_f64", "err", "iters")),
    "robust_f64": (True, None, 0, ("xyz_f64", "err")),
    "robust_f32": (True, None, T.F32, ("xyz_f64", "err")),
}
DTYPES = {"float2": "float32", "double2": "float64", "ushort2": "uint16"}


@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available()
    return torch


def _rig(nc):
    return S.ring_rig(nc) if nc <= 8 else S.ring_rig(nc, rings=((6000.0, 3000.0), (9000.0, 5000.0)))


def _frames(torch, cams, dtype):
    xy = S.generate_frames(cams, N + 1, device="cuda:0", p_missing=0.35, p_outlier=0.05)
    if dtype == "uint16":  # integer pixels; (-1, -1) -> the (0xFFFF, 0xFFFF) marker
        return xy.to(torch.int32).bitwise_and(0xFFFF).to(torch.uint16)
    return xy.to(getattr(torch, dtype))


def _empty(torch, key, n, off):
    """An output buffer for n frames; off = 1 starts it one element in, so it is not vector-aligned."""
    shape, dt = {"xyz_f32": ((n + off, 3), torch.float32), "xyz_f64": ((n + off, 3), torch.float64),
                 "mask": ((n + off,), torch.int32), "err": ((n + off,), torch.float64),
                 "iters": ((n + off,), torch.int32)}[key]
    return torch.full(shape, -7, dtype=dt, device="cuda:0")[off:]


def _run(torch, eng, spec, xy, keys, off):
    """-> (outputs, number of kernel launches)"""
    robust, mode, flags, _ = spec
    out = {k: _empty(torch, k, xy.shape[1], off) for k in keys}
    before = eng.kernel_launches
    if robust:
        eng.triangulate_points_robust_device(xy, 2.0, flags | T.ALLOW_TOO_FEW, out=out)
    else:
        eng.triangulate_points_device(mode, xy, flags | T.ALLOW_TOO_FEW, out=out)
    eng.device_status()
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in out.items()}, eng.kernel_launches - before


def _one_kernel(nc, mode, pix):
    """The modes whose every frame takes one kernel even on aligned rows: double2 pixels on a one-frame-per-thread
    generic kernel, and the robust solve wherever its tile does not apply (double2 pixels, more than 8 cameras)."""
    if mode.startswith("robust"):
        return pix == "double2" or nc > 8
    return pix == "double2" and mode in ("matrix_f64", "ray_closed_f64", "ray_lm_f64")


@pytest.mark.parametrize("pix", list(DTYPES))
@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("nc", [8, 12, 32])
def test_kernel_paths_bit_identical(torch, nc, mode, pix):
    spec = MODES[mode]
    cams = _rig(nc)
    eng = T.Engine(cams, 0)
    xy = _frames(torch, cams, DTYPES[pix])
    lean, wide = ("xyz_f32", "mask"), ("xyz_f32", "mask") + spec[3]
    a, na = _run(torch, eng, spec, xy[:, :N], lean, 0)         # aligned rows, lean outputs
    b, nb = _run(torch, eng, spec, xy[:, :N], wide, 0)         # aligned rows, wide outputs
    c, n_c = _run(torch, eng, spec, xy[:, 1:N + 1], wide, 1)   # rows and outputs one frame in: scalar / tail kernels
    assert n_c == 1
    if _one_kernel(nc, mode, pix):
        assert na == nb == 1
    else:
        assert na >= 2 and nb >= 2
    assert (a["mask"] != 0).any()
    for k in lean:
        assert np.array_equal(a[k], b[k]), (k, "lean vs wide")
    for k in wide:
        eq = np.array_equal(b[k][1:], c[k][:-1], equal_nan=k == "err")
        assert eq, (k, "aligned vs offset")
