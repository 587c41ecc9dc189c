"""ctypes binding of oracle/liboracle_robust.so -- TEST INFRASTRUCTURE ONLY (see tri_oracle.h): the CUDA engine's
outlier-robust batch (tri_triangulate_points_robust) restated serially in FP64 (tri_oracle_robust.c, linked with the
plain oracle tri_oracle.c whose DLT it uses).  Cameras are oracle_py.make_camera structures."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

import oracle_py as O

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "liboracle_robust.so")
SOURCES = ("tri_oracle_robust.c", "tri_oracle.c")


def build():
    """Compile liboracle_robust.so with the plain oracle's flags (oracle/Makefile: no FMA contraction)."""
    subprocess.check_call(["gcc", "-O2", "-fPIC", "-fopenmp", "-ffp-contract=off", "-Wall", "-Wextra", "-std=c11", "-shared", "-o", LIB]
                          + [os.path.join(HERE, s) for s in SOURCES] + ["-lm"])


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB):
            build()
        _lib = C.CDLL(LIB)
    return _lib


def triangulate_points_robust(cams, xy, max_reproj_px, allow_too_few=False):
    """xy: [n_point_cams][n_frames][2] float64 | float32 ((-1,-1) missing) or uint16 ((0xFFFF, 0xFFFF) missing).
    -> dict(xyz, err, mask, margin, status, first_bad_frame)."""
    arr = O.camera_array(cams)
    xy = np.asarray(xy)
    if xy.dtype == np.uint16:
        miss = (xy == 0xFFFF).all(axis=2)
        xy = xy.astype(np.float64)
        xy[miss] = -1.0
    xy = np.ascontiguousarray(xy, np.float64)
    npc, nf = xy.shape[0], xy.shape[1]
    out, err, mask, margin = np.zeros((nf, 3)), np.zeros(nf), np.zeros(nf, np.uint32), np.zeros(nf)
    bad = C.c_int64(-1)
    st = lib().orc_triangulate_points_robust(arr, len(cams), npc, O._p(xy), C.c_int64(nf), C.c_double(max_reproj_px),
                                             int(allow_too_few), O._p(out), O._p(err), O._p(mask, C.c_uint32), O._p(margin),
                                             C.byref(bad))
    return dict(xyz=out, err=err, mask=mask, margin=margin, status=st, first_bad_frame=bad.value)
