"""tri_b200 -- Python binding (ctypes) of libtri_b200.so, the B200-native batched triangulation engine.

The product is the CUDA library behind the C ABI of ``include/tri_b200.h`` and the C++ host mirror of
the reference's interface under ``host/``.  This module is the thin harness the tests and ``bench.py``
drive it with: it loads the in-tree ``libtri_b200.so`` (and fails loudly if it is missing -- there is
no CPU path), builds the camera constants the way ``tdr::Camera`` does (src/Camera.h:78-187 of the
reference) and hands raw device / host pointers to the C entry points.

The directory name is not an importable identifier; import it through the root-level ``tri_b200``
shim (``import tri_b200``).
"""
from __future__ import annotations

import ctypes as C
import math
import os
import re
from dataclasses import dataclass, field

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libtri_b200.so")

MATRIX, RAY = 0, 1
OK, ERR_DIM, ERR_TOO_FEW, ERR_ARG, ERR_CUDA, ERR_NO_DEVICE, ERR_CAPACITY = range(7)
F32 = 1 << 0
ALLOW_TOO_FEW = 1 << 1
RAY_REFERENCE_LM = 1 << 2
RAY_CLOSED_FORM = 1 << 3
PIX_F64 = 1 << 4
PIX_U16 = 1 << 5
RAY_ANALYTIC_LM = 1 << 6
CLS_LAZY = 1 << 7
MAX_CAMS = 32

# the runtime_error texts of the reference, re-raised by the adapters
MSG_DIM = "Every camera should have the same number of points"  # MatrixTriangulator.cpp:74-75
MSG_TOO_FEW = {MATRIX: "Too few rays are found",  # MatrixTriangulator.cpp:93
               RAY: "Too few detections are found"}  # RayTriangulator.cpp:73


class TriError(RuntimeError):
    def __init__(self, status, msg):
        super().__init__(msg)
        self.status = status


class _Camera(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("fovy_deg", C.c_double), ("P", C.c_double * 12),
                ("position", C.c_double * 3), ("quat", C.c_double * 4)]


class _BatchOut(C.Structure):
    _fields_ = [("xyz_f32", C.c_void_p), ("xyz_f64", C.c_void_p), ("mask", C.c_void_p), ("err", C.c_void_p),
                ("iters", C.c_void_p)]


class ClassifyStats(C.Structure):
    _fields_ = [(n, C.c_int64) for n in ("nodes", "solves", "leaves", "lm_iters", "phase1", "phase2", "ties",
                                         "max_frontier", "enumerate_us", "link_us")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


EXPORTS = ["tri_version", "tri_last_error", "tri_device_count", "tri_create", "tri_destroy", "tri_engine_device",
           "tri_engine_cameras", "tri_kernel_launches", "tri_triangulate_points", "tri_triangulate_points_multi",
           "tri_triangulate_points_device", "tri_triangulate_points_robust", "tri_triangulate_points_robust_device",
           "tri_project_points", "tri_project_points_device", "tri_device_status", "tri_enable_peer_access",
           "tri_ipc_export", "tri_ipc_open", "tri_ipc_close", "tri_copy_device", "tri_triangulate_subsets", "tri_dist_from_ray",
           "tri_classify", "tri_classify_state_bytes", "tri_classify_begin", "tri_classify_finish", "tri_classify_multi", "tri_classify_sequences", "tri_host_alloc",
           "tri_host_free", "tri_device_alloc", "tri_device_free", "tri_copy_to_device", "tri_copy_to_host"]

_lib = None


def lib():
    """The loaded C ABI.  Raises if the CUDA library has not been built: nothing here computes on the CPU."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError("libtri_b200.so is missing (%s): build it with `python -c 'import __graft_entry__ as g; "
                              "g.build()'` or `make -C 3d-reconstruction-triangulation_b200/csrc`; there is no CPU "
                              "fallback" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        L.tri_last_error.restype = C.c_char_p
        L.tri_kernel_launches.restype = C.c_int64
        L.tri_create.argtypes = [C.c_int, C.POINTER(_Camera), C.c_int, C.POINTER(C.c_void_p)]
        L.tri_destroy.argtypes = [C.c_void_p]
        L.tri_destroy.restype = None
        L.tri_kernel_launches.argtypes = [C.c_void_p]
        L.tri_engine_device.argtypes = [C.c_void_p]
        L.tri_engine_cameras.argtypes = [C.c_void_p]
        L.tri_triangulate_points.argtypes = [C.c_void_p, C.c_int, C.c_uint, C.c_void_p, C.c_int, C.c_int64, C.c_int64,
                                             C.POINTER(_BatchOut), C.POINTER(C.c_int64)]
        L.tri_triangulate_points_multi.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_uint, C.c_void_p, C.c_int, C.c_int64,
                                                   C.c_int64, C.POINTER(_BatchOut), C.POINTER(C.c_int64)]
        L.tri_triangulate_points_device.argtypes = [C.c_void_p, C.c_int, C.c_uint, C.c_void_p, C.c_int, C.c_int64,
                                                    C.c_int64, C.POINTER(_BatchOut), C.c_void_p]
        L.tri_triangulate_points_robust.argtypes = [C.c_void_p, C.c_uint, C.c_double, C.c_void_p, C.c_int, C.c_int64, C.c_int64,
                                                    C.POINTER(_BatchOut), C.POINTER(C.c_int64)]
        L.tri_triangulate_points_robust_device.argtypes = [C.c_void_p, C.c_uint, C.c_double, C.c_void_p, C.c_int, C.c_int64,
                                                           C.c_int64, C.POINTER(_BatchOut), C.c_void_p]
        L.tri_project_points.argtypes = [C.c_void_p, C.c_uint, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]
        L.tri_project_points_device.argtypes = [C.c_void_p, C.c_uint, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64,
                                                C.c_void_p, C.c_void_p]
        L.tri_enable_peer_access.argtypes = [C.c_void_p, C.c_int]
        L.tri_ipc_export.argtypes = [C.c_void_p, C.c_void_p, C.c_char_p]
        L.tri_ipc_open.argtypes = [C.c_void_p, C.c_char_p, C.POINTER(C.c_void_p)]
        L.tri_ipc_close.argtypes = [C.c_void_p, C.c_void_p]
        L.tri_copy_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]
        L.tri_device_alloc.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.c_uint64]
        L.tri_device_free.argtypes = [C.c_void_p, C.c_void_p]
        L.tri_device_status.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_int64)]
        L.tri_triangulate_subsets.argtypes = [C.c_void_p, C.c_int, C.c_uint, C.c_int64, C.c_void_p, C.c_void_p,
                                              C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.tri_dist_from_ray.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.tri_classify.argtypes = [C.c_void_p, C.c_int, C.c_uint, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.POINTER(ClassifyStats)]
        L.tri_classify_sequences.argtypes = [C.c_void_p, C.c_int, C.c_uint, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                             C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(ClassifyStats)]
        L.tri_classify_begin.argtypes = [C.c_void_p, C.c_int, C.c_uint, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
        L.tri_classify_finish.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.POINTER(ClassifyStats)]
        L.tri_classify_multi.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_uint, C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                                         C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(ClassifyStats)]
        L.tri_host_alloc.argtypes = [C.POINTER(C.c_void_p), C.c_uint64]
        L.tri_host_free.argtypes = [C.c_void_p]
        _lib = L
    return _lib


def _check(st, mode=MATRIX):
    if st == OK:
        return
    msg = lib().tri_last_error().decode()
    if st == ERR_DIM and not msg:
        msg = MSG_DIM
    raise TriError(st, msg)


# ------------------------------------------------------------------------------------------------
# tdr::Camera (src/Camera.h) -- host-side constants, same arithmetic as the reference
# ------------------------------------------------------------------------------------------------
RAD_TO_DEG = 57.29577951308232087679  # Camera.h:23-26
DEG_TO_RAD = 0.01745329251994329576


def _inv3(S):
    """cv::Mat::inv() on a 3x3 CV_64F (closed-form branch of cv::invert, DECOMP_LU)."""
    d = (S[0][0] * (S[1][1] * S[2][2] - S[1][2] * S[2][1]) - S[0][1] * (S[1][0] * S[2][2] - S[1][2] * S[2][0])
         + S[0][2] * (S[1][0] * S[2][1] - S[1][1] * S[2][0]))
    if d == 0.0:
        return [[0.0] * 3 for _ in range(3)]
    d = 1.0 / d
    return [[(S[1][1] * S[2][2] - S[1][2] * S[2][1]) * d, (S[0][2] * S[2][1] - S[0][1] * S[2][2]) * d,
             (S[0][1] * S[1][2] - S[0][2] * S[1][1]) * d],
            [(S[1][2] * S[2][0] - S[1][0] * S[2][2]) * d, (S[0][0] * S[2][2] - S[0][2] * S[2][0]) * d,
             (S[0][2] * S[1][0] - S[0][0] * S[1][2]) * d],
            [(S[1][0] * S[2][1] - S[1][1] * S[2][0]) * d, (S[0][1] * S[2][0] - S[0][0] * S[2][1]) * d,
             (S[0][0] * S[1][1] - S[0][1] * S[1][0]) * d]]


@dataclass
class Camera:
    """createCamera (src/utils.cpp:94-107) + Camera::compCamParams (src/Camera.h:177-187)."""
    cam_id: int
    width: int
    height: int
    focal: float
    position: tuple  # "tvec": world position (utils.cpp:101)
    quat: tuple  # "rquat": (w,i,j,k) as stored, never normalised (utils.cpp:103)
    cx: int = 0
    cy: int = 0
    fx: float = 0.0
    fy: float = 0.0
    fovx: float = 0.0
    fovy: float = 0.0
    K: np.ndarray = field(default=None, repr=False)
    E: np.ndarray = field(default=None, repr=False)
    P: np.ndarray = field(default=None, repr=False)

    def __post_init__(self):
        w, h = int(self.width), int(self.height)
        if w == 0 or h == 0:
            raise RuntimeError("Camera: image size is not set")  # Camera.h:79-80
        self.cx = int(math.floor(w / 2.0 + 0.5))  # Camera.h:81-82: C round(), half away from zero (Python's round() is half-to-even)
        self.cy = int(math.floor(h / 2.0 + 0.5))
        fx = float(self.focal)
        if fx == 0:
            raise RuntimeError("Camera: focal length is not set")  # Camera.h:90
        self.fovx = 2 * math.atan(w / (2 * fx)) * 57.2958  # Camera.h:91 (truncated constant)
        self.fovy = 2.0 * math.atan(math.tan(self.fovx * 0.5 * DEG_TO_RAD) / (float(w) / float(h))) * RAD_TO_DEG
        self.fx = (w / 2.0) / math.tan((self.fovx / 2.0) * DEG_TO_RAD)  # Camera.h:114-115
        self.fy = (h / 2.0) / math.tan((self.fovy / 2.0) * DEG_TO_RAD)
        a, b, c, d = (float(v) for v in self.quat)  # Camera.h:274-287, raw quaternion
        R0 = [[1 - 2 * (c * c + d * d), 2 * (b * c - a * d), 2 * (b * d + a * c)],
              [2 * (b * c + a * d), 1 - 2 * (b * b + d * d), 2 * (c * d - a * b)],
              [2 * (b * d - a * c), 2 * (c * d + a * b), 1 - 2 * (b * b + c * c)]]
        R = _inv3(R0)  # Camera.h:134 (inverse, not transpose)
        p = [float(v) for v in self.position]
        cam_pos = [-(R[i][0] * p[0] + R[i][1] * p[1] + R[i][2] * p[2]) for i in range(3)]  # Camera.h:167-170
        if self.fx == 0 or self.fy == 0 or self.cx == 0 or self.cy == 0:
            raise RuntimeError("Camera: intrinsics are not set")  # Camera.h:124
        K = [[self.fx, 0.0, float(self.cx)], [0.0, self.fy, float(self.cy)], [0.0, 0.0, 1.0]]
        E = [[R[i][0], R[i][1], R[i][2], cam_pos[i]] for i in range(3)]
        P = [[0.0] * 4 for _ in range(3)]
        for i in range(3):
            for j in range(4):
                s = 0.0
                for k in range(3):
                    s += K[i][k] * E[k][j]
                P[i][j] = s
        self.K, self.E, self.P = np.array(K), np.array(E), np.array(P)

    def as_struct(self):
        c = _Camera()
        c.width, c.height, c.fovy_deg = int(self.width), int(self.height), float(self.fovy)
        c.P[:] = [float(v) for v in self.P.reshape(-1)]
        c.position[:] = [float(v) for v in self.position]
        c.quat[:] = [float(v) for v in self.quat]
        return c


def _two_ints(text):
    """`std::stringstream(text) >> a >> b` for ints (utils.cpp:64-71): a failed extraction leaves 0."""
    vals, pos = [0, 0], 0
    for k in range(2):
        m = re.match(r"\s*([+-]?\d+)", text[pos:])
        if not m:
            break
        vals[k] = int(m.group(1))
        pos += m.end()
    return vals


def load_cameras_xml(path):
    """loadCamerasXML (src/utils.cpp:46-92): every <Camera> with a <ControlFrame>, in document order."""
    txt = open(path).read()
    cams = []
    for m in re.finditer(r"<Camera\b([^>]*)>(.*?)</Camera>", txt, re.S):
        cf = re.search(r"<ControlFrame\b([^>]*)/>", m.group(2))
        if not cf:
            continue
        at = dict(re.findall(r'(\w+)="([^"]*)"', cf.group(1)))
        dev = int(re.search(r'DEVICEID="(-?\d+)"', m.group(1)).group(1))
        w, h = (2 * v for v in _two_ints(at["PRINCIPAL_POINT"]))
        cams.append(Camera(dev, w, h, float(at["FOCAL_LENGTH"]), tuple(float(v) for v in at["POSITION"].split()),
                           tuple(float(v) for v in at["ORIENTATION"].split())))
    if not cams:
        raise RuntimeError("no cameras found in " + path)
    return cams


# ------------------------------------------------------------------------------------------------
# Engine
# ------------------------------------------------------------------------------------------------
def _np_ptr(a):
    return C.c_void_p(a.ctypes.data) if a is not None else None


_PIX_DTYPES = {np.dtype(np.float32): 0, np.dtype(np.float64): PIX_F64, np.dtype(np.uint16): PIX_U16}


class Engine:
    """One GPU + one camera rig (`new MatrixTriangulator(cameras)` / `new RayTriangulator(cameras)`)."""

    def __init__(self, cameras, device=0):
        self.cameras = list(cameras)
        arr = (_Camera * len(self.cameras))(*[c.as_struct() for c in self.cameras])
        h = C.c_void_p()
        _check(lib().tri_create(len(self.cameras), arr, int(device), C.byref(h)))
        self._h = h
        self.device = int(device)

    def close(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.tri_destroy(self._h)
        self._h = None

    __del__ = close

    @property
    def kernel_launches(self):
        return int(lib().tri_kernel_launches(self._h))

    # ---- device-resident batch (torch tensors on this engine's GPU), asynchronous on the current stream ----
    def triangulate_points_device(self, mode, xy, flags=0, out=None, want=("xyz_f32",), n_frames=None):
        """xy: torch tensor [n_point_cams, n_frames, 2] (float32 | float64 | uint16) on cuda:<device>.
        Returns a dict of torch tensors.  Call device_status() to collect the too-few-views latch."""
        import torch
        assert xy.is_cuda and xy.dim() == 3 and xy.shape[2] == 2 and xy.stride(2) == 1 and xy.stride(1) == 2
        fmt = {torch.float32: 0, torch.float64: PIX_F64, torch.uint16: PIX_U16}[xy.dtype]
        npc, nf = xy.shape[0], xy.shape[1] if n_frames is None else n_frames
        stride = xy.stride(0) // 2 if npc > 1 else nf
        if out is None:
            out = {}
            dev = xy.device
            for k in want:
                if k == "xyz_f32":
                    out[k] = torch.empty((nf, 3), dtype=torch.float32, device=dev)
                elif k == "xyz_f64":
                    out[k] = torch.empty((nf, 3), dtype=torch.float64, device=dev)
                elif k == "mask":
                    out[k] = torch.empty((nf,), dtype=torch.int32, device=dev)
                elif k == "err":
                    out[k] = torch.empty((nf,), dtype=torch.float64, device=dev)
                elif k == "iters":
                    out[k] = torch.empty((nf,), dtype=torch.int32, device=dev)
        bo = _BatchOut(*[out[k].data_ptr() if k in out else None for k in ("xyz_f32", "xyz_f64", "mask", "err", "iters")])
        stream = torch.cuda.current_stream(xy.device).cuda_stream
        _check(lib().tri_triangulate_points_device(self._h, mode, flags | fmt, C.c_void_p(xy.data_ptr()), npc, nf, stride,
                                                   C.byref(bo), C.c_void_p(stream)), mode)
        return out

    def enable_peer_access(self, peer_device):
        """Let this engine's kernels store straight into `peer_device`'s memory (fused gather over NVLink)."""
        _check(lib().tri_enable_peer_access(self._h, int(peer_device)))

    # ---- raw device buffers + CUDA IPC (fused gather into another rank's result array) ----
    def device_alloc(self, nbytes):
        p = C.c_void_p()
        _check(lib().tri_device_alloc(self._h, C.byref(p), int(nbytes)))
        return p.value

    def device_free(self, ptr):
        _check(lib().tri_device_free(self._h, C.c_void_p(ptr)))

    def ipc_export(self, ptr):
        buf = C.create_string_buffer(64)
        _check(lib().tri_ipc_export(self._h, C.c_void_p(ptr), buf))
        return buf.raw

    def ipc_open(self, handle):
        p = C.c_void_p()
        _check(lib().tri_ipc_open(self._h, handle, C.byref(p)))
        return p.value

    def ipc_close(self, ptr):
        _check(lib().tri_ipc_close(self._h, C.c_void_p(ptr)))

    def copy_device(self, dst_ptr, src_ptr, nbytes):
        _check(lib().tri_copy_device(self._h, C.c_void_p(dst_ptr), C.c_void_p(src_ptr), int(nbytes)))

    def triangulate_points_device_raw(self, mode, flags, xy_ptr, npc, nf, stride, xyz_f32_ptr, stream=None):
        """Device entry point with raw addresses (the output may be a peer / IPC pointer)."""
        bo = _BatchOut(xyz_f32_ptr, None, None, None, None)
        _check(lib().tri_triangulate_points_device(self._h, mode, flags, C.c_void_p(xy_ptr), npc, nf, stride, C.byref(bo),
                                                   C.c_void_p(stream)), mode)

    def device_status(self):
        """Synchronise the current stream; raises TriError(ERR_TOO_FEW) if a frame had < 2 views."""
        import torch
        stream = torch.cuda.current_stream(torch.device("cuda", self.device)).cuda_stream
        bad = C.c_int64(-1)
        st = lib().tri_device_status(self._h, C.c_void_p(stream), C.byref(bad))
        return st, bad.value

    # ---- host-buffer batch: Triangulator::triangulatePoints ----
    def triangulate_points(self, mode, xy, flags=0, want=("xyz_f64",), out=None):
        """xy: numpy [n_point_cams, n_frames, 2] float32 | float64 | uint16 (host memory, ideally pinned).
        Raises TriError with the reference's text where the reference throws."""
        xy = np.asarray(xy)
        if xy.ndim != 3 or xy.shape[2] != 2:
            raise TriError(ERR_DIM, MSG_DIM)
        if not xy.flags.c_contiguous:
            xy = np.ascontiguousarray(xy)
        fmt = _PIX_DTYPES[xy.dtype]
        npc, nf = xy.shape[0], xy.shape[1]
        if out is None:
            out = {}
            for k in want:
                out[k] = np.empty({"xyz_f32": (nf, 3), "xyz_f64": (nf, 3)}.get(k, (nf,)),
                                  {"xyz_f32": np.float32, "xyz_f64": np.float64, "mask": np.uint32, "err": np.float64,
                                   "iters": np.int32}[k])
        bo = _BatchOut(*[out[k].ctypes.data if k in out else None for k in ("xyz_f32", "xyz_f64", "mask", "err", "iters")])
        bad = C.c_int64(-1)
        st = lib().tri_triangulate_points(self._h, mode, flags | fmt, _np_ptr(xy), npc, nf, nf, C.byref(bo), C.byref(bad))
        out["first_bad_frame"] = bad.value
        _check(st, mode)
        return out

    def triangulate_points_raw(self, mode, flags, xy_ptr, npc, nf, stride, xyz_f32_ptr=None, xyz_f64_ptr=None,
                               mask_ptr=None, err_ptr=None, iters_ptr=None):
        """Host-buffer entry with raw addresses (pinned torch tensors in bench.py)."""
        bo = _BatchOut(xyz_f32_ptr, xyz_f64_ptr, mask_ptr, err_ptr, iters_ptr)
        bad = C.c_int64(-1)
        st = lib().tri_triangulate_points(self._h, mode, flags, C.c_void_p(xy_ptr), npc, nf, stride, C.byref(bo), C.byref(bad))
        _check(st, mode)
        return bad.value

    # ---- outlier-robust matrix-mode batch (two-view consensus, inlier refit; an extension of the reference) ----
    def triangulate_points_robust(self, xy, max_reproj_px, flags=0, want=("xyz_f64", "mask", "err")):
        """xy: numpy [n_point_cams, n_frames, 2] float32 | float64 | uint16 (host memory).  mask = the inlier set,
        err = RMS reprojection error in pixels over it (NaN where no two views agree within max_reproj_px)."""
        xy = np.asarray(xy)
        if xy.ndim != 3 or xy.shape[2] != 2:
            raise TriError(ERR_DIM, MSG_DIM)
        xy = np.ascontiguousarray(xy)
        npc, nf = xy.shape[0], xy.shape[1]
        out = {k: np.empty({"xyz_f32": (nf, 3), "xyz_f64": (nf, 3)}.get(k, (nf,)),
                           {"xyz_f32": np.float32, "xyz_f64": np.float64, "mask": np.uint32, "err": np.float64}[k]) for k in want}
        bo = _BatchOut(*[out[k].ctypes.data if k in out else None for k in ("xyz_f32", "xyz_f64", "mask", "err", "iters")])
        bad = C.c_int64(-1)
        st = lib().tri_triangulate_points_robust(self._h, flags | _PIX_DTYPES[xy.dtype], float(max_reproj_px), _np_ptr(xy), npc, nf,
                                                 nf, C.byref(bo), C.byref(bad))
        out["first_bad_frame"] = bad.value
        _check(st)
        return out

    def triangulate_points_robust_device(self, xy, max_reproj_px, flags=0, out=None, want=("xyz_f64", "mask", "err")):
        """xy: torch tensor [n_point_cams, n_frames, 2] on cuda:<device>, asynchronous on the current stream; the
        too-few latch is collected by device_status().  Outputs as triangulate_points_robust, as torch tensors."""
        import torch
        assert xy.is_cuda and xy.dim() == 3 and xy.shape[2] == 2 and xy.stride(2) == 1 and xy.stride(1) == 2
        fmt = {torch.float32: 0, torch.float64: PIX_F64, torch.uint16: PIX_U16}[xy.dtype]
        npc, nf = xy.shape[0], xy.shape[1]
        stride = xy.stride(0) // 2 if npc > 1 else nf
        if out is None:
            out = {k: torch.empty({"xyz_f32": (nf, 3), "xyz_f64": (nf, 3)}.get(k, (nf,)),
                                  dtype={"xyz_f32": torch.float32, "xyz_f64": torch.float64, "mask": torch.int32,
                                         "err": torch.float64}[k], device=xy.device) for k in want}
        bo = _BatchOut(*[out[k].data_ptr() if k in out else None for k in ("xyz_f32", "xyz_f64", "mask", "err", "iters")])
        stream = torch.cuda.current_stream(xy.device).cuda_stream
        _check(lib().tri_triangulate_points_robust_device(self._h, flags | fmt, float(max_reproj_px), C.c_void_p(xy.data_ptr()), npc, nf,
                                                          stride, C.byref(bo), C.c_void_p(stream)))
        return out

    # ---- forward projection: points -> per-camera pixels in the batch input layout (an extension of the reference) ----
    def project_points(self, xyz, flags=0, pix_dtype=np.float32):
        """xyz: numpy [n, 3] float32 | float64 (host memory; the dtype picks the input).  FP64 unless flags has F32.
        -> {"xy": [n_cams, n, 2] pix_dtype (float32 | float64 | uint16), "mask": uint32 [n] (bit c = camera c sees the
        point)}; views a camera does not see hold the missing marker ((-1,-1), 0xFFFF pairs for uint16)."""
        xyz = np.ascontiguousarray(xyz)
        if xyz.ndim != 2 or xyz.shape[1] != 3 or xyz.dtype not in (np.float32, np.float64):
            raise TriError(ERR_ARG, "xyz must be a float32 or float64 array of shape [n, 3]")
        n = xyz.shape[0]
        fmt = _PIX_DTYPES[np.dtype(pix_dtype)]
        out = {"xy": np.empty((len(self.cameras), n, 2), pix_dtype), "mask": np.empty(n, np.uint32)}
        f32 = xyz.dtype == np.float32
        _check(lib().tri_project_points(self._h, flags | fmt, _np_ptr(xyz) if f32 else None, None if f32 else _np_ptr(xyz), n,
                                        _np_ptr(out["xy"]), n, _np_ptr(out["mask"])))
        return out

    def project_points_device(self, xyz, flags=0, pix_dtype=None, out=None, want=("xy", "mask")):
        """xyz: torch tensor [n, 3] float32 | float64 on cuda:<device>, rows packed (stride (3, 1)); asynchronous on the
        current stream.  out: optional dict with "xy" [n_cams, n, 2] (pairs packed, any camera stride >= n) and / or
        "mask" int32 [n] tensors, written in place.  Returns the dict (torch tensors)."""
        import torch
        pix_dtype = pix_dtype or torch.float32
        nc = len(self.cameras)
        dev = torch.device("cuda", self.device)

        def need(ok, what):
            if not ok:
                raise TriError(ERR_ARG, "project_points_device: " + what)

        # the kernel reads 12 or 24 B per point and writes all n_cams rows: every buffer is checked against that
        need(xyz.is_cuda and xyz.device == dev, "xyz must be on the engine's GPU")
        need(xyz.dtype in (torch.float32, torch.float64), "xyz must be float32 or float64")
        need(xyz.dim() == 2 and xyz.shape[1] == 3 and (xyz.shape[0] <= 1 or xyz.stride() == (3, 1)), "xyz must be packed [n, 3]")
        n = xyz.shape[0]
        if out is None:
            out = {}
            if "xy" in want:
                out["xy"] = torch.empty((nc, n, 2), dtype=pix_dtype, device=dev)
            if "mask" in want:
                out["mask"] = torch.empty((n,), dtype=torch.int32, device=dev)
        xy, mask = out.get("xy"), out.get("mask")
        stride = n
        fmt = 0
        if xy is not None:
            need(xy.is_cuda and xy.device == dev, "out['xy'] must be on the engine's GPU")
            need(xy.dtype in (torch.float32, torch.float64, torch.uint16), "out['xy'] must be float32, float64 or uint16")
            need(xy.dim() == 3 and tuple(xy.shape) == (nc, n, 2), "out['xy'] must be [n_cams, n, 2]")
            need(n == 0 or (xy.stride(2) == 1 and xy.stride(1) == 2), "out['xy'] must hold packed pixel pairs")
            need(nc == 1 or (xy.stride(0) % 2 == 0 and xy.stride(0) // 2 >= n), "out['xy'] camera rows must not overlap")
            fmt = {torch.float32: 0, torch.float64: PIX_F64, torch.uint16: PIX_U16}[xy.dtype]
            stride = xy.stride(0) // 2 if nc > 1 else n
        if mask is not None:
            need(mask.is_cuda and mask.device == dev, "out['mask'] must be on the engine's GPU")
            need(mask.dtype in (torch.int32, torch.uint32) and mask.dim() == 1 and mask.numel() == n
                 and (n <= 1 or mask.stride(0) == 1), "out['mask'] must be a contiguous int32 / uint32 tensor of n elements")
        f32 = xyz.dtype == torch.float32
        p = C.c_void_p(xyz.data_ptr())
        stream = torch.cuda.current_stream(xyz.device).cuda_stream
        _check(lib().tri_project_points_device(self._h, flags | fmt, p if f32 else None, None if f32 else p, n,
                                               C.c_void_p(xy.data_ptr()) if xy is not None else None, stride,
                                               C.c_void_p(mask.data_ptr()) if mask is not None else None, C.c_void_p(stream)))
        return out

    # ---- Triangulator::triangulatePoint over many camera subsets ----
    def triangulate_subsets(self, mode, items, flags=0):
        """items: list of (cam_idx list, xy list-of-pairs).  -> (xyz [n,3], err [n], iters [n])."""
        n = len(items)
        offs = np.zeros(n + 1, np.int32)
        for i, (ci, _) in enumerate(items):
            offs[i + 1] = offs[i] + len(ci)
        cam = np.concatenate([np.asarray(ci, np.int32) for ci, _ in items]) if n else np.zeros(0, np.int32)
        xy = np.concatenate([np.asarray(p, np.float64).reshape(-1, 2) for _, p in items]) if n else np.zeros((0, 2))
        xyz, err, it = np.zeros((n, 3)), np.zeros(n), np.zeros(n, np.int32)
        _check(lib().tri_triangulate_subsets(self._h, mode, flags, n, _np_ptr(offs), _np_ptr(cam), _np_ptr(xy),
                                             _np_ptr(xyz), _np_ptr(err), _np_ptr(it)), mode)
        return xyz, err, it

    def triangulate_point(self, mode, cam_idx, xy, flags=0):
        xyz, err, it = self.triangulate_subsets(mode, [(cam_idx, xy)], flags)
        return xyz[0], float(err[0]), int(it[0])

    def dist_from_ray(self, cam_idx, xy, points):
        cam = np.ascontiguousarray(cam_idx, np.int32)
        xy = np.ascontiguousarray(xy, np.float64).reshape(-1, 2)
        pts = np.ascontiguousarray(points, np.float64).reshape(-1, 3)
        out = np.zeros(len(cam))
        _check(lib().tri_dist_from_ray(self._h, len(cam), _np_ptr(cam), _np_ptr(xy), _np_ptr(pts), _np_ptr(out)))
        return out

    # ---- DroneClassifier::classifyDrones ----
    def classify(self, mode, n_drones, det_offsets, dets_xy, n_frames, flags=0):
        n_cams = len(self.cameras)
        offs = np.ascontiguousarray(det_offsets, np.int32)
        xy = np.ascontiguousarray(dets_xy, np.float64)
        paths = np.zeros((n_drones, n_frames, 3))
        assign = np.zeros((n_drones, n_frames, n_cams), np.int8)
        phase = np.zeros((n_drones, n_frames), np.uint8)
        st = ClassifyStats()
        _check(lib().tri_classify(self._h, mode, flags, n_drones, _np_ptr(offs), _np_ptr(xy), n_frames, _np_ptr(paths),
                                  _np_ptr(assign), _np_ptr(phase), C.byref(st)), mode)
        return dict(paths=paths, assign=assign, phase=phase, stats=st.as_dict())


    def classify_sequences(self, mode, n_drones, seq_bounds, det_offsets, dets_xy, n_frames, flags=0):
        """Independent sequences back to back in one CSR: seq_bounds [n_seq + 1] frame indices (tri_classify_sequences)."""
        n_cams = len(self.cameras)
        sb = np.ascontiguousarray(seq_bounds, np.int32)
        offs = np.ascontiguousarray(det_offsets, np.int32)
        xy = np.ascontiguousarray(dets_xy, np.float64)
        paths = np.zeros((n_drones, n_frames, 3))
        assign = np.zeros((n_drones, n_frames, n_cams), np.int8)
        phase = np.zeros((n_drones, n_frames), np.uint8)
        st = ClassifyStats()
        _check(lib().tri_classify_sequences(self._h, mode, flags, n_drones, len(sb) - 1, _np_ptr(sb), _np_ptr(offs), _np_ptr(xy), n_frames,
                                            _np_ptr(paths), _np_ptr(assign), _np_ptr(phase), C.byref(st)), mode)
        return dict(paths=paths, assign=assign, phase=phase, stats=st.as_dict())

    # ---- frame-sharded classification: enumerate now, link when the previous shard's state has arrived ----
    def classify_begin(self, mode, n_drones, det_offsets, dets_xy, n_frames, flags=0):
        offs = np.ascontiguousarray(det_offsets, np.int32)
        xy = np.ascontiguousarray(dets_xy, np.float64)
        self._cls_job = (mode, n_drones, n_frames)
        _check(lib().tri_classify_begin(self._h, mode, flags, n_drones, _np_ptr(offs), _np_ptr(xy), n_frames), mode)

    def classify_finish(self, state=None):
        """state: the bytes the previous shard's classify_finish returned (None at the start of the sequence).
        Returns the same dict as classify() for this shard's frames, plus 'state' for the next shard."""
        mode, n_drones, n_frames = self._cls_job
        n_cams = len(self.cameras)
        paths = np.zeros((n_drones, n_frames, 3))
        assign = np.zeros((n_drones, n_frames, n_cams), np.int8)
        phase = np.zeros((n_drones, n_frames), np.uint8)
        st = ClassifyStats()
        nb = lib().tri_classify_state_bytes()
        s_in = None
        if state is not None:
            s_in = np.frombuffer(bytes(state), np.uint8).copy()
            assert s_in.size == nb
        s_out = np.zeros(nb, np.uint8)
        _check(lib().tri_classify_finish(self._h, _np_ptr(s_in) if s_in is not None else None, _np_ptr(s_out), _np_ptr(paths),
                                         _np_ptr(assign), _np_ptr(phase), C.byref(st)), mode)
        return dict(paths=paths, assign=assign, phase=phase, stats=st.as_dict(), state=s_out.tobytes())


def classify_multi(engines, mode, n_drones, det_offsets, dets_xy, n_frames, flags=0):
    """tri_classify_multi: one sequence, frame-sharded over several engines (one per GPU) from one process."""
    n_cams = len(engines[0].cameras)
    offs = np.ascontiguousarray(det_offsets, np.int32)
    xy = np.ascontiguousarray(dets_xy, np.float64)
    paths = np.zeros((n_drones, n_frames, 3))
    assign = np.zeros((n_drones, n_frames, n_cams), np.int8)
    phase = np.zeros((n_drones, n_frames), np.uint8)
    st = ClassifyStats()
    hs = (C.c_void_p * len(engines))(*[e._h for e in engines])
    _check(lib().tri_classify_multi(hs, len(engines), mode, flags, n_drones, _np_ptr(offs), _np_ptr(xy), n_frames, _np_ptr(paths),
                                    _np_ptr(assign), _np_ptr(phase), C.byref(st)), mode)
    return dict(paths=paths, assign=assign, phase=phase, stats=st.as_dict())


def triangulate_points_multi(engines, mode, xy, flags=0, want=("xyz_f64",)):
    """tri_triangulate_points_multi: one host batch sharded over several engines (one per GPU)."""
    xy = np.ascontiguousarray(xy)
    fmt = _PIX_DTYPES[xy.dtype]
    npc, nf = xy.shape[0], xy.shape[1]
    out = {k: np.empty({"xyz_f32": (nf, 3), "xyz_f64": (nf, 3)}.get(k, (nf,)),
                       {"xyz_f32": np.float32, "xyz_f64": np.float64, "mask": np.uint32, "err": np.float64, "iters": np.int32}[k])
           for k in want}
    bo = _BatchOut(*[out[k].ctypes.data if k in out else None for k in ("xyz_f32", "xyz_f64", "mask", "err", "iters")])
    hs = (C.c_void_p * len(engines))(*[e._h for e in engines])
    bad = C.c_int64(-1)
    st = lib().tri_triangulate_points_multi(hs, len(engines), mode, flags | fmt, _np_ptr(xy), npc, nf, nf, C.byref(bo), C.byref(bad))
    out["first_bad_frame"] = bad.value
    _check(st, mode)
    return out


def pinned_empty(shape, dtype):
    """A page-locked numpy array owned by the library's allocator (tri_host_alloc)."""
    dtype = np.dtype(dtype)
    n = int(np.prod(shape)) * dtype.itemsize
    p = C.c_void_p()
    _check(lib().tri_host_alloc(C.byref(p), n))
    buf = (C.c_char * max(n, 1)).from_address(p.value)
    arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
    return arr, p


def pinned_free(p):
    lib().tri_host_free(p)
