"""ctypes wrapper around oracle_mls/libppp_oracle_mls.so -- CPU ORACLE of the MLS pre-filter, TEST
INFRASTRUCTURE ONLY (the same rules as oracle/ppp_oracle.py: the product package never imports it)."""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libppp_oracle_mls.so")
_SRCS = [os.path.join(_HERE, "ppp_oracle_mls.cpp"), os.path.join(_HERE, "..", "oracle", "ppp_oracle.cpp")]

_f32p = C.POINTER(C.c_float)
_i32p = C.POINTER(C.c_int32)


def build(force=False):
    if force or not os.path.exists(_SO) or any(os.path.getmtime(s) > os.path.getmtime(_SO) for s in _SRCS):
        subprocess.check_call(["make", "-C", _HERE, "-s"])
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_SO)
        L.ppo_cloud_create.restype = C.c_void_p
        L.ppo_cloud_create.argtypes = [_f32p, C.c_int64, C.c_int64]
        L.ppo_cloud_destroy.argtypes = [C.c_void_p]
        L.ppo_mls_smooth.restype = C.c_int64
        L.ppo_mls_smooth.argtypes = [C.c_void_p, C.c_double, C.c_int, _f32p, _f32p, _i32p, C.POINTER(C.c_int8), C.c_int]
        _lib = L
    return _lib


def mls_smooth(pts, radius=15.0, order=3, threads=0):
    """MovingLeastSquares as the reference's smooth() runs it.  pts: (N, >=3) float32 records.
    Returns (xyz (m, 3) float32, normals (m, 4) float32 {nx, ny, nz, curvature}, src_index (m,) int32,
    fit (m,) int8: 1 = polynomial projection, 0 = plane projection)."""
    pts = np.ascontiguousarray(pts, dtype=np.float32)
    n = pts.shape[0]
    L = lib()
    h = L.ppo_cloud_create(pts.ctypes.data_as(_f32p), n, pts.shape[1])
    try:
        xyz = np.empty((max(n, 1), 3), np.float32)
        nrm = np.empty((max(n, 1), 4), np.float32)
        src = np.empty(max(n, 1), np.int32)
        fit = np.empty(max(n, 1), np.int8)
        m = L.ppo_mls_smooth(h, float(radius), int(order), xyz.ctypes.data_as(_f32p), nrm.ctypes.data_as(_f32p),
                             src.ctypes.data_as(_i32p), fit.ctypes.data_as(C.POINTER(C.c_int8)), int(threads))
    finally:
        L.ppo_cloud_destroy(h)
    if m < 0:
        raise ValueError("order must be 0..3")
    return xyz[:m].copy(), nrm[:m].copy(), src[:m].copy(), fit[:m].copy()
