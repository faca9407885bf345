"""ctypes wrapper around oracle_voxel/libppp_oracle_voxel.so -- CPU ORACLE of the VoxelGrid pre-filter, TEST
INFRASTRUCTURE ONLY (the same rules as oracle/ppp_oracle.py: the product package never imports it)."""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libppp_oracle_voxel.so")
_SRC = os.path.join(_HERE, "ppp_oracle_voxel.cpp")

_f32p = C.POINTER(C.c_float)
_i32p = C.POINTER(C.c_int32)
_i64p = C.POINTER(C.c_int64)

PCL_ORDER = 0      # libstdc++ std::sort with PCL's comparator: the order PCL sums each voxel in
STABLE_ORDER = 1   # std::stable_sort: ascending source index inside each voxel (the device's order)


class Overflow(Exception):
    """PCL warns "Leaf size is too small for the input dataset. Integer indices would overflow." and keeps the input."""


def build(force=False):
    if force or not os.path.exists(_SO) or os.path.getmtime(_SRC) > os.path.getmtime(_SO):
        subprocess.check_call(["make", "-C", _HERE, "-s"])
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_SO)
        L.ppo_voxel_grid.restype = C.c_int64
        L.ppo_voxel_grid.argtypes = [_f32p, C.c_int64, C.c_int64, _f32p, _f32p, _i64p, _i32p, C.c_int]
        _lib = L
    return _lib


def voxel_grid(pts, leaf, order=STABLE_ORDER):
    """VoxelGrid::applyFilter as the reference's voxel_down() runs it.  pts: (N, sf) float32 records (sf >= 5: float 4
    holds the rgba bits); leaf: a float or three.  Returns (records (m, sf) float32, row_offsets (m + 1,) int64, members
    (n_finite,) int32).  Raises ValueError for an invalid leaf and Overflow where PCL keeps the input."""
    pts = np.ascontiguousarray(pts, dtype=np.float32)
    n, sf = pts.shape
    lf = np.broadcast_to(np.asarray(leaf, np.float32), (3,)).copy()
    out = np.empty((max(n, 1), sf), np.float32)
    off = np.empty(max(n, 1) + 1, np.int64)
    mem = np.empty(max(n, 1), np.int32)
    m = lib().ppo_voxel_grid(pts.ctypes.data_as(_f32p), n, sf, lf.ctypes.data_as(_f32p), out.ctypes.data_as(_f32p),
                             off.ctypes.data_as(_i64p), mem.ctypes.data_as(_i32p), int(order))
    if m == -1:
        raise ValueError("leaf sizes must be > 0 and finite, with a finite float inverse")
    if m == -2:
        raise Overflow("Leaf size is too small for the input dataset. Integer indices would overflow.")
    if m == -3:
        raise Overflow("coordinate / leaf size exceeds the int range of the voxel coordinates")
    off = off[:m + 1].copy()
    return out[:m].copy(), off, mem[:int(off[-1])].copy()
