"""ctypes view of tests/native/libnearest_oracle.so, the CPU reference of the nearest-triangle query — TEST
INFRASTRUCTURE ONLY.  It computes the point-triangle distance in the same binary32 operation order as k_nearest and
defines rt_query_nearest's result as a brute force over every triangle (lowest id on exact ties)."""
from __future__ import annotations

import ctypes as C
import importlib
import os
import subprocess

import numpy as np

rt = importlib.import_module("raytracing2-fork_b200")
NATIVE_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "native")

_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        path = os.path.join(NATIVE_DIR, "libnearest_oracle.so")
        if not os.path.exists(path):
            subprocess.check_call(["make", "-C", NATIVE_DIR, path])
        L = C.CDLL(path)
        L.nro_point_triangle.restype = C.c_float
        _lib = L
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def point_triangle(p, tri):
    """(dist, u, v, closest point) of one point and one rt.TRIANGLE record."""
    p = np.ascontiguousarray(p, dtype=np.float32)
    t = np.ascontiguousarray(tri, dtype=rt.TRIANGLE).reshape(1)
    u, v = C.c_float(), C.c_float()
    q = np.zeros(3, np.float32)
    d = lib().nro_point_triangle(_p(p), _p(t), C.byref(u), C.byref(v), _p(q))
    return np.float32(d), np.float32(u.value), np.float32(v.value), q


def nearest_points(tris, points, max_dist=None):
    """Brute-force nearest triangle of every point: (tri_id, dist, u, v, closest (N, 3))."""
    tris = np.ascontiguousarray(tris, dtype=rt.TRIANGLE)
    p = np.ascontiguousarray(points, dtype=np.float32).reshape(-1, 3)
    n = p.shape[0]
    md = None if max_dist is None else np.ascontiguousarray(np.broadcast_to(np.float32(max_dist), (n,)), np.float32)
    tri = np.zeros(n, np.int32)
    dist, bu, bv = (np.zeros(n, np.float32) for _ in range(3))
    closest = np.zeros((n, 3), np.float32)
    rc = lib().nro_nearest_points(_p(tris), C.c_int64(tris.size), _p(p), _p(md), C.c_int64(n), _p(tri), _p(dist),
                                  _p(bu), _p(bv), _p(closest))
    assert rc == 0, rc
    return tri, dist, bu, bv, closest
