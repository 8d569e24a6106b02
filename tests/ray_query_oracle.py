"""ctypes binding for tests/ray_query_oracle.cpp: the CPU oracle's answers to the ray queries (TEST INFRASTRUCTURE ONLY).

The library is compiled once per process into a temporary directory (the tree is never written), with the flags of
oracle/Makefile, and takes the prepared-scene handles of oracle.pyoracle (the same oracle.cpp is compiled into it).
"""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_CXX = os.environ.get("ORACLE_CXX", "/usr/bin/g++")
_FLAGS = ["-O2", "-ffp-contract=off", "-fno-fast-math", "-pthread", "-fPIC", "-std=c++17", "-Wall", "-Wextra"]
_lib = None


def lib():
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="ray_query_oracle_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libray_query_oracle.so")
        subprocess.check_call([_CXX, *_FLAGS, "-shared", "-o", so, os.path.join(_HERE, "ray_query_oracle.cpp")])
        L = C.CDLL(so)
        vp, i64, i32 = C.c_void_p, C.c_int64, C.c_int32
        L.oracle_intersect_rays.restype = C.c_int
        L.oracle_intersect_rays.argtypes = [vp, vp, i64, vp, vp, vp, i32]
        L.oracle_trace_rays.restype = C.c_int
        L.oracle_trace_rays.argtypes = [vp, vp, i64, vp, i32]
        _lib = L
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def intersect_rays(prepared, rays, want_pn=False, threads=0):
    """objs_hit per ray on an oracle.pyoracle.Prepared (rays: (n, 6) float32 origin, direction).  Returns (index int32[n]
    in the scene's sphere order or -1, t float32[n] or +inf, pn float32[n][6] or None)."""
    r = np.ascontiguousarray(rays, dtype=np.float32).reshape(-1, 6)
    n = r.shape[0]
    index = np.empty(n, np.int32)
    t = np.empty(n, np.float32)
    pn = np.empty((n, 6), np.float32) if want_pn else None
    rc = lib().oracle_intersect_rays(prepared._h, _p(r), n, _p(index), _p(t), _p(pn), int(threads))
    if rc != 0:
        raise RuntimeError(f"oracle_intersect_rays failed ({rc}: 2 = the leaf fold disagrees with objs_hit)")
    return index, t, pn


def trace_rays(prepared, rays, threads=0):
    """ray_colour objs r 50 per ray: float32[n][3], before quantisation."""
    r = np.ascontiguousarray(rays, dtype=np.float32).reshape(-1, 6)
    colour = np.empty((r.shape[0], 3), np.float32)
    if lib().oracle_trace_rays(prepared._h, _p(r), r.shape[0], _p(colour), int(threads)) != 0:
        raise RuntimeError("oracle_trace_rays failed")
    return colour
