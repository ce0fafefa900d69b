"""TEST / BASELINE INFRASTRUCTURE ONLY -- ctypes wrapper of oracle/advect_rk4_3d.c (C + OpenMP restatement of
Kernel.execute([AdvectionRK4_3D, DeleteParticle]) on a float64-coordinate, float32-data rectilinear A-grid).
Never imported by the product."""

from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "_build", "liboracle_c.so")


class _Grid(C.Structure):
    _fields_ = [("lon", C.c_void_p), ("lat", C.c_void_p), ("depth", C.c_void_p), ("time", C.c_void_p), ("nx", C.c_int),
                ("ny", C.c_int), ("nz", C.c_int), ("nt", C.c_int), ("spherical", C.c_int), ("deg2m", C.c_double),
                ("U", C.c_void_p), ("V", C.c_void_p), ("W", C.c_void_p)]  # fmt: skip


def needs_build():
    return not os.path.exists(LIB) or os.path.getmtime(LIB) < os.path.getmtime(os.path.join(HERE, "advect_rk4_3d.c"))


def build():
    """Compile to ``LIB`` (set it to a path outside the tree to build there)."""
    if needs_build():
        subprocess.run(["make", "-C", HERE, "-B", f"LIB={LIB}", LIB], check=True, capture_output=True)
    return LIB


_lib = None


def _load():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        _lib.advect_rk4_3d.restype = C.c_long
        _lib.advect_rk4_3d.argtypes = [C.POINTER(_Grid), C.c_long] + [C.c_void_p] * 6 + [C.c_double, C.c_double]
    return _lib


def advect_rk4_3d(*, lon, lat, depth, time, U, V, W, spherical, deg2m, pdata, dt, endtime, threads=None):
    """In-place on pdata (x, y, z f32; t f64; state, ei i32); deleted particles are compacted like the reference does.
    Returns the number of particle-steps."""
    lib = _load()
    arrs = [np.ascontiguousarray(a, dtype=np.float64) for a in (lon, lat, depth, np.asarray(time) - np.asarray(time)[0])]
    fld = [np.ascontiguousarray(a, dtype=np.float32) for a in (U, V, W)]
    T, Z, Y, X = fld[0].shape
    g = _Grid(*(a.ctypes.data for a in arrs), X, Y, Z, T, int(bool(spherical)), float(deg2m), *(a.ctypes.data for a in fld))
    if threads:
        os.environ["OMP_NUM_THREADS"] = str(threads)
    ei = np.ascontiguousarray(pdata["ei"][:, -1])
    n = len(pdata["x"])
    steps = lib.advect_rk4_3d(C.byref(g), n, *(pdata[k].ctypes.data for k in ("x", "y", "z", "t", "state")), ei.ctypes.data,
                              float(dt), float(endtime))  # fmt: skip
    pdata["ei"][:, -1] = ei
    keep = pdata["state"] != 30
    if not keep.all():
        for k in pdata:
            pdata[k] = pdata[k][keep]
    return steps
