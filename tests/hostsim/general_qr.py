"""ctypes front end of the test-only CPU build of the general-matrix step (see general_qr.cpp).

Compiled with g++ on first use into a temporary directory of this process, with the flags of tests/hostsim/gating.py
(-ffp-contract=off: only the explicit fma_ calls of the header fuse, like the nvcc build)."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "general_qr.cpp")

_lib = None
ALGO = {"qr2": 0, "jacobi": 1, "precomputed": 2}
TRI3 = [(0, 0), (0, 1), (0, 2), (1, 1), (1, 2), (2, 2)]
TRI4 = [(0, 0), (0, 1), (0, 2), (0, 3), (1, 1), (1, 2), (1, 3), (2, 2), (2, 3), (3, 3)]


def lib():
    global _lib
    if _lib is None:
        tmp = tempfile.mkdtemp(prefix="hostsim_general_qr_")
        atexit.register(shutil.rmtree, tmp, True)
        so = os.path.join(tmp, "libhostsim_general_qr.so")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-x", "c++", "-ffp-contract=off", "-fPIC", "-shared", "-o", so, SRC])
        _lib = C.CDLL(so)
    return _lib


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


def tri(M, idx):
    """[N,k,k] -> [len(idx),N] upper triangle, row-major."""
    M = np.asarray(M, dtype=np.float64)
    return np.stack([M[:, i, j] for i, j in idx])


def replay(streams, dt, acc_ref, mag_ref, Q, R, *, precision="f32", algo="qr2", isotropic=False):
    """One replay from the reference's initial state.  streams [T,9,N] float32; dt float or [T]; acc_ref, mag_ref [3,N];
    Q [N,3,3], R [N,4,4] (isotropic: q [N], r [N] and the isotropic step of the same build).  Returns dict(traj [T,N,4],
    flips [T,N] bool, x [4,N], p [10,N] (unscaled)), float64."""
    streams = np.ascontiguousarray(streams, dtype=np.float32)
    T, _, N = streams.shape
    dt = np.atleast_1d(np.asarray(dt, dtype=np.float64))
    acc_ref = np.ascontiguousarray(acc_ref, dtype=np.float32)
    mag_ref = np.ascontiguousarray(mag_ref, dtype=np.float32)
    if isotropic:
        q_tri = np.ascontiguousarray(np.broadcast_to(np.asarray(Q, dtype=np.float32), (N,)))
        r_tri = np.ascontiguousarray(np.broadcast_to(np.asarray(R, dtype=np.float32), (N,)))
    else:
        q_tri = np.ascontiguousarray(tri(Q, TRI3), dtype=np.float32)
        r_tri = np.ascontiguousarray(tri(R, TRI4), dtype=np.float32)
    out = dict(traj=np.empty((T, N, 4)), flips=np.zeros((T, N), dtype=np.uint8), x=np.empty((4, N)), p=np.empty((10, N)))
    rc = lib().hostsim_general_qr(C.c_int({"f32": 0, "f64": 1}[precision]), C.c_int(ALGO[algo]), C.c_int(0 if isotropic else 1),
                                  C.c_int64(N), C.c_int64(T), _p(streams, C.c_float), _p(dt, C.c_double),
                                  C.c_int(int(dt.size > 1)), _p(acc_ref, C.c_float), _p(mag_ref, C.c_float),
                                  _p(q_tri, C.c_float), _p(r_tri, C.c_float), _p(out["traj"], C.c_double),
                                  _p(out["flips"], C.c_uint8), _p(out["x"], C.c_double), _p(out["p"], C.c_double))
    assert rc == 0
    out["flips"] = out["flips"].astype(bool)
    return out
