"""ctypes front end of the test-only CPU build of the general-matrix innovation terms and gate (see
general_innovation.cpp).

Compiled with g++ on first use into a temporary directory of this process, with the flags of tests/hostsim/gating.py
(-ffp-contract=off: only the explicit fma_ calls of the header fuse, like the nvcc build)."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

from tests.hostsim.general_qr import ALGO, TRI3, TRI4, tri

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "general_innovation.cpp")

_lib = None


def lib():
    global _lib
    if _lib is None:
        tmp = tempfile.mkdtemp(prefix="hostsim_general_innovation_")
        atexit.register(shutil.rmtree, tmp, True)
        so = os.path.join(tmp, "libhostsim_general_innovation.so")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-x", "c++", "-ffp-contract=off", "-fPIC", "-shared", "-o", so, SRC])
        _lib = C.CDLL(so)
    return _lib


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


def replay(streams, dt, acc_ref, mag_ref, Q, R, *, model="full", gamma=None, precision="f32", algo="qr2"):
    """One replay from the reference's initial state.  streams [T,9,N] float32; dt float or [T]; acc_ref, mag_ref [3,N];
    Q [N,3,3], R [N,4,4]; model "full" or "tangent"; gamma None (ungated) or the NIS3 threshold.  Returns dict(terms
    [2,T,N] (NIS_t, ln det S_t), gated [T,N] bool, innov [2,N] the sums of the same build, traj [T,N,4]), float64."""
    streams = np.ascontiguousarray(streams, dtype=np.float32)
    T, _, N = streams.shape
    dt = np.atleast_1d(np.asarray(dt, dtype=np.float64))
    acc_ref = np.ascontiguousarray(acc_ref, dtype=np.float32)
    mag_ref = np.ascontiguousarray(mag_ref, dtype=np.float32)
    q_tri = np.ascontiguousarray(tri(Q, TRI3), dtype=np.float32)
    r_tri = np.ascontiguousarray(tri(R, TRI4), dtype=np.float32)
    out = dict(terms=np.empty((2, T, N)), gated=np.zeros((T, N), dtype=np.uint8), innov=np.empty((2, N)),
               traj=np.empty((T, N, 4)))
    rc = lib().hostsim_general_innovation(
        C.c_int({"f32": 0, "f64": 1}[precision]), C.c_int(ALGO[algo]), C.c_int({"full": 0, "tangent": 1}[model]),
        C.c_int(gamma is not None), C.c_float(0.0 if gamma is None else gamma), C.c_int64(N), C.c_int64(T),
        _p(streams, C.c_float), _p(dt, C.c_double), C.c_int(int(dt.size > 1)), _p(acc_ref, C.c_float),
        _p(mag_ref, C.c_float), _p(q_tri, C.c_float), _p(r_tri, C.c_float), _p(out["terms"], C.c_double),
        _p(out["gated"], C.c_uint8), _p(out["innov"], C.c_double), _p(out["traj"], C.c_double))
    assert rc == 0
    out["gated"] = out["gated"].astype(bool)
    return out
