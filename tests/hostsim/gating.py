"""ctypes front end of the test-only CPU build of the innovation gate (see gating.cpp).

Compiled with g++ on first use into a temporary directory of this process, with the flags of tests/hostsim/innovation.py
(-ffp-contract=off: only the explicit fma_ calls of the header fuse, like the nvcc build)."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "gating.cpp")

_lib = None


def lib():
    global _lib
    if _lib is None:
        tmp = tempfile.mkdtemp(prefix="hostsim_gating_")
        atexit.register(shutil.rmtree, tmp, True)
        so = os.path.join(tmp, "libhostsim_gating.so")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-x", "c++", "-ffp-contract=off", "-fPIC", "-shared", "-o", so, SRC])
        _lib = C.CDLL(so)
    return _lib


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t)) if a is not None else None


def replay(streams, dt, acc_ref, mag_ref, q, r, *, gamma=np.inf, gate=True, precision="f32", algo="qr2",
           compensated=False, innov_model=None):
    """One replay from the reference's initial state.  streams [T,9,N] float32; dt float or [T]; acc_ref, mag_ref
    [3,N]; q, r scalar or [N].  gate False runs the ungated step of the same build.  innov_model None, "full" or
    "tangent".  Returns dict(traj [T,N,4], gated [T,N] bool, x [4,N], p [10,N] (P/r), innov [2,N]), float64."""
    streams = np.ascontiguousarray(streams, dtype=np.float32)
    T, _, N = streams.shape
    dt = np.atleast_1d(np.asarray(dt, dtype=np.float64))
    acc_ref = np.ascontiguousarray(acc_ref, dtype=np.float32)
    mag_ref = np.ascontiguousarray(mag_ref, dtype=np.float32)
    q = np.ascontiguousarray(np.broadcast_to(np.asarray(q, dtype=np.float32), (N,)))
    r = np.ascontiguousarray(np.broadcast_to(np.asarray(r, dtype=np.float32), (N,)))
    out = dict(traj=np.empty((T, N, 4)), gated=np.zeros((T, N), dtype=np.uint8), x=np.empty((4, N)), p=np.empty((10, N)),
               innov=np.empty((2, N)))
    rc = lib().hostsim_gating(C.c_int({"f32": 0, "f64": 1, "f32x2": 2}[precision]), C.c_int(0 if algo == "qr2" else 1),
                              C.c_int(int(compensated)), C.c_int(int(gate)),
                              C.c_int({None: 0, "full": 1, "tangent": 2}[innov_model]), C.c_float(gamma), C.c_int64(N),
                              C.c_int64(T), _p(streams, C.c_float), _p(dt, C.c_double), C.c_int(int(dt.size > 1)),
                              _p(acc_ref, C.c_float), _p(mag_ref, C.c_float), _p(q, C.c_float), _p(r, C.c_float),
                              _p(out["traj"], C.c_double), _p(out["gated"], C.c_uint8), _p(out["x"], C.c_double),
                              _p(out["p"], C.c_double), _p(out["innov"], C.c_double))
    assert rc == 0
    out["gated"] = out["gated"].astype(bool)
    return out
