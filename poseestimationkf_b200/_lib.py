"""ctypes binding of libposekf_b200.so (the C ABI declared in include/posekf.h).

There is no CPU implementation behind this module: if the CUDA library is missing, or a call
returns non-zero, an exception is raised."""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

_i64, _int, _f32, _vp = C.c_int64, C.c_int, C.c_float, C.c_void_p

EINVAL, EALIGN, ENODEV = -1, -2, -3
WAHBA = {"qr2": 0, "jacobi": 1, "precomputed": 2}
STAGING = {"auto": 0, "ldg": 1, "tma": 2, "tma_packed": 3}
INNOV_MODEL = {"full": 0, "tangent": 1}      # POSEKF_INNOV_*

_SIGNATURES = {
    "posekf_replay_f32": [_i64, _i64, _vp, _i64, _vp, _int, _vp, _vp, _vp, _vp, _f32, _f32, _vp, _vp, _vp, _vp, _vp,
                          _vp, _vp, _vp, _int, _int, _int, _vp],
    "posekf_replay_innovation_f32": [_i64, _i64, _vp, _i64, _vp, _int, _vp, _vp, _vp, _vp, _f32, _f32, _vp, _vp, _vp, _vp,
                                     _vp, _vp, _vp, _vp, _vp, _int, _int, _int, _vp],
    "posekf_replay_innovation_ex_f32": [_i64, _i64, _vp, _i64, _vp, _int, _vp, _vp, _vp, _vp, _f32, _f32, _vp, _vp, _vp,
                                        _vp, _vp, _vp, _vp, _vp, _vp, _int, _int, _int, _int, _vp],
    "posekf_replay_batch_f32": [_i64, _i64, _vp, _i64, _vp, _int, _vp, _vp, _vp, _vp, _f32, _f32, _vp, _vp, _vp, _vp, _vp,
                                _vp, _vp, _vp, _vp, _int, _int, _int, _int, _vp, _vp, _vp],
    "posekf_replay_gated_f32": [_i64, _i64, _vp, _i64, _vp, _int, _vp, _vp, _vp, _vp, _f32, _f32, _vp, _vp, _vp, _vp, _vp,
                                _vp, _vp, _vp, _vp, _int, _int, _int, _int, _vp, _vp, _vp, _f32, _vp, _vp],
    "posekf_replay_general_f32": [_i64, _i64, _vp, _i64, _vp, _int, _vp, _vp, _vp, _i64, _vp, _i64, _f32, _f32, _vp, _vp, _vp,
                                  _vp, _vp, _vp, _vp, _vp, _vp, _int, _int, _int, _int, _vp, _vp, _vp],
    "posekf_replay_host_f32": [_i64, _i64, _vp, _f32, _vp, _vp, _vp, _vp, _f32, _f32, _vp, _vp, _vp, _vp, _vp, _i64,
                               _int, _int, _int, _vp],
    "posekf_host_workspace_create": [_int, _i64, _i64, _int, C.POINTER(C.c_void_p)],
    "posekf_host_workspace_destroy": [_vp],
    "posekf_wahba_f32": [_i64, _vp, _vp, _int, _vp, _vp, _vp, _vp, _f32, _f32, _int, _vp, _vp, _int, _int, _vp],
    "posekf_tracks_f32": [_i64, _i64, _vp, _i64, _vp, _int, _vp, _vp, _f32, _f32, _int, _vp, _vp, _vp, _int, _vp],
    "posekf_traj2rpy_f32": [_i64, _vp, _vp, _vp],
    "posekf_measurement_stream_f32": [_i64, _i64, _vp, _vp, _vp, _f32, _f32, _vp, _vp, _int, _vp],
    "posekf_initial_values_f32": [_i64, _i64, _vp, _int, _vp, _vp, _vp],
    "posekf_preprocess_f32": [_i64, _i64, _vp, _vp, _vp, _vp, _f32, _f32, _vp, _vp, _vp],
    "posekf_align_events_f32": [_i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp,
                                _vp],
    "posekf_rot2quat_f32": [_i64, _vp, _vp, _vp],
    "posekf_predict_f32": [_i64, _vp, _vp, _int, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "posekf_correct_f32": [_i64, _vp, _vp, _vp, _vp, _int, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _int, _vp],
    "posekf_rk4_f32": [_i64, _vp, _vp, _int, _vp, _vp, _vp],
    "posekf_jacobians_f32": [_i64, _vp, _vp, _vp, _vp, _vp],
    "posekf_comparator_f32": [_i64, _vp, _vp, _vp, _vp],
    "posekf_lowpass_f32": [_i64, _i64, _vp, _f32, _vp, _vp, _vp],
    "posekf_quat2rpy_f32": [_i64, _vp, _vp, _vp],
    "posekf_norm_f32": [_i64, _int, _vp, _vp, _vp],
    "posekf_copy_async": [_vp, _vp, _i64, _int, _vp],
    "posekf_stream_sync": [_vp],
    "posekf_fp32_peak_tflops": [_int, C.POINTER(C.c_double), C.POINTER(C.c_double)],
}
EXPORTS = ["posekf_version"] + list(_SIGNATURES)

_lib = None


class PosekfError(RuntimeError):
    pass


def load(build_if_missing: bool = True) -> C.CDLL:
    """Load (building first if the sources are newer and nvcc is present) the CUDA library."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("POSEKF_LIB", _build.LIB_PATH)      # override: experiment builds (tools/)
    if path == _build.LIB_PATH and build_if_missing and _build.needs_build():
        try:
            _build.build()
        except Exception as exc:  # no nvcc on this machine: use the shipped .so if there is one
            if not os.path.exists(path):
                raise PosekfError(f"libposekf_b200.so is missing and could not be built: {exc}") from exc
    if not os.path.exists(path):
        raise PosekfError(f"{path} not found: build it with `python -m poseestimationkf_b200.build` "
                          "(the package has no CPU fallback)")
    lib = C.CDLL(path)
    lib.posekf_version.restype = C.c_char_p
    lib.posekf_version.argtypes = []
    for name, argtypes in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = _int
        fn.argtypes = argtypes
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc == 0:
        return
    if rc < 0:
        reason = {EINVAL: "invalid argument", EALIGN: "alignment/stride requirement not met",
                  ENODEV: "no usable device / driver entry point"}.get(rc, "error")
        raise PosekfError(f"{what}: {reason} (code {rc})")
    raise PosekfError(f"{what}: CUDA error {rc}")
