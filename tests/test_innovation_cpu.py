"""Innovation likelihood (the ground-truth-free (Q,R) tuning objective) without a GPU: the CPU build of the device
header (tests/hostsim/innovation.cpp) against the float64 definition (tests/innovation_ref.py), the float and
packed-lane builds against each other, and the argument checks of posekf_replay_innovation_f32."""
import math

import numpy as np
import pytest

from oracle import ekf_oracle as O
from poseestimationkf_b200 import _lib
from tests import innovation_ref as IR
from tests.hostsim import innovation as H

# (q, r, precise): the plain variant, and both extremes of the precise one (R >> Q, Q >> R)
CELLS = [(1.0, 0.1, False), (1e-3, 1e3, True), (1e3, 1e-3, True)]


def _ref(g, tag, q, r):
    S = g[tag + "_streams"].astype(np.float64)
    T = S.shape[0]
    # the CPU build takes q, r (and dt) as the kernels do, in float32: the reference gets the same values
    return IR.replay_innovation(np.full(T, float(np.float32(g["dt"])) * 1e9), S[:, 0:3], S[:, 3:6], S[:, 6:9],
                                g[tag + "_acc_ref"].T, g[tag + "_mag_ref"].T, float(np.float32(q)), float(np.float32(r)))


def test_reference_replays_the_oracle_recursion(golden_traj):
    """The float64 definition runs the oracle's own recursion: same trajectory and flips, bit for bit."""
    g = golden_traj
    S = g["noisy_streams"].astype(np.float64)
    T = S.shape[0]
    args = (np.full(T, float(g["dt"]) * 1e9), S[:, 0:3], S[:, 3:6], S[:, 6:9], g["noisy_acc_ref"].T, g["noisy_mag_ref"].T, 1.0, 0.1)
    a, b = IR.replay_innovation(*args), O.replay_batched(*args)
    np.testing.assert_array_equal(a["X"], b["X"])
    np.testing.assert_array_equal(a["flips"], b["flips"])
    # and its terms are what they claim: NIS >= 0, ln det S = ln det(P + rI) >= 4 ln r
    assert (a["nis"] >= 0).all() and (a["logdet"] >= 4 * math.log(0.1) - 1e-12).all()


@pytest.mark.parametrize("tag", ["clean", "noisy"])
@pytest.mark.parametrize("q,r,precise", CELLS)
def test_hostsim_f64_sums_equal_reference(golden_traj, tag, q, r, precise):
    g = golden_traj
    ref = _ref(g, tag, q, r)
    got = H.innovation(g[tag + "_streams"], float(g["dt"]), g[tag + "_acc_ref"], g[tag + "_mag_ref"], q, r, precision="f64",
                       compensated=precise)
    want = np.stack([ref["nis"].sum(0), ref["logdet"].sum(0)])
    np.testing.assert_allclose(got[1], want[1], rtol=1e-9, atol=0)
    # NIS at Q >> R: e = y - z is nearly tangent (e.z ~ -|e|^2/2 ~ 1e-9 here), and S^-1 weighs that component with
    # 1/r = 1e3; both float64 forms form it as a difference of unit quaternions, so each carries ~1e-16/1e-9 relative
    # error there (5e-8 measured): the definition itself is no more accurate than that in float64
    np.testing.assert_allclose(got[0], want[0], rtol=2e-7 if q / r > 1e4 else 1e-9, atol=0)


@pytest.mark.parametrize("q,r,precise", CELLS)
def test_hostsim_f32_close_to_reference(golden_traj, q, r, precise):
    """The float32 arithmetic of the kernels (CPU build): within the device bar of the float64 sums."""
    g = golden_traj
    ref = _ref(g, "noisy", q, r)
    got = H.innovation(g["noisy_streams"], float(g["dt"]), g["noisy_acc_ref"], g["noisy_mag_ref"], q, r, precision="f32",
                       compensated=precise)
    np.testing.assert_allclose(got[0], ref["nis"].sum(0), rtol=1e-4)
    np.testing.assert_allclose(got[1], ref["logdet"].sum(0), rtol=1e-4)


@pytest.mark.parametrize("precise", [False, True])
def test_hostsim_float_and_packed_lanes_bitwise(golden_traj, precise):
    g = golden_traj
    n = g["noisy_streams"].shape[2]
    q = np.logspace(-3, 3, n).astype(np.float32)
    r = np.logspace(2, -2, n).astype(np.float32)
    args = (g["noisy_streams"], float(g["dt"]), g["noisy_acc_ref"], g["noisy_mag_ref"], q, r)
    a = H.innovation(*args, precision="f32", compensated=precise)
    b = H.innovation(*args, precision="f32x2", compensated=precise)
    assert np.isfinite(a).all()
    np.testing.assert_array_equal(a, b)


def _call(lib, n=8, t=4, ns=8, innov=True, flags=0, wahba=0):
    buf = (np.zeros((2, max(n, 1)), dtype=np.float32) if innov else None)
    ptr = None if buf is None else buf.ctypes.data
    return lib.posekf_replay_innovation_f32(n, t, None, ns, None, 0, None, None, None, None, -1.0, -1.0, None, None, None, None,
                                            None, None, None, None, ptr, wahba, 0, flags, None)


def test_entry_point_rejects_bad_arguments_without_gpu():
    lib = _lib.load()
    assert _call(lib, innov=False) == _lib.EINVAL            # innov_acc is required
    assert _call(lib, n=-1) == _lib.EINVAL                    # bad sizes
    assert _call(lib, t=-1) == _lib.EINVAL
    assert _call(lib, ns=3) == _lib.EINVAL                    # N % Ns != 0 ... (and null streams)
    assert _call(lib, ns=0) == _lib.EINVAL
    assert _call(lib, flags=4) == _lib.EINVAL                 # unknown state flag
    assert _call(lib, wahba=7) == _lib.EINVAL
    assert _call(lib, n=0) == 0                               # empty batch: no-op


def test_innovation_nll_helper():
    import torch
    from poseestimationkf_b200 import batched as B
    a = torch.tensor([[3.0, 40.0], [-20.0, 8.0]])
    nll, nis = B.innovation_nll(a, 10)
    want = 0.5 * (a[0].double() + a[1].double()) + 20 * math.log(2 * math.pi)
    assert torch.allclose(nll, want) and torch.allclose(nis, a[0].double() / 10)
    st = B.ReplayState(torch.zeros(4, 2), torch.zeros(10, 2), innov=a)
    assert torch.equal(B.innovation_nll(st, 10)[0], nll) and torch.equal(st.clone().innov, a)
    with pytest.raises(ValueError):
        B.innovation_nll(B.ReplayState(torch.zeros(4, 2), torch.zeros(10, 2)), 10)
