"""Tangent-space innovation likelihood without a GPU: the float64 definition (tests/innovation_tangent_ref.py) against the
oracle, against a second basis and against the basis-free algebra of the kernels; the CPU build of the device header
(tests/hostsim/innovation_tangent.cpp) against the definition; the argument checks of posekf_replay_innovation_ex_f32;
the 3-DOF constant of innovation_nll; and where the objective puts its argmin."""
import math

import numpy as np
import pytest

from oracle import ekf_oracle as O
from poseestimationkf_b200 import _lib
from poseestimationkf_b200.synth import make_imu
from tests import innovation_tangent_ref as TR
from tests.hostsim import innovation_tangent as HT

# (q, r, precise): the plain variant, and both extremes of the precise one (R >> Q, Q >> R)
CELLS = [(1.0, 0.1, False), (1e-3, 1e3, True), (1e3, 1e-3, True)]


def _args(g, tag, q, r):
    S = g[tag + "_streams"].astype(np.float64)
    T = S.shape[0]
    # the CPU build takes q, r (and dt) as the kernels do, in float32: the definition gets the same values
    return (np.full(T, float(np.float32(g["dt"])) * 1e9), S[:, 0:3], S[:, 3:6], S[:, 6:9], g[tag + "_acc_ref"].T,
            g[tag + "_mag_ref"].T, float(np.float32(q)), float(np.float32(r)))


def _sums(d):
    return np.stack([d["nis"].sum(0), d["logdet"].sum(0)])


def test_definition_replays_the_oracle_recursion(golden_traj):
    g = golden_traj
    S = g["noisy_streams"].astype(np.float64)
    T = S.shape[0]
    args = (np.full(T, float(g["dt"]) * 1e9), S[:, 0:3], S[:, 3:6], S[:, 6:9], g["noisy_acc_ref"].T, g["noisy_mag_ref"].T, 1.0, 0.1)
    a, b = TR.replay_tangent(*args), O.replay_batched(*args)
    np.testing.assert_array_equal(a["X"], b["X"])
    np.testing.assert_array_equal(a["flips"], b["flips"])
    # NIS3 >= 0; S3 = E^T (P + rI) E >= rI3, so ln det S3 >= 3 ln r
    assert (a["nis"] >= 0).all() and (a["logdet"] >= 3 * math.log(0.1) - 1e-12).all()


def test_bases_are_orthonormal_and_tangent():
    rng = np.random.default_rng(1)
    u = rng.standard_normal((64, 4))
    u[0] = [1, 0, 0, 0]
    u[1] = [-1, 0, 0, 0]
    u /= np.linalg.norm(u, axis=1)[:, None]
    for name, f in TR.BASES.items():
        E = f(u)
        np.testing.assert_allclose(E.transpose(0, 2, 1) @ E, np.tile(np.identity(3), (64, 1, 1)), atol=1e-14, err_msg=name)
        np.testing.assert_allclose(np.einsum("nij,ni->nj", E, u), 0.0, atol=1e-14, err_msg=name)


@pytest.mark.parametrize("tag", ["clean", "noisy"])
@pytest.mark.parametrize("q,r,precise", CELLS)
def test_definition_does_not_depend_on_the_basis(golden_traj, tag, q, r, precise):
    args = _args(golden_traj, tag, q, r)
    a, b = _sums(TR.replay_tangent(*args, basis="householder")), _sums(TR.replay_tangent(*args, basis="qr"))
    np.testing.assert_allclose(a, b, rtol=1e-12, atol=0)


@pytest.mark.parametrize("tag", ["clean", "noisy"])
@pytest.mark.parametrize("q,r,precise", CELLS)
def test_schur_algebra_equals_definition(golden_traj, tag, q, r, precise):
    args = _args(golden_traj, tag, q, r)
    want, got = _sums(TR.replay_tangent(*args)), _sums(TR.replay_tangent(*args, form="schur"))
    np.testing.assert_allclose(got, want, rtol=1e-9, atol=0)


@pytest.mark.parametrize("tag", ["clean", "noisy"])
@pytest.mark.parametrize("q,r,precise", CELLS)
def test_hostsim_f64_sums_equal_definition(golden_traj, tag, q, r, precise):
    g = golden_traj
    want = _sums(TR.replay_tangent(*_args(g, tag, q, r)))
    got = HT.innovation_tangent(g[tag + "_streams"], float(g["dt"]), g[tag + "_acc_ref"], g[tag + "_mag_ref"], q, r,
                                precision="f64", compensated=precise)
    np.testing.assert_allclose(got[1], want[1], rtol=1e-9, atol=0)
    # NIS3 = s - b^2/c: at Q >> R the metric S~^-1 weighs the previous state's direction ~1 and the tangent directions
    # ~4r/q, so s and b^2/c nearly cancel when the state moves slowly (measured 3e-11 on these trajectories)
    np.testing.assert_allclose(got[0], want[0], rtol=1e-8 if q / r > 1e4 else 1e-9, atol=0)


@pytest.mark.parametrize("tag", ["clean", "noisy"])
@pytest.mark.parametrize("q,r,precise", CELLS)
def test_hostsim_f32_close_to_definition(golden_traj, tag, q, r, precise):
    """The float32 arithmetic of the kernels (CPU build): within 1e-4 of the float64 sums, relative to the likelihood they
    form (|sum NIS3| + |sum ln det S3|)."""
    g = golden_traj
    want = _sums(TR.replay_tangent(*_args(g, tag, q, r)))
    got = HT.innovation_tangent(g[tag + "_streams"], float(g["dt"]), g[tag + "_acc_ref"], g[tag + "_mag_ref"], q, r,
                                precision="f32", compensated=precise)
    scale = np.abs(want[0]) + np.abs(want[1])
    assert float(np.max(np.abs(got - want) / scale)) <= 1e-4


@pytest.mark.parametrize("precise", [False, True])
def test_hostsim_float_and_packed_lanes_bitwise(golden_traj, precise):
    g = golden_traj
    n = g["noisy_streams"].shape[2]
    q = np.logspace(-3, 3, n).astype(np.float32)
    r = np.logspace(2, -2, n).astype(np.float32)
    args = (g["noisy_streams"], float(g["dt"]), g["noisy_acc_ref"], g["noisy_mag_ref"], q, r)
    a = HT.innovation_tangent(*args, precision="f32", compensated=precise)
    b = HT.innovation_tangent(*args, precision="f32x2", compensated=precise)
    assert np.isfinite(a).all()
    np.testing.assert_array_equal(a, b)


def _call(lib, n=8, t=4, ns=8, innov=True, flags=0, wahba=0, model=1):
    buf = (np.zeros((2, max(n, 1)), dtype=np.float32) if innov else None)
    ptr = None if buf is None else buf.ctypes.data
    return lib.posekf_replay_innovation_ex_f32(n, t, None, ns, None, 0, None, None, None, None, -1.0, -1.0, None, None, None,
                                               None, None, None, None, None, ptr, model, wahba, 0, flags, None)


def test_ex_entry_point_rejects_bad_arguments_without_gpu():
    lib = _lib.load()
    for model in (0, 1):
        assert _call(lib, innov=False, model=model) == _lib.EINVAL      # innov_acc is required
        assert _call(lib, n=-1, model=model) == _lib.EINVAL
        assert _call(lib, t=-1, model=model) == _lib.EINVAL
        assert _call(lib, ns=3, model=model) == _lib.EINVAL
        assert _call(lib, ns=0, model=model) == _lib.EINVAL
        assert _call(lib, flags=4, model=model) == _lib.EINVAL          # unknown state flag
        assert _call(lib, wahba=7, model=model) == _lib.EINVAL
        assert _call(lib, n=0, model=model) == 0                        # empty batch: no-op
    for model in (-1, 2, 7):
        assert _call(lib, model=model) == _lib.EINVAL                   # unknown model
        assert _call(lib, n=0, model=model) == _lib.EINVAL


def test_innovation_nll_applies_the_model_constant():
    import torch
    from poseestimationkf_b200 import batched as B
    a = torch.tensor([[3.0, 40.0], [-20.0, 8.0]])
    base = 0.5 * (a[0].double() + a[1].double())
    nll3, nis3 = B.innovation_nll(a, 10, model="tangent")
    assert torch.allclose(nll3, base + 15 * math.log(2 * math.pi)) and torch.allclose(nis3, a[0].double() / 10)
    assert torch.allclose(B.innovation_nll(a, 10)[0], base + 20 * math.log(2 * math.pi))      # a bare tensor: "full"
    st = B.ReplayState(torch.zeros(4, 2), torch.zeros(10, 2), innov=a, innov_model="tangent")
    assert torch.equal(B.innovation_nll(st, 10)[0], nll3)                                      # the state's own model
    assert torch.equal(B.innovation_nll(st, 10, model="tangent")[0], nll3)
    assert st.clone().innov_model == "tangent"
    with pytest.raises(ValueError):
        B.innovation_nll(st, 10, model="full")                                                 # contradicts the state
    with pytest.raises(ValueError):
        B.innovation_nll(a, 10, model="3d")
    full = B.ReplayState(torch.zeros(4, 2), torch.zeros(10, 2), innov=a)                      # sums of f5: "full"
    with pytest.raises(ValueError):
        B.innovation_nll(full, 10, model="tangent")


def test_host_api_refuses_a_contradicting_accumulator():
    import torch
    from poseestimationkf_b200 import batched as B
    st = B.ReplayState(torch.zeros(4, 2), torch.zeros(10, 2), innov=torch.zeros(2, 2), innov_model="full")
    with pytest.raises(ValueError):
        B._innovation_buffer(st.innov, 2, "cpu", st, "tangent")
    with pytest.raises(ValueError):
        B.replay(torch.zeros(1, 9, 2), torch.zeros(3, 2), torch.zeros(3, 2), dt=0.01, innovation=True, innovation_model="3d")


@pytest.mark.parametrize("sigma,r_star", [(0.01, 1e-4), (0.03, 1e-3)])
def test_tangent_objective_has_an_interior_minimum_in_r(sigma, r_star):
    """The float64 definition over q = 1e-7..1e1, r = 1e-8..1e1 (one value per decade), 8 trajectories x 300 steps: the
    argmin is interior on both axes, the mean NIS there is that of a consistent 3-DOF model (about 3), and r* follows
    the sensor noise (tripling sigma moves it up one decade)."""
    T, Ns = 300, 8
    imu = make_imu(Ns, T, seed=3, sigma=sigma)
    S = imu.streams.numpy().astype(np.float64)
    qs, rs = 10.0 ** np.arange(-7, 2), 10.0 ** np.arange(-8, 2)
    G = qs.size * rs.size
    q = np.repeat(qs, rs.size * Ns)
    r = np.tile(np.repeat(rs, Ns), qs.size)
    d = TR.replay_tangent(np.full(T, float(np.float32(imu.dt)) * 1e9), np.tile(S[:, 0:3], G), np.tile(S[:, 3:6], G),
                          np.tile(S[:, 6:9], G), np.tile(imu.acc_ref.numpy().T, (G, 1)), np.tile(imu.mag_ref.numpy().T, (G, 1)),
                          q, r)
    nll = TR.nll(d["nis"].sum(0), d["logdet"].sum(0), T).reshape(qs.size, rs.size, Ns).mean(2) / T
    nis = d["nis"].mean(0).reshape(qs.size, rs.size, Ns).mean(2)
    iq, ir = np.unravel_index(int(nll.argmin()), nll.shape)
    assert 0 < iq < qs.size - 1 and 0 < ir < rs.size - 1, (qs[iq], rs[ir])
    assert 2.0 <= nis[iq, ir] <= 4.0, nis[iq, ir]
    assert rs[ir] == pytest.approx(r_star), (qs[iq], rs[ir])
