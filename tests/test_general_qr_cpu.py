"""General Q and R matrices (GEN in ekf_math.cuh) without a GPU: the float64 definition (tests/general_qr_ref.py) against
the oracle's own KalmanFilter, the CPU build of the header (tests/hostsim/general_qr.cpp) in float64 and float32 against
the definition, Q = qI / R = rI through the general step against the isotropic step, and the argument rules of
posekf_replay_general_f32 and of replay(q=<matrix>, r=<matrix>)."""
import numpy as np
import pytest
import torch

from oracle import ekf_oracle as O
from poseestimationkf_b200 import _lib
from poseestimationkf_b200 import batched as B
from poseestimationkf_b200.synth import make_imu
from tests import general_qr_ref as GR
from tests.hostsim import general_qr as HQ


def _f32(M):
    """The float32 values of a [N,k,k] matrix stack, as the kernels see them (upper triangle mirrored)."""
    U = np.triu(np.asarray(M, dtype=np.float64)).astype(np.float32).astype(np.float64)
    return U + np.triu(U, 1).transpose(0, 2, 1)


def _matrices(kind, N, seed=0):
    """(Q, R) [N,3,3], [N,4,4]: full (random eigenvectors), diagonal, and eigenvalue ratios inside the plain range."""
    rng = np.random.default_rng(seed)
    if kind == "full":
        return GR.random_spd(rng, N, 3, 1e-4, 1e-2), GR.random_spd(rng, N, 4, 1e-3, 1e-1)
    if kind == "diag":
        return (np.einsum("nk,kj->nkj", np.exp(rng.uniform(np.log(1e-4), np.log(1e-2), (N, 3))), np.eye(3)),
                np.einsum("nk,kj->nkj", np.exp(rng.uniform(np.log(1e-3), np.log(1e-1), (N, 4))), np.eye(4)))
    if kind == "q_over_r_1e4":
        return GR.random_spd(rng, N, 3, 1e-1, 1e0), GR.random_spd(rng, N, 4, 1e-5, 1e-4)
    if kind == "r_over_q_100":
        return GR.random_spd(rng, N, 3, 1e-3, 1e-2), GR.random_spd(rng, N, 4, 1e-1, 1e0)
    raise ValueError(kind)


def _data(N, T, seed=3):
    imu = make_imu(N, T, seed=seed, sigma=0.01)
    S = imu.streams.numpy()
    return imu, S, imu.acc_ref.numpy(), imu.mag_ref.numpy()


def _definition(imu, S, ar, mr, Q, R):
    Sd = S.astype(np.float64)
    T = S.shape[0]
    return GR.replay_general(np.full(T, float(np.float32(imu.dt)) * 1e9), Sd[:, 0:3], Sd[:, 3:6], Sd[:, 6:9],
                             ar.T.astype(np.float64), mr.T.astype(np.float64), _f32(Q), _f32(R))


def test_definition_is_the_oracle_kalman_filter():
    imu, S, ar, mr = _data(3, 200)
    Q, R = _matrices("full", 3)
    ref = _definition(imu, S, ar, mr, Q, R)
    Sd = S.astype(np.float64)
    for n in range(3):
        kf = GR.replay_kf(np.full(200, float(np.float32(imu.dt)) * 1e9), Sd[:, 0:3, n], Sd[:, 3:6, n], Sd[:, 6:9, n],
                          ar[:, n].astype(np.float64), mr[:, n].astype(np.float64), _f32(Q)[n], _f32(R)[n])
        assert np.abs(kf["X"] - ref["X"][:, n]).max() < 1e-12
        assert np.array_equal(kf["flips"], ref["flips"][:, n])
        assert np.abs(kf["P"] - ref["P"][n]).max() < 1e-12


@pytest.mark.parametrize("kind", ["full", "diag", "q_over_r_1e4", "r_over_q_100"])
@pytest.mark.parametrize("algo", ["qr2", "jacobi"])
def test_float64_build_matches_definition(kind, algo):
    imu, S, ar, mr = _data(8, 400)
    Q, R = _matrices(kind, 8)
    ref = _definition(imu, S, ar, mr, Q, R)
    out = HQ.replay(S, imu.dt, ar, mr, _f32(Q), _f32(R), precision="f64", algo=algo)
    assert O.quat_angle(out["traj"], ref["X"]).max() < 1e-9
    assert np.array_equal(out["flips"], ref["flips"])
    assert np.abs(out["p"] - HQ.tri(ref["P"], HQ.TRI4)).max() < 1e-9 * np.abs(ref["P"]).max()


@pytest.mark.parametrize("kind", ["full", "diag", "q_over_r_1e4", "r_over_q_100"])
@pytest.mark.parametrize("algo", ["qr2", "jacobi"])
def test_float32_build_matches_definition(kind, algo):
    imu, S, ar, mr = _data(16, 1000)
    Q, R = _matrices(kind, 16)
    ref = _definition(imu, S, ar, mr, Q, R)
    out = HQ.replay(S, imu.dt, ar, mr, Q, R, precision="f32", algo=algo)
    assert O.quat_angle(out["traj"], ref["X"]).max() < 1e-5
    assert np.array_equal(out["flips"], ref["flips"])


def test_precomputed_measurements_match_definition():
    imu, S, ar, mr = _data(8, 400)
    Q, R = _matrices("full", 8)
    ref = _definition(imu, S, ar, mr, Q, R)
    # a measurement stream: rows 3-6 hold the reference-signed float32 Wahba quaternion of the definition's own solver
    Sd = S.astype(np.float64)
    ys = np.stack([O.wahba_batched(ar.T.astype(np.float64), mr.T.astype(np.float64), Sd[t, 3:6].T, Sd[t, 6:9].T,
                                   np.abs(Sd[t, 5]), 1 - np.abs(Sd[t, 5])) for t in range(S.shape[0])])     # [T,N,4]
    M = S.copy()
    M[:, 3:7] = ys.transpose(0, 2, 1).astype(np.float32)
    M[:, 7:9] = 0
    out = HQ.replay(M, imu.dt, ar, mr, Q, R, precision="f32", algo="precomputed")
    assert O.quat_angle(out["traj"], ref["X"]).max() < 1e-5
    assert np.array_equal(out["flips"], ref["flips"])


@pytest.mark.parametrize("q,r", [(1.0, 0.1), (1e-3, 1e-2), (1e-2, 1e-5), (1e-3, 3e-2)])
def test_isotropic_matrices_match_the_isotropic_step(q, r):
    imu, S, ar, mr = _data(8, 1000)
    N = S.shape[2]
    gen = HQ.replay(S, imu.dt, ar, mr, np.tile(q * np.eye(3), (N, 1, 1)), np.tile(r * np.eye(4), (N, 1, 1)), precision="f32")
    iso = HQ.replay(S, imu.dt, ar, mr, np.full(N, q), np.full(N, r), precision="f32", isotropic=True)
    assert O.quat_angle(gen["traj"], iso["traj"]).max() < 1e-6
    assert np.array_equal(gen["flips"], iso["flips"])


# ---- argument rules ----------------------------------------------------------------------------------------------------
def _general(lib, N=4, T=2, nq=1, nr=1, q_tri=True, r_tri=True, x_lo=False, innov=False, model=0):
    M = max(N, 1)
    bufs = {k: np.ones(n, dtype=np.float32) for k, n in dict(s=T * 9 * M, dt=1, ar=3 * M, mr=3 * M, q=6 * max(nq, 1),
                                                             r=10 * max(nr, 1), x=4 * M, xlo=4 * M, p=10 * M, acc=2 * M).items()}
    p = lambda k: bufs[k].ctypes.data
    return lib.posekf_replay_general_f32(N, T, p("s"), N, p("dt"), 0, p("ar"), p("mr"), p("q") if q_tri else None, nq,
                                         p("r") if r_tri else None, nr, -1.0, -1.0, p("x"), p("xlo") if x_lo else None, p("p"),
                                         None, None, None, None, None, p("acc") if innov else None, model, 0, 1, 0, None,
                                         None, None)


def test_capi_argument_rules():
    lib = _lib.load()
    assert _general(lib, x_lo=True) == _lib.EINVAL                 # no precise variant
    assert _general(lib, innov=True) == _lib.EINVAL                # no innovation sums
    assert _general(lib, model=2) == _lib.EINVAL                   # unknown innovation model
    assert _general(lib, nq=2) == _lib.EINVAL                      # nq is 1 or N
    assert _general(lib, nr=3) == _lib.EINVAL
    assert _general(lib, nq=0) == _lib.EINVAL
    assert _general(lib, q_tri=False) == _lib.EINVAL
    assert _general(lib, r_tri=False) == _lib.EINVAL
    assert _general(lib, N=-1) == _lib.EINVAL


def test_matrix_checks():
    rng = np.random.default_rng(1)
    Q, R = _matrices("full", 5)
    q_tri, r_tri = B.general_qr_tri(Q, R, 5, "cpu")
    assert q_tri.shape == (6, 5) and r_tri.shape == (10, 5) and q_tri.dtype == torch.float32
    assert np.array_equal(r_tri.numpy(), HQ.tri(R, HQ.TRI4).astype(np.float32))
    q_tri, r_tri = B.general_qr_tri(Q[0], 0.1, 5, "cpu")          # one shared Q, R = 0.1 I
    assert q_tri.shape == (6, 1) and r_tri.shape == (10, 1)
    assert np.array_equal(r_tri[:, 0].numpy(), np.float32([0.1, 0, 0, 0, 0.1, 0, 0, 0.1, 0, 0.1]))
    q_tri, _ = B.general_qr_tri(np.diag([0.0, 1.0, 2.0]), R, 5, "cpu")     # positive semidefinite Q
    assert q_tri.shape == (6, 1)
    with pytest.raises(ValueError, match="positive definite"):
        B.general_qr_tri(Q, np.diag([1.0, 1.0, 1.0, 0.0]), 5, "cpu")
    with pytest.raises(ValueError, match="positive definite"):
        B.general_qr_tri(Q, np.diag([1.0, 1.0, 1.0, -1e-3]), 5, "cpu")
    with pytest.raises(ValueError, match="semidefinite"):
        B.general_qr_tri(np.diag([1.0, 1.0, -1e-3]), R, 5, "cpu")
    A = rng.standard_normal((4, 4))
    with pytest.raises(ValueError, match="symmetric"):
        B.general_qr_tri(Q, A @ A.T + np.triu(np.ones((4, 4)), 1), 5, "cpu")
    with pytest.raises(ValueError, match="matrix"):
        B.general_qr_tri(Q[:4], R, 5, "cpu")                       # [N',3,3] with N' != N
    with pytest.raises(ValueError, match="matrix"):
        B.general_qr_tri(np.eye(4), R, 5, "cpu")
    with pytest.raises(ValueError, match="matrix"):
        B.general_qr_tri(Q, np.ones((5, 3, 3)), 5, "cpu")
