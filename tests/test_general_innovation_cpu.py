"""Innovation terms and the gate with general Q and R matrices (GEN with INNOV / GATE in ekf_math.cuh) without a GPU:
the float64 definition (tests/general_innovation_ref.py) pinned to the general recursion and to the isotropic
definitions, the CPU build of the header (tests/hostsim/general_innovation.cpp) against the definition, its float32
sums against its own per-step terms, the argument rules of posekf_replay_general_innovation_f32 and the host rules of
replay_general, build_matrix_sweep and make_imu(gyro_sigma=...)."""
import numpy as np
import pytest
import torch

from poseestimationkf_b200 import _lib
from poseestimationkf_b200 import batched as B
from poseestimationkf_b200 import workloads as WL
from poseestimationkf_b200.synth import make_imu
from tests import gating_ref as GT
from tests import general_innovation_ref as GI
from tests import general_qr_ref as GR
from tests import innovation_ref as IR
from tests import innovation_tangent_ref as TR
from tests.hostsim import general_innovation as HI

KINDS = ("full", "diag", "q_over_r_1e4", "r_over_q_100")


def _f32(M):
    """The float32 values of a [N,k,k] matrix stack, as the kernels see them (upper triangle mirrored)."""
    U = np.triu(np.asarray(M, dtype=np.float64)).astype(np.float32).astype(np.float64)
    return U + np.triu(U, 1).transpose(0, 2, 1)


def _matrices(kind, N, seed=0):
    """(Q, R) [N,3,3], [N,4,4]: full (random eigenvectors), diagonal, and the edges of the plain range."""
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
    return imu, imu.streams.numpy(), imu.acc_ref.numpy(), imu.mag_ref.numpy()


def _definition(imu, S, ar, mr, Q, R, **kw):
    Sd = S.astype(np.float64)
    T = S.shape[0]
    return GI.replay(np.full(T, float(np.float32(imu.dt)) * 1e9), Sd[:, 0:3], Sd[:, 3:6], Sd[:, 6:9],
                     ar.T.astype(np.float64), mr.T.astype(np.float64), Q, R, **kw)


def test_definition_at_infinity_is_the_oracle_kalman_filter():
    imu, S, ar, mr = _data(3, 200)
    Q, R = (_f32(M) for M in _matrices("full", 3))
    ref = _definition(imu, S, ar, mr, Q, R)
    assert not ref["gated"].any()
    Sd = S.astype(np.float64)
    for n in range(3):
        kf = GR.replay_kf(np.full(200, float(np.float32(imu.dt)) * 1e9), Sd[:, 0:3, n], Sd[:, 3:6, n], Sd[:, 6:9, n],
                          ar[:, n].astype(np.float64), mr[:, n].astype(np.float64), Q[n], R[n])
        assert np.abs(kf["X"] - ref["X"][:, n]).max() < 1e-12
        assert np.array_equal(kf["flips"], ref["flips"][:, n])


def test_definition_with_isotropic_matrices_is_the_isotropic_definitions():
    imu, S, ar, mr = _data(4, 150)
    Sd = S.astype(np.float64)
    q, r = np.array([1e-3, 1e-2, 1e-1, 1.0]), np.array([1e-2, 1e-1, 1e-2, 1e-3])
    Q, R = q[:, None, None] * np.eye(3), r[:, None, None] * np.eye(4)
    args = (np.full(150, float(np.float32(imu.dt)) * 1e9), Sd[:, 0:3], Sd[:, 3:6], Sd[:, 6:9], ar.T.astype(np.float64),
            mr.T.astype(np.float64))
    ref = GI.replay(*args, Q, R)
    full = IR.replay_innovation(*args, q, r)
    tan = TR.replay_tangent(*args, q, r)
    scale = np.abs(ref["nis4"]) + np.abs(ref["logdet4"])
    assert (np.abs(ref["nis4"] - full["nis"]) / scale).max() < 1e-12
    assert (np.abs(ref["logdet4"] - full["logdet"]) / scale).max() < 1e-12
    scale3 = np.abs(ref["nis3"]) + np.abs(ref["logdet3"])
    assert (np.abs(ref["nis3"] - tan["nis"]) / scale3).max() < 1e-12
    assert (np.abs(ref["logdet3"] - tan["logdet"]) / scale3).max() < 1e-12
    # the gated recursion: the same decisions and states as the isotropic gate's definition
    gamma = float(np.quantile(ref["nis3"], 0.8))
    gd = GI.replay(*args, Q, R, gamma=gamma)
    gi = GT.replay_gated(*args, q, r, gamma=gamma)
    assert gd["gated"].any() and np.array_equal(gd["gated"], gi["gated"])
    assert np.abs(gd["X"] - gi["X"]).max() < 1e-12
    assert (np.abs(gd["nis3"] - gi["nis"]) / (np.abs(gi["nis"]) + np.abs(gi["logdet"]))).max() < 1e-12


def _gamma(imu, S, ar, mr, Q, R):
    """A threshold that gates about a fifth of the steps of the ungated definition."""
    return float(np.quantile(_definition(imu, S, ar, mr, Q, R)["nis3"], 0.8))


def _rel(got, nis, ld):
    """|got - definition| relative to |NIS_t| + |ln det S_t| of the step."""
    return np.abs(got[0] - nis) / (np.abs(nis) + np.abs(ld)), np.abs(got[1] - ld) / (np.abs(nis) + np.abs(ld))


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("model", ["full", "tangent"])
@pytest.mark.parametrize("gated", [False, True])
def test_hostsim_f64_terms_match_definition(kind, model, gated):
    imu, S, ar, mr = _data(6, 200)
    Q, R = (_f32(M) for M in _matrices(kind, 6))
    gamma = _gamma(imu, S, ar, mr, Q, R) if gated else None
    h = HI.replay(S, imu.dt, ar, mr, Q, R, model=model, gamma=gamma, precision="f64")
    # the gated definition follows the build's own decisions (a threshold tie cannot send the recursions apart)
    ref = _definition(imu, S, ar, mr, Q, R, decisions=h["gated"] if gated else None)
    if gated:
        assert h["gated"].any() and not h["gated"].all()
        assert np.array_equal(h["gated"], ref["nis3"] > gamma)
    nis, ld = GI.terms(ref, model)
    en, el = _rel(h["terms"], nis, ld)
    assert en.max() < 1e-9 and el.max() < 1e-9, (en.max(), el.max())


@pytest.mark.parametrize("model", ["full", "tangent"])
@pytest.mark.parametrize("gated", [False, True])
@pytest.mark.parametrize("algo", ["qr2", "jacobi"])
def test_hostsim_f32_sums_are_the_running_sums_of_the_terms(model, gated, algo):
    imu, S, ar, mr = _data(8, 300, seed=5)
    Q, R = (_f32(M) for M in _matrices("full", 8, seed=2))
    h = HI.replay(S, imu.dt, ar, mr, Q, R, model=model, gamma=_gamma(imu, S, ar, mr, Q, R) if gated else None, algo=algo)
    terms = h["terms"].astype(np.float32)
    assert np.array_equal(terms.astype(np.float64), h["terms"])
    acc = np.zeros((2, terms.shape[2]), dtype=np.float32)
    for t in range(terms.shape[1]):
        acc = acc + terms[:, t]                          # float32: one rounding per step, as the kernel adds them
    # each sum adds exactly the term written out: both sums are the float32 running sums of the per-step terms
    assert np.array_equal(acc.astype(np.float64), h["innov"])
    # and the float32 terms stay within the f5/f6 bar of the definition
    ref = _definition(imu, S, ar, mr, Q, R, decisions=h["gated"] if gated else None)
    nis, ld = GI.terms(ref, model)
    bar = np.abs(nis.sum(0)) + np.abs(ld.sum(0))
    assert (np.abs(h["innov"][0] - nis.sum(0)) / bar).max() < 1e-4
    assert (np.abs(h["innov"][1] - ld.sum(0)) / bar).max() < 1e-4


def test_hostsim_pivots_at_the_range_edges_do_not_overflow():
    # pivots down to 1e-18 and up to 1e18: the log-determinant is summed from pivot pairs, never the 4-pivot product
    # (the first steps leave P = I far from the scale of R, where the float32 step is outside its plain range: the terms
    # are compared once the filter has settled)
    imu, S, ar, mr = _data(2, 40)
    for scale in (1e-18, 1e18):
        Q = np.broadcast_to(scale * 0.05 * np.eye(3), (2, 3, 3)).copy()
        R = np.broadcast_to(scale * np.diag([1.0, 2.0, 3.0, 4.0]), (2, 4, 4)).copy()
        for model in ("full", "tangent"):
            h = HI.replay(S, imu.dt, ar, mr, _f32(Q), _f32(R), model=model)
            ref = _definition(imu, S, ar, mr, _f32(Q), _f32(R))
            nis, ld = GI.terms(ref, model)
            assert np.isfinite(h["terms"]).all()
            assert (np.abs(h["terms"][1, 20:] - ld[20:]) / np.abs(ld[20:])).max() < 1e-5


def _capi(lib, N=4, T=2, nq=1, nr=1, q_tri=True, r_tri=True, x_lo=False, model=0, gamma=float("inf"), out=True,
          stride=None, out_offset=0):
    M = max(N, 1)
    bufs = {k: np.ones(n, dtype=np.float32) for k, n in dict(s=T * 9 * M, dt=1, ar=3 * M, mr=3 * M, q=6 * max(nq, 1),
                                                             r=10 * max(nr, 1), x=4 * M, xlo=4 * M, p=10 * M,
                                                             o=2 * T * M + 1).items()}
    p = lambda k: bufs[k].ctypes.data
    return lib.posekf_replay_general_innovation_f32(
        N, T, p("s"), N, p("dt"), 0, p("ar"), p("mr"), p("q") if q_tri else None, nq, p("r") if r_tri else None, nr, -1.0,
        -1.0, p("x"), p("xlo") if x_lo else None, p("p"), None, None, None, None, None, None, model, 0, 1, 0, None, None,
        None, gamma, None, None, (p("o") + out_offset) if out else None, T * M if stride is None else stride)


def test_capi_argument_rules():
    lib = _lib.load()
    assert _capi(lib, x_lo=True) == _lib.EINVAL                     # no precise variant
    assert _capi(lib, model=2) == _lib.EINVAL                       # unknown innovation model
    assert _capi(lib, gamma=float("nan")) == _lib.EINVAL            # NaN decides nothing
    assert _capi(lib, nq=2) == _lib.EINVAL                          # nq / nr are 1 or N
    assert _capi(lib, nr=3) == _lib.EINVAL
    assert _capi(lib, nq=0) == _lib.EINVAL
    assert _capi(lib, q_tri=False) == _lib.EINVAL
    assert _capi(lib, r_tri=False) == _lib.EINVAL
    assert _capi(lib, N=-1) == _lib.EINVAL
    assert _capi(lib, stride=7) == _lib.EINVAL                      # plane stride < T N
    assert _capi(lib, out_offset=2) == _lib.EALIGN                  # out_innov 4-byte aligned
    assert _capi(lib, N=0, out=False) == 0                          # an empty launch


def test_existing_entry_points_keep_refusing():
    lib = _lib.load()
    N, T = 4, 2
    bufs = {k: np.ones(n, dtype=np.float32) for k, n in dict(s=T * 9 * N, dt=1, ar=3 * N, mr=3 * N, q=6, r=10, x=4 * N,
                                                             p=10 * N, acc=2 * N).items()}
    p = lambda k: bufs[k].ctypes.data
    rc = lib.posekf_replay_general_f32(N, T, p("s"), N, p("dt"), 0, p("ar"), p("mr"), p("q"), 1, p("r"), 1, -1.0, -1.0,
                                       p("x"), None, p("p"), None, None, None, None, None, p("acc"), 0, 0, 1, 0, None, None,
                                       None)
    assert rc == _lib.EINVAL                                        # still no innovation sums there


def test_replay_general_refuses_scalars():
    imu = make_imu(4, 3, seed=1)
    for q, r in ((1.0, 0.1), (torch.ones(4), 0.1), (1.0, torch.full((4,), 0.1))):
        with pytest.raises(ValueError, match="use replay"):
            B.replay_general(imu.streams, imu.acc_ref, imu.mag_ref, dt=imu.dt, q=q, r=r, innovation=True)


class _Batch:
    def __init__(self, Ns, T):
        imu = make_imu(Ns, T, seed=2)
        self.streams, self.acc_ref, self.mag_ref, self.dt = imu.streams, imu.acc_ref, imu.mag_ref, imu.dt
        self.lengths = torch.full((Ns,), T, dtype=torch.int32)


def test_build_matrix_sweep_shapes():
    b = _Batch(4, 5)
    Qs = np.stack([np.diag([a, a, 3 * a]) for a in (1e-3, 1e-2, 1e-1)])
    w = WL.build_matrix_sweep(b, Qs, np.eye(4) * 0.1)
    assert w.n_candidates == 3 and w.n_filters == 12
    assert w.q.shape == (12, 3, 3) and w.r.shape == (4, 4)
    assert torch.equal(w.q[4 * 2 + 1], torch.as_tensor(Qs[2]))       # candidate n // Ns
    w = WL.build_matrix_sweep(b, np.eye(3) * 1e-2, np.stack([np.eye(4) * v for v in (0.1, 0.2)]))
    assert w.n_candidates == 2 and w.q.shape == (3, 3) and w.r.shape == (8, 4, 4)
    w = WL.build_matrix_sweep(b, Qs, np.stack([np.eye(4) * v for v in (0.1, 0.2, 0.3)]))
    assert w.q.shape == (12, 3, 3) and w.r.shape == (12, 4, 4)
    with pytest.raises(ValueError, match="agree"):
        WL.build_matrix_sweep(b, Qs, np.stack([np.eye(4)] * 2))
    with pytest.raises(ValueError, match=r"\[M,3,3\]"):
        WL.build_matrix_sweep(b, np.eye(4), np.eye(4))


def test_make_imu_default_draws_are_unchanged():
    # gyro_sigma=None is the old code path itself; an isotropic gyro_sigma equal to sigma draws the same numbers in the
    # same order, and an anisotropic one changes the gyro rows only
    base = make_imu(4, 16, seed=5, sigma=0.01, keep_truth=True)
    none = make_imu(4, 16, seed=5, sigma=0.01, keep_truth=True, gyro_sigma=None)
    iso = make_imu(4, 16, seed=5, sigma=0.01, keep_truth=True, gyro_sigma=(0.01, 0.01, 0.01))
    aniso = make_imu(4, 16, seed=5, sigma=0.01, keep_truth=True, gyro_sigma=(0.01, 0.01, 0.1))
    for other in (none, iso):
        assert torch.equal(base.streams, other.streams) and torch.equal(base.q_true, other.q_true)
        assert torch.equal(base.acc_ref, other.acc_ref) and torch.equal(base.mag_ref, other.mag_ref)
    assert torch.equal(base.streams[:, 3:], aniso.streams[:, 3:]) and torch.equal(base.streams[:, :2], aniso.streams[:, :2])
    dz = (aniso.streams[:, 2] - base.streams[:, 2]).double()
    assert torch.allclose(dz, 9.0 * (base.streams[:, 2].double() - _noiseless_gyro_z()), atol=1e-5)


def _noiseless_gyro_z():
    # the gyro z row without noise: the same motion model with sigma = 0 draws the motion first and no noise
    return make_imu(4, 16, seed=5, sigma=0.0).streams[:, 2].double()
