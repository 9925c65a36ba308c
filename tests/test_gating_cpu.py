"""Innovation gate (GATE in ekf_math.cuh) without a GPU: the CPU build of the header (tests/hostsim/gating.cpp) against
the float64 definition (tests/gating_ref.py), float32 against the packed lanes, the gate at +inf against the ungated
build, and the argument rules of posekf_replay_gated_f32 and of replay(gate=...)."""
import math

import numpy as np
import pytest
import torch

from poseestimationkf_b200 import _lib
from poseestimationkf_b200 import batched as B
from poseestimationkf_b200.synth import add_disturbances, make_imu
from tests import gating_ref as GR
from tests.hostsim import gating as HG

GAMMA = B.GATE_CHI2_3_999


def _disturbed(N, T, seed=5, sigma=0.01):
    imu = make_imu(N, T, seed=seed, sigma=sigma, dt=0.01)
    mask = add_disturbances(imu.streams, seed=1, n_mag=1, n_acc=1, length=(40, 80), margin=(60, 100))
    return imu, mask.numpy()


def _ref(imu, q, r, gamma, decisions=None):
    S = imu.streams.numpy().astype(np.float64)
    T = S.shape[0]
    return GR.replay_gated(np.full(T, float(np.float32(imu.dt)) * 1e9), S[:, 0:3], S[:, 3:6], S[:, 6:9],
                           imu.acc_ref.numpy().T.astype(np.float64), imu.mag_ref.numpy().T.astype(np.float64),
                           float(np.float32(q)), float(np.float32(r)), gamma, decisions)


def _host(imu, q, r, **kw):
    return HG.replay(imu.streams.numpy(), imu.dt, imu.acc_ref.numpy(), imu.mag_ref.numpy(), q, r, **kw)


# (q, r) of the plain variant's range (the tangent argmin of sigma = 0.01 data) and of both precise extremes
TUNINGS = [(False, 7.9e-6, 1e-4), (True, 1e-3, 1e3), (True, 1e3, 1e-3), (False, 1.0, 0.1)]


@pytest.mark.parametrize("comp,q,r", TUNINGS)
def test_float64_build_matches_definition(comp, q, r):
    imu, mask = _disturbed(6, 400)
    got = _host(imu, q, r, gamma=GAMMA, precision="f64", compensated=comp)
    free = _ref(imu, q, r, GAMMA)
    # decisions: the same except at threshold ties
    tie = np.abs(free["nis"] / GAMMA - 1.0) < 1e-9
    assert not np.any((got["gated"] != free["gated"]) & ~tie)
    ref = _ref(imu, q, r, GAMMA, decisions=got["gated"])
    # at q/r = 1e6 the definition's own K = P (P + R)^-1 and P - K P lose float64 digits (1.4e-8 rad and 1e-6 apart
    # without the gate too): there the bars are the distances of the ungated build from the ungated definition
    free_b, free_r = _host(imu, q, r, gate=False, precision="f64", compensated=comp), _ref(imu, q, r, math.inf)
    ang = GR.angle(got["traj"], ref["X"])
    bar = max(1e-9, 1.01 * GR.angle(free_b["traj"], free_r["X"]).max())
    assert ang.max() <= bar, (ang.max(), bar)

    def p_err(p, Pdef):
        Pd = B.tri_from_full(torch.from_numpy(Pdef)).numpy()
        return (np.linalg.norm(p * np.float32(r) - Pd, axis=0) / np.linalg.norm(Pd, axis=0)).max()
    rel, bar_p = p_err(got["p"], ref["P"]), max(1e-9, 10 * p_err(free_b["p"], free_r["P"]))
    assert rel <= bar_p, (rel, bar_p)
    if q == 7.9e-6:
        assert got["gated"][mask].mean() > 0.5 and got["gated"].any()


@pytest.mark.parametrize("comp,q,r", TUNINGS)
@pytest.mark.parametrize("model", [None, "full", "tangent"])
def test_float32_equals_packed_lanes(comp, q, r, model):
    imu, _ = _disturbed(8, 300, seed=7)
    a = _host(imu, q, r, gamma=GAMMA, precision="f32", compensated=comp, innov_model=model)
    b = _host(imu, q, r, gamma=GAMMA, precision="f32x2", compensated=comp, innov_model=model)
    for k in a:
        assert np.array_equal(a[k], b[k], equal_nan=True), k


@pytest.mark.parametrize("comp,q,r", TUNINGS)
@pytest.mark.parametrize("model", [None, "full", "tangent"])
@pytest.mark.parametrize("precision,algo", [("f32", "qr2"), ("f32", "jacobi"), ("f32x2", "qr2")])
def test_gate_at_infinity_is_the_ungated_build(comp, q, r, model, precision, algo):
    imu, _ = _disturbed(8, 300, seed=9)
    a = _host(imu, q, r, gamma=math.inf, precision=precision, algo=algo, compensated=comp, innov_model=model)
    b = _host(imu, q, r, gate=False, precision=precision, algo=algo, compensated=comp, innov_model=model)
    assert not a["gated"].any()
    for k in a:
        assert np.array_equal(a[k], b[k], equal_nan=True), k


def test_gate_at_zero_is_pure_prediction():
    imu, _ = _disturbed(4, 200)
    q, r = 1e-3, 1e-2
    got = _host(imu, q, r, gamma=0.0, precision="f64")
    assert got["gated"].all()
    ref = _ref(imu, q, r, 0.0)
    assert ref["gated"].all()
    assert GR.angle(got["traj"], ref["X"]).max() <= 1e-9


def test_nan_statistic_is_not_gated():
    imu, _ = _disturbed(4, 200)
    imu.streams[50, 6:9, 1] = float("nan")
    got = _host(imu, 1e-3, 1e-2, gamma=GAMMA, precision="f32")
    assert not got["gated"][50, 1]
    assert np.isnan(got["traj"][50:, 1]).all()          # NaN propagates as in the reference
    assert np.isfinite(got["traj"][:, 0]).all()


def test_gated_covariance_keeps_its_small_diagonal():
    """P^- of a gated step is formed with its own diagonal constant, not as S - I: at P^-/r ~ 2.5e-3 (the lower edge of
    the plain variant) the float32 P after a run of gated steps stays within 1e-5 relative of float64."""
    imu, _ = _disturbed(4, 300)
    q, r = 1e-3, 0.099      # r/q just inside the plain variant's range
    f32 = _host(imu, q, r, gamma=0.0, precision="f32")
    f64 = _host(imu, q, r, gamma=0.0, precision="f64")
    rel = np.linalg.norm(f32["p"] - f64["p"], axis=0) / np.linalg.norm(f64["p"], axis=0)
    assert rel.max() <= 1e-5, rel.max()


# ---- argument rules -------------------------------------------------------------------------------------------------
def _gated(lib, N=8, T=4, gate=16.0, gate_count=None, **over):
    args = dict(n_filters=N, n_steps=T, streams=None, n_streams=N, dt=None, dt_per_step=0, acc_ref=None, mag_ref=None,
                q=None, r=None, a=-1.0, m=-1.0, x=None, xlo=None, p=None, lpf=None, traj=None, flip=None, truth=None,
                loss=None, innov=None, model=0, algo=0, staging=0, flags=0, stream=None, dt_cols=None, n_valid=None)
    args.update(over)
    return lib.posekf_replay_gated_f32(*args.values(), gate, gate_count, None)


def test_capi_argument_rules():
    lib = _lib.load()
    assert _gated(lib, gate=float("nan")) == _lib.EINVAL
    assert _gated(lib, N=0, gate=float("nan")) == _lib.EINVAL        # the threshold is checked first
    assert _gated(lib, N=0, gate=float("inf")) == 0                  # empty batch: a no-op
    assert _gated(lib, model=2) == _lib.EINVAL                       # unknown innovation model
    assert _gated(lib) == _lib.EINVAL                                # null buffers
    assert _gated(lib, N=-1) == _lib.EINVAL


def test_replay_argument_rules():
    s = torch.zeros((4, 9, 8))
    ref = torch.zeros((3, 8))
    with pytest.raises(ValueError, match="need gate"):
        B.replay(s, ref, ref, dt=0.01, gate_count=torch.zeros(8, dtype=torch.int32))
    with pytest.raises(ValueError, match="need gate"):
        B.replay(s, ref, ref, dt=0.01, out_gated=torch.zeros((4, 8), dtype=torch.uint8))
    with pytest.raises(ValueError, match="NaN"):
        B.replay(s, ref, ref, dt=0.01, gate=float("nan"))
    with pytest.raises(ValueError, match="gate_count"):
        B._gate_buffers(torch.zeros(8, dtype=torch.float32), None, 8, 4, "cpu")
    with pytest.raises(ValueError, match="out_gated"):
        B._gate_buffers(None, torch.zeros((4, 7), dtype=torch.uint8), 8, 4, "cpu")
    with pytest.raises(_lib.PosekfError):
        B._gate_buffers(torch.zeros(8, dtype=torch.int32), None, 8, 4, "cpu")


def test_disturbances_are_reproducible_and_unit():
    a = make_imu(6, 700, seed=3, sigma=0.01).streams
    b = a.clone()
    ma = add_disturbances(a, seed=4, n_mag=3, n_acc=2)
    mb = add_disturbances(b, seed=4, n_mag=3, n_acc=2)
    assert torch.equal(a, b) and torch.equal(ma, mb)
    assert ma.any() and not ma[:200].any()
    assert (a[:, 3:9].reshape(700, 2, 3, 6).norm(dim=2) - 1).abs().max() < 1e-6
    assert torch.equal(make_imu(6, 700, seed=3, sigma=0.01).streams[~ma.any(1)], a[~ma.any(1)])
