"""Per-step innovation output without a GPU: the CPU build of the header (tests/hostsim/innovation_steps.cpp) against
the float64 definitions (tests/innovation_ref.py, tests/innovation_tangent_ref.py, tests/gating_ref.py), float32
against the packed lanes, the per-step terms against the sums of the same build, the argument rules of
posekf_replay_innovation_steps_f32 and the host checks of replay(out_innovation=...) and window_innovation_nll."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from poseestimationkf_b200 import _lib
from poseestimationkf_b200 import batched as B
from poseestimationkf_b200 import workloads as W
from poseestimationkf_b200.synth import add_disturbances, make_imu
from tests import gating_ref as GR
from tests import innovation_ref as IR
from tests import innovation_tangent_ref as TR
from tests.hostsim import innovation_steps as HS

GAMMA = B.GATE_CHI2_3_999
# (q, r) of the plain variant's range and of both precise extremes
TUNINGS = [(False, 1.0, 0.1), (False, 7.9e-6, 1e-4), (True, 1e-3, 1e3), (True, 1e3, 1e-3)]


def _imu(N, T, seed, disturbed=False):
    imu = make_imu(N, T, seed=seed, sigma=0.01, dt=0.01)
    if disturbed:
        add_disturbances(imu.streams, seed=1, n_mag=1, n_acc=1, length=(40, 80), margin=(60, 100))
    return imu


def _ref_args(imu):
    S = imu.streams.numpy().astype(np.float64)
    T = S.shape[0]
    return (np.full(T, float(np.float32(imu.dt)) * 1e9), S[:, 0:3], S[:, 3:6], S[:, 6:9],
            imu.acc_ref.numpy().T.astype(np.float64), imu.mag_ref.numpy().T.astype(np.float64))


def _host(imu, q, r, **kw):
    return HS.replay(imu.streams.numpy(), imu.dt, imu.acc_ref.numpy(), imu.mag_ref.numpy(), q, r, **kw)


@pytest.mark.parametrize("comp,q,r", TUNINGS)
@pytest.mark.parametrize("model", ["full", "tangent"])
def test_float64_terms_match_definition(comp, q, r, model):
    imu = _imu(4, 150, seed=3)
    got = _host(imu, q, r, model=model, precision="f64", compensated=comp)
    fn = IR.replay_innovation if model == "full" else TR.replay_tangent
    ref = fn(*_ref_args(imu), float(np.float32(q)), float(np.float32(r)))
    nis, ld = got["terms"]
    # per step, relative to |NIS_t| + |ln det S_t| (the terms a sum of them adds).  At Q >> R (q/r = 1e6) the
    # definition's own K = P (P + R)^-1, P - K P and e = y - z lose float64 digits (see test_innovation_cpu.py): the bar
    # there is that of the sums
    bar = 2e-7 if q / r > 1e4 else 1e-9
    scale = np.abs(ref["nis"]) + np.abs(ref["logdet"])
    assert (np.abs(ld - ref["logdet"]) / scale).max() < bar
    assert (np.abs(nis - ref["nis"]) / scale).max() < bar


@pytest.mark.parametrize("comp,q,r", TUNINGS[:2])
def test_float64_gated_terms_match_definition(comp, q, r):
    imu = _imu(4, 300, seed=5, disturbed=True)
    got = _host(imu, q, r, model="tangent", gamma=GAMMA, precision="f64", compensated=comp)
    ref = GR.replay_gated(*_ref_args(imu), float(np.float32(q)), float(np.float32(r)), GAMMA, decisions=got["gated"])
    nis, ld = got["terms"]
    scale = np.abs(ref["nis"]) + np.abs(ref["logdet"])
    assert (np.abs(nis - ref["nis"]) / scale).max() < 1e-9
    assert (np.abs(ld - ref["logdet"]) / scale).max() < 1e-9
    # the gate thresholded plane 0: decisions equal nis > gamma except at ties
    tie = np.abs(nis / GAMMA - 1.0) < 1e-9
    assert not np.any((got["gated"] != (nis > GAMMA)) & ~tie)
    if q == 7.9e-6:
        assert got["gated"].any()


@pytest.mark.parametrize("comp,q,r", TUNINGS)
@pytest.mark.parametrize("model", ["full", "tangent"])
@pytest.mark.parametrize("gamma", [None, GAMMA])
def test_float32_terms_equal_packed_lanes(comp, q, r, model, gamma):
    imu = _imu(4, 250, seed=7, disturbed=True)
    a = _host(imu, q, r, model=model, gamma=gamma, precision="f32", compensated=comp)
    b = _host(imu, q, r, model=model, gamma=gamma, precision="f32x2", compensated=comp)
    for k in a:
        assert np.array_equal(a[k], b[k], equal_nan=True), k


@pytest.mark.parametrize("comp,q,r", TUNINGS)
@pytest.mark.parametrize("model", ["full", "tangent"])
@pytest.mark.parametrize("algo", ["qr2", "jacobi"])
def test_float32_running_sum_of_terms_is_the_sum(comp, q, r, model, algo):
    imu = _imu(4, 300, seed=11)
    got = _host(imu, q, r, model=model, precision="f32", compensated=comp, algo=algo)
    terms = got["terms"].astype(np.float32)
    # ln det S_t is the addend of the sum itself: its float32 running sum is the build's sum bit for bit
    ld = np.zeros(terms.shape[2], dtype=np.float32)
    for t in range(terms.shape[1]):
        ld = ld + terms[1, t]
    assert np.array_equal(ld, got["innov"][1].astype(np.float32))
    # NIS_t is the product the sum's fused multiply-add adds: one float32 rounding per step apart
    nis = np.zeros(terms.shape[2], dtype=np.float32)
    bound = np.zeros(terms.shape[2])
    for t in range(terms.shape[1]):
        nis = nis + terms[0, t]
        bound += np.spacing(np.abs(nis).astype(np.float32)).astype(np.float64)
    assert np.all(np.abs(nis.astype(np.float64) - got["innov"][0]) <= bound)


def test_window_nll_of_whole_recording_is_innovation_nll():
    rng = np.random.default_rng(0)
    T, Ns, reps = 50, 4, 3
    terms = torch.from_numpy(rng.uniform(0.1, 5.0, size=(2, T, Ns * reps)).astype(np.float32))
    lengths = torch.tensor([50, 17, 0, 33])
    bounds = torch.stack((torch.zeros_like(lengths), lengths), dim=1)
    nll, nis = W.window_innovation_nll(terms, bounds, 3)
    assert nll.shape == (1, Ns * reps) and nll.dtype == torch.float64
    L = lengths.repeat(reps)
    sums = torch.stack([terms[:, :L[n], n].double().sum(1) for n in range(Ns * reps)], dim=1)
    want_nll, want_nis = B.innovation_nll(sums, L, "tangent")
    assert torch.allclose(nll[0], want_nll, rtol=1e-12, atol=0)
    ok = L > 0
    assert torch.allclose(nis[0][ok], want_nis[ok], rtol=1e-12) and torch.isnan(nis[0][~ok]).all()
    # two windows per stream
    w2 = torch.tensor([[[0, 10]] * Ns, [[10, 17]] * Ns])
    nll2, _ = W.window_innovation_nll(terms, w2, 4)
    assert nll2.shape == (2, Ns * reps)
    s = terms[:, 10:17].double().sum(1)
    assert torch.allclose(nll2[1], 0.5 * (s[0] + s[1]) + 2.0 * 7 * math.log(2 * math.pi), rtol=1e-12)


def test_window_nll_refuses_bad_windows():
    terms = torch.zeros((2, 10, 4))
    with pytest.raises(ValueError):
        W.window_innovation_nll(terms, torch.tensor([[0, 11]] * 4), 3)
    with pytest.raises(ValueError):
        W.window_innovation_nll(terms, torch.tensor([[5, 4]] * 4), 3)
    with pytest.raises(ValueError):
        W.window_innovation_nll(terms, torch.tensor([[0, 4]] * 3), 3)
    with pytest.raises(ValueError):
        W.window_innovation_nll(terms, torch.tensor([[0, 4]] * 4), 5)


# ---- argument rules of the C entry point (all refused before any device work) ----------------------------------
def _call(out_innov=1 << 20, stride=64 * 32, model=0, gate=math.inf, x_lo=None, q=1 << 12, N=64, T=32):
    lib = _lib.load()
    a = 1 << 12     # fake but aligned device pointers: every call below is refused on the host
    return lib.posekf_replay_innovation_steps_f32(
        N, T, a, N, a, 0, a, a, q, a, -1.0, -1.0, a, x_lo, a, None, None, None, None, None, None, model, 0, 0, 0, None,
        None, None, gate, None, None, out_innov, stride)


def test_capi_refuses_bad_arguments():
    assert _call(out_innov=None) == _lib.EINVAL
    assert _call(out_innov=(1 << 20) + 2) == _lib.EALIGN
    assert _call(stride=64 * 32 - 1) == _lib.EINVAL
    assert _call(gate=math.nan) == _lib.EINVAL
    assert _call(model=2) == _lib.EINVAL
    assert _call(model=-1) == _lib.EINVAL
    assert _call(q=None) == _lib.EINVAL          # scalar Q and R only: there is no general-matrix twin
    assert _call(T=-1) == _lib.EINVAL


def test_capi_accepts_null_output_for_an_empty_launch():
    # a launch with no step or no filter writes nothing (torch's zero-element tensors have data pointer 0)
    assert _call(out_innov=None, T=0, stride=0) == 0
    assert _call(out_innov=None, N=0, stride=0) == 0


# ---- host checks of replay(out_innovation=...) -------------------------------------------------------------------
def test_check_innovation_steps_shapes_and_strides():
    full = torch.zeros((2, 10, 8))
    # a time slice of a full-length buffer is accepted (its plane stride is T_total N); these CPU tensors are then refused
    # only for not being on the device
    for t in (full, full[:, 3:7]):
        with pytest.raises(_lib.PosekfError):
            B._check_innovation_steps(t, 8, t.shape[1])
    with pytest.raises(ValueError):
        B._check_innovation_steps(full.double(), 8, 10)
    with pytest.raises(ValueError):
        B._check_innovation_steps(full, 8, 9)
    with pytest.raises(ValueError):
        B._check_innovation_steps(full[:, :, :4], 4, 10)                            # rows not contiguous
    with pytest.raises(ValueError):
        B._check_innovation_steps(torch.zeros((10, 2, 8)).transpose(0, 1), 8, 10)   # planes interleaved
