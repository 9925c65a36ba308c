"""A batch of recordings in one launch (posekf_replay_batch_f32 / replay(dt=[T,Ns], lengths=[Ns])): every recording with
its own time steps and length gives, bit for bit, what its own single-recording replay gives, on every staging, variant
and output; held steps change nothing and read nothing; chunked equals unchunked; parity with the float64 oracle and the
float64 innovation definitions per recording; and the pooled multi-recording (Q,R) sweep."""
import math

import numpy as np
import pytest
import torch

from oracle import c_oracle as CO
from oracle import ekf_oracle as O
from poseestimationkf_b200 import batched as B
from poseestimationkf_b200 import logio
from poseestimationkf_b200 import workloads as WL
from poseestimationkf_b200.synth import make_imu
from tests import innovation_ref as IR
from tests import innovation_tangent_ref as TR

pytestmark = pytest.mark.gpu

STAGINGS = ("ldg", "tma", "tma_packed")


def _jittered_dt(T, K, seed, dt=0.01, jitter=0.2, device="cuda"):
    g = torch.Generator(device="cpu").manual_seed(seed)
    d = dt * (1.0 + jitter * (2 * torch.rand((T, K), generator=g, dtype=torch.float64) - 1))
    return d.to(torch.float32).to(device).contiguous()


def _recordings(cuda, K=64, T=200, seed=31):
    imu = make_imu(K, T, seed=seed, sigma=0.01, device=cuda, keep_truth=True)
    truth = imu.q_true.permute(0, 2, 1).to(torch.float32).contiguous()
    return imu, _jittered_dt(T, K, seed + 1, device=cuda), truth


def _tunings(K, cuda, precise):
    if precise:
        q = torch.where(torch.arange(K, device=cuda) % 2 == 0, 1e-3, 1e3).float()
        r = torch.where(torch.arange(K, device=cuda) % 2 == 0, 1e3, 1e-3).float()
    else:
        q = torch.logspace(-1, 1, K, device=cuda)
        r = torch.logspace(0.5, -1.5, K, device=cuda)
    return q.contiguous(), r.contiguous()


def _runs(truth_ok):
    """(kwargs, name) of the output combinations: per-step outputs with the truth objective (the AUX kernels), the 4-D
    innovation sums alone (the sweep path of the packed kernel), and the tangent sums with a trajectory."""
    runs = [(dict(store_trajectory=True, store_flips=True), "aux"),
            (dict(innovation=True, innovation_model="full"), "innov"),
            (dict(innovation=True, innovation_model="tangent", store_trajectory=True), "tangent+traj")]
    if truth_ok:
        runs[0][0]["truth"] = True
    return runs


def _call(streams, acc_ref, mag_ref, dt, q, r, kw, truth, precise, wahba, staging, lpf, lengths=None):
    kw = dict(kw)
    if kw.pop("truth", False):
        kw["truth"] = truth
    if lpf:
        kw.update(lpf_alpha_acc=0.3, lpf_alpha_mag=0.3)
    st, traj, flips = B.replay(streams, acc_ref, mag_ref, dt=dt, q=q, r=r, precise_state=precise, wahba=wahba, staging=staging,
                               allow_imprecise=True, lengths=lengths, **kw)
    return st, traj, flips


def _single(streams, acc_ref, mag_ref, dt_cols, q, r, kw, truth, precise, wahba, lpf, k, L=None):
    """Recording k alone, its first L steps, with its own dt [L] (the existing per-step dt path)."""
    L = streams.shape[0] if L is None else L
    sl = slice(k, k + 1)
    tr = truth[:L, sl].contiguous() if truth is not None else None
    return _call(streams[:L, :, sl].contiguous(), acc_ref[:, sl].contiguous(), mag_ref[:, sl].contiguous(),
                 dt_cols[:L, k].contiguous(), q[sl].contiguous(), r[sl].contiguous(), kw, tr, precise, wahba, "auto", lpf)


def _bits(t):
    return t.contiguous().view(torch.int32) if t.dtype == torch.float32 else t


def _assert_column_equal(batch, single, k, L, T):
    st, traj, flips = batch
    s_st, s_traj, s_flips = single
    assert torch.equal(_bits(st.x[:, k]), _bits(s_st.x[:, 0])), k
    assert torch.equal(_bits(st.p[:, k]), _bits(s_st.p[:, 0])), k
    if st.x_lo is not None and s_st.x_lo is not None:
        assert torch.equal(_bits(st.x_lo[:, k]), _bits(s_st.x_lo[:, 0])), k
    if st.loss is not None:
        assert torch.equal(_bits(st.loss[k]), _bits(s_st.loss[0])), k
    if st.innov is not None:
        assert torch.equal(_bits(st.innov[:, k]), _bits(s_st.innov[:, 0])), k
    if traj is not None:
        assert torch.equal(_bits(traj[:L, k]), _bits(s_traj[:, 0])), k
        if L < T and L > 0:       # held rows repeat the final state
            assert torch.equal(_bits(traj[L:, k]), _bits(traj[L - 1:L, k].expand(T - L, 4))), k
    if flips is not None:
        assert torch.equal(flips[:L, k], s_flips[:, 0]), k
        assert not flips[L:, k].any(), k


def _streams_for(imu, wahba):
    if wahba == "precomputed":
        return B.measurement_stream(imu.streams, imu.acc_ref, imu.mag_ref)[0]
    return imu.streams


CONFIGS = [(w, lpf) for w in ("qr2", "jacobi", "precomputed") for lpf in (False, True) if not (w == "precomputed" and lpf)]


@pytest.mark.parametrize("wahba,lpf", CONFIGS)
def test_per_stream_dt_equals_separate_replays(cuda, wahba, lpf):
    K, T = 64, 200
    imu, dt_cols, truth = _recordings(cuda, K, T)
    streams = _streams_for(imu, wahba)
    for precise in (False, True):
        q, r = _tunings(K, cuda, precise)
        for kw, name in _runs(truth_ok=True):
            singles = [_single(streams, imu.acc_ref, imu.mag_ref, dt_cols, q, r, kw, truth, precise, wahba, lpf, k)
                       for k in range(K)]
            for staging in STAGINGS:
                if wahba == "jacobi" and staging == "tma_packed":
                    continue
                out = _call(streams, imu.acc_ref, imu.mag_ref, dt_cols, q, r, kw, truth, precise, wahba, staging, lpf)
                for k in range(K):
                    _assert_column_equal(out, singles[k], k, T, T)


@pytest.mark.parametrize("staging", STAGINGS)
def test_identical_columns_equal_the_shared_dt_replay(cuda, staging):
    K, T = 256, 300
    imu = make_imu(K, T, seed=41, sigma=0.01, device=cuda)
    dt = _jittered_dt(T, 1, 42, device=cuda)[:, 0].contiguous()
    cols = dt[:, None].expand(T, K).contiguous()
    for precise in (False, True):
        q, r = _tunings(K, cuda, precise)
        for kw, name in _runs(truth_ok=False):
            a = _call(imu.streams, imu.acc_ref, imu.mag_ref, dt, q, r, kw, None, precise, "qr2", staging, False)
            b = _call(imu.streams, imu.acc_ref, imu.mag_ref, cols, q, r, kw, None, precise, "qr2", staging, False)
            for x, y in ((a[0].x, b[0].x), (a[0].p, b[0].p), (a[1], b[1]), (a[2], b[2]), (a[0].innov, b[0].innov)):
                assert (x is None) == (y is None)
                if x is not None:
                    assert torch.equal(_bits(x), _bits(y)), (name, precise)
    # a scalar dt with lengths all T runs the batched kernels and gives the plain launch's bits
    a = B.replay(imu.streams, imu.acc_ref, imu.mag_ref, dt=imu.dt, staging=staging, store_trajectory=True)
    b = B.replay(imu.streams, imu.acc_ref, imu.mag_ref, dt=imu.dt, staging=staging, store_trajectory=True,
                 lengths=torch.full((K,), T, dtype=torch.int32, device=cuda))
    assert torch.equal(_bits(a[0].x), _bits(b[0].x)) and torch.equal(_bits(a[1]), _bits(b[1]))


def _ragged_lengths(K, T, seed, cuda):
    g = torch.Generator(device="cpu").manual_seed(seed)
    L = torch.randint(T // 3, T + 1, (K,), generator=g)
    L[::13] = 0
    L[1] = T
    L[2] = 1
    return L.to(torch.int32).to(cuda)


def _nan_padded(x, L, axis_col):
    """x [T, ..., Ns] or [T, Ns, ...] with every step t >= L[c] of column c set to NaN."""
    x = x.clone()
    T = x.shape[0]
    t = torch.arange(T, device=x.device)
    dead = t[:, None] >= L[None, :].long()                 # [T, Ns]
    shape = [T] + [1] * (x.dim() - 1)
    shape[axis_col] = L.numel()
    x[dead.view(shape).expand_as(x)] = float("nan")
    return x


@pytest.mark.parametrize("wahba,lpf", CONFIGS)
def test_ragged_lengths_hold_and_read_nothing(cuda, wahba, lpf):
    K, T = 64, 200
    imu, dt_cols, truth = _recordings(cuda, K, T, seed=51)
    L = _ragged_lengths(K, T, 52, cuda)
    streams = _streams_for(imu, wahba)
    nan_streams = _nan_padded(streams, L, 2)
    nan_dt = _nan_padded(dt_cols, L, 1)
    nan_truth = _nan_padded(truth, L, 1)
    Lh = L.tolist()
    for precise in (False, True):
        q, r = _tunings(K, cuda, precise)
        for kw, name in _runs(truth_ok=True):
            singles = {k: _single(streams, imu.acc_ref, imu.mag_ref, dt_cols, q, r, kw, truth, precise, wahba, lpf, k, Lh[k])
                       for k in range(K) if Lh[k] > 0}
            for staging in STAGINGS:
                if wahba == "jacobi" and staging == "tma_packed":
                    continue
                out = _call(nan_streams, imu.acc_ref, imu.mag_ref, nan_dt, q, r, kw, nan_truth, precise, wahba, staging, lpf,
                            lengths=L)
                st, traj, flips = out
                for t in (st.x, st.p, st.x_lo, st.loss, st.innov, traj):
                    if t is not None:
                        assert torch.isfinite(t).all(), (name, staging)
                for k in range(K):
                    if Lh[k] > 0:
                        _assert_column_equal(out, singles[k], k, Lh[k], T)
                    else:               # no step at all: the initial state (through the frame round trip), nothing added
                        assert torch.allclose(st.x[:, k], torch.tensor([1.0, 0, 0, 0], device=cuda), atol=1e-6)
                        if st.innov is not None:
                            assert not st.innov[:, k].any()
                        if st.loss is not None:
                            assert st.loss[k].item() == 0.0
                        if traj is not None:
                            assert torch.equal(traj[:, k], traj[:1, k].expand(T, 4))
                        if flips is not None:
                            assert not flips[:, k].any()


@pytest.mark.parametrize("staging", STAGINGS)
def test_chunked_equals_unchunked(cuda, staging):
    K, T, chunk = 256, 256, 64
    imu, dt_cols, _ = _recordings(cuda, K, T, seed=61)
    L = _ragged_lengths(K, T, 62, cuda)
    L[3:12] = torch.tensor([63, 64, 65, 127, 128, 129, 192, 191, 193], dtype=torch.int32, device=cuda)
    lb = logio.LogBatch(_nan_padded(imu.streams, L, 2), imu.acc_ref, imu.mag_ref, _nan_padded(dt_cols, L, 1), L, K)
    q, r = _tunings(K, cuda, False)
    for model in ("full", "tangent"):
        ref, traj, flips = B.replay(lb.streams, lb.acc_ref, lb.mag_ref, dt=lb.dt, q=q, r=r, lengths=lb.lengths,
                                    staging=staging, innovation=True, innovation_model=model, store_trajectory=True,
                                    store_flips=True)
        st = None
        trs, fls = [], []
        for t0 in range(0, T, chunk):
            w = lb.window(t0, t0 + chunk)
            st, tr, fl = B.replay(w.streams, w.acc_ref, w.mag_ref, dt=w.dt, q=q, r=r, lengths=w.lengths, state=st,
                                  staging=staging, innovation=True if st is None else st.innov, innovation_model=model,
                                  store_trajectory=True, store_flips=True, keep_filter_frame=t0 + chunk < T)
            trs.append(tr)
            fls.append(fl)
        assert torch.equal(_bits(st.x), _bits(ref.x)) and torch.equal(_bits(st.p), _bits(ref.p))
        assert torch.equal(_bits(st.innov), _bits(ref.innov))
        assert torch.equal(_bits(torch.cat(trs)), _bits(traj)) and torch.equal(torch.cat(fls), flips)


@pytest.mark.parametrize("staging", ("auto", "tma", "ldg"))
def test_oracle_parity_per_recording(cuda, staging):
    K, T = 256, 2000
    imu = make_imu(K, T, seed=71, sigma=0.01, device=cuda)
    dt_cols = _jittered_dt(T, K, 72, device=cuda)
    g = torch.Generator(device="cpu").manual_seed(73)
    L = torch.randint(T // 2, T + 1, (K,), generator=g).to(torch.int32)
    L[0] = T
    st, traj, flips = B.replay(imu.streams, imu.acc_ref, imu.mag_ref, dt=dt_cols, q=1.0, r=0.1, lengths=L.to(cuda),
                               staging=staging, store_trajectory=True, store_flips=True)
    torch.cuda.synchronize()
    S, D = imu.streams.cpu().numpy(), dt_cols.double().cpu().numpy() * 1e9
    ar, mr = imu.acc_ref.cpu().numpy(), imu.mag_ref.cpu().numpy()
    got, fl = traj.cpu().numpy(), flips.cpu().numpy().astype(bool)
    worst, mism = 0.0, 0
    for k in range(K):
        Lk = int(L[k])
        ref = CO.replay(S[:Lk, :, k:k + 1], D[:Lk, k], ar[:, k:k + 1], mr[:, k:k + 1], 1.0, 0.1)
        g_k = got[:Lk, k:k + 1]
        ang = O.quat_angle(g_k, ref["X"])
        worst = max(worst, float(ang.max()))
        assert (np.sum(g_k * ref["X"], axis=-1) > 0).all(), k          # same quaternion sign as the oracle
        mism += int((fl[:Lk, k:k + 1] != ref["flips"]).sum()) + int(fl[Lk:, k].sum())
    assert worst <= 1e-5, worst
    assert mism == 0


@pytest.mark.parametrize("model", ("full", "tangent"))
@pytest.mark.parametrize("staging", STAGINGS)
def test_innovation_sums_per_recording(cuda, model, staging):
    K, T = 64, 300
    imu, dt_cols, _ = _recordings(cuda, K, T, seed=81)
    L = _ragged_lengths(K, T, 82, cuda)
    q, r = _tunings(K, cuda, False)
    st, _, _ = B.replay(_nan_padded(imu.streams, L, 2), imu.acc_ref, imu.mag_ref, dt=_nan_padded(dt_cols, L, 1), q=q, r=r,
                        lengths=L, staging=staging, innovation=True, innovation_model=model)
    S = imu.streams.cpu().numpy().astype(np.float64)
    R = (TR.replay_tangent if model == "tangent" else IR.replay_innovation)(
        dt_cols.double().cpu().numpy() * 1e9, S[:, 0:3], S[:, 3:6], S[:, 6:9], imu.acc_ref.cpu().numpy().T,
        imu.mag_ref.cpu().numpy().T, q.cpu().numpy().astype(np.float64), r.cpu().numpy().astype(np.float64))
    Lh = L.cpu().numpy()
    live = np.arange(T)[:, None] < Lh[None, :]
    nis, logdet = np.where(live, R["nis"], 0).sum(0), np.where(live, R["logdet"], 0).sum(0)
    got = st.innov.double().cpu().numpy()
    # Error bar: 1e-4 of the magnitude the float32 sums carry, sum_t (|NIS_t| + |ln det S_t|).  On a recording whose
    # ln det S_t change sign the sum cancels (|sum NIS| + |sum ln det S| can be 1 % of it), and what is left is the
    # rounding of the float32 running sum, not an error of any step; without cancellation this is the bar
    # |sum NIS| + |sum ln det S| of tests/test_gpu_innovation*.py.
    scale = np.where(live, np.abs(R["nis"]) + np.abs(R["logdet"]), 0).sum(0)
    nz = Lh > 0
    assert np.max(np.abs(got[0] - nis)[nz] / scale[nz]) <= 1e-4
    assert np.max(np.abs(got[1] - logdet)[nz] / scale[nz]) <= 1e-4
    assert not got[:, ~nz].any()
    nll, mnis = B.innovation_nll(st, L)
    dof = 3 if model == "tangent" else 4
    ref_nll = 0.5 * (nis + logdet) + 0.5 * dof * Lh * math.log(2 * math.pi)
    assert np.max(np.abs(nll.cpu().numpy() - ref_nll)[nz] / (scale[nz] + 0.5 * dof * Lh[nz] * math.log(2 * math.pi))) <= 1e-4
    assert np.max(np.abs(mnis.cpu().numpy() - nis / np.maximum(Lh, 1))[nz] / (scale / np.maximum(Lh, 1))[nz]) <= 1e-4


def _log_from(imu, k, L, dt_ns, t0_ns):
    """recording k of a synthetic batch as a LogData with timestamps t0 + cumsum(dt)."""
    s = imu.streams[:L, :, k].double().cpu().numpy()
    t = np.concatenate([[t0_ns], t0_ns + np.cumsum(dt_ns[:L])])
    return logio.LogData(mag_0=imu.mag_ref[:, k].double().cpu().numpy(), acc_0=imu.acc_ref[:, k].double().cpu().numpy(),
                         gyro=s[:, 0:3], acc_1=s[:, 3:6], mag_1=s[:, 6:9], timestamp=t[:, None])


def test_pooled_sweep_equals_single_recording_sweeps(cuda):
    K, T, G, lo, step = 8, 300, 16, -5.0, 0.3
    imu = make_imu(K, T, seed=91, sigma=0.01, device=cuda)
    rng = np.random.default_rng(92)
    lens = [T, 170, 233, 101, 300, 256, 150, 280]
    logs = [_log_from(imu, k, lens[k], np.rint(1e7 * (1 + 0.2 * rng.uniform(-1, 1, T))).astype(np.int64),
                      1_600_000_000_000_000_000 + 10**9 * k) for k in range(K)]
    w = WL.build_multi_recording_sweep(logs, cuda, grid=G, lo=lo, step=step)
    Ns = w.streams.shape[2]
    assert Ns == 8 and w.lengths.tolist() == lens
    st = WL.run_c3(w, objective="innovation_tangent")
    multi = st.innov.reshape(2, G, G, Ns)
    singles = []
    for k in range(K):
        ws = WL.build_recording_sweep(logs[k], cuda, grid=G, lo=lo, step=step)
        ss = WL.run_c3(ws, objective="innovation_tangent")
        singles.append(ss.innov.reshape(2, G, G))
        assert torch.equal(_bits(multi[..., k].contiguous()), _bits(ss.innov.reshape(2, G, G))), k
    nll, nis = WL.pooled_innovation_surface(w, st)
    # float64 definition: every (cell, recording) filter through the tangent reference over its own steps
    q = w.q.double().cpu().numpy()
    r = w.r.double().cpu().numpy()
    S = w.streams.double().cpu().numpy()
    N = q.size
    Sn = np.tile(S, (1, 1, N // Ns))
    D = np.tile(w.dt.double().cpu().numpy() * 1e9, (1, N // Ns))
    R = TR.replay_tangent(D, Sn[:, 0:3], Sn[:, 3:6], Sn[:, 6:9], np.tile(w.acc_ref.cpu().numpy().T, (N // Ns, 1)),
                          np.tile(w.mag_ref.cpu().numpy().T, (N // Ns, 1)), q, r)
    Lf = np.tile(np.asarray(lens, dtype=np.float64), N // Ns)
    live = np.arange(T)[:, None] < Lf[None, :]
    a0, a1 = np.where(live, R["nis"], 0).sum(0), np.where(live, R["logdet"], 0).sum(0)
    per = 0.5 * (a0 + a1) + 1.5 * Lf * math.log(2 * math.pi)
    ref_nll = per.reshape(G, G, Ns).sum(2) / sum(lens)
    scale = (np.abs(a0) + np.abs(a1)).reshape(G, G, Ns).sum(2) / sum(lens)
    got = nll.cpu().numpy()
    assert np.max(np.abs(got - ref_nll) / scale) <= 1e-4
    assert np.argmin(got) == np.argmin(ref_nll)
    assert np.max(np.abs(nis.cpu().numpy() - a0.reshape(G, G, Ns).sum(2) / sum(lens)) / scale) <= 1e-4
