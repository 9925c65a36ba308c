"""Innovation likelihood on the device (posekf_replay_innovation_f32 / replay(innovation=...)): against the float64
definition on every path, bitwise properties across stagings, chunking and the mixed-precision sweep, a small tuning
sweep, and guard bands around the accumulator."""
import math

import numpy as np
import pytest
import torch

from oracle import ekf_oracle as O
from poseestimationkf_b200 import batched as B
from poseestimationkf_b200 import workloads as WL
from poseestimationkf_b200.synth import make_imu
from tests import innovation_ref as IR

pytestmark = pytest.mark.gpu

# Error bar of the per-filter sums, relative to the likelihood they form (|sum NIS| + |sum ln det S|): at Q >> R the filter
# copies its measurement and sum NIS is ~1e-7 of the NLL, below what a float32 innovation (a difference of unit
# quaternions) resolves -- there only its share of the NLL is meaningful.  Measured maximum on B200: DESIGN.md section 5.
RTOL = 1e-4


def _lowpassed(S, alpha):
    """float64 low-pass of the acc / mag rows of a [T,9,N] stream (PKF/Test.py:27-33), state from 0."""
    out = S.copy()
    y = np.zeros_like(S[0, 3:9])
    for t in range(S.shape[0]):
        y = alpha * S[t, 3:9] + (1 - alpha) * y
        out[t, 3:9] = y
    return out


def _ref_sums(imu, q, r, alpha=None):
    S = imu.streams.cpu().numpy().astype(np.float64)
    if alpha is not None:
        S = _lowpassed(S, float(np.float32(alpha)))
    T = S.shape[0]
    q64 = q.cpu().numpy().astype(np.float64); r64 = r.cpu().numpy().astype(np.float64)
    ref = IR.replay_innovation(np.full(T, float(np.float32(imu.dt)) * 1e9), S[:, 0:3], S[:, 3:6], S[:, 6:9],
                               imu.acc_ref.cpu().numpy().T, imu.mag_ref.cpu().numpy().T, q64, r64)
    return ref["nis"].sum(0), ref["logdet"].sum(0)


def _err(got, nis, logdet):
    """max over filters and both sums of |error| / (|sum NIS| + |sum ln det S|)."""
    scale = np.abs(nis) + np.abs(logdet)
    return float(max(np.max(np.abs(got[0] - nis) / scale), np.max(np.abs(got[1] - logdet) / scale)))


def _tunings(N, device, precise):
    if not precise:       # inside the plain variant's range
        q = torch.logspace(-1, 1, N, device=device); r = torch.logspace(0.5, -1.5, N, device=device)
    else:                 # both extremes: R >> Q and Q >> R
        q = torch.where(torch.arange(N, device=device) % 2 == 0, 1e-3, 1e3).float()
        r = torch.where(torch.arange(N, device=device) % 2 == 0, 1e3, 1e-3).float()
    return q.contiguous(), r.contiguous()


@pytest.mark.parametrize("precise", [False, True])
def test_sums_match_reference_every_path(cuda, precise):
    N, T = 512, 300
    imu = make_imu(N, T, seed=21, sigma=0.01, device=cuda)
    q, r = _tunings(N, cuda, precise)
    ref = _ref_sums(imu, q, r)
    worst = 0.0
    for wahba in ("qr2", "jacobi", "precomputed"):
        streams = imu.streams if wahba != "precomputed" else B.measurement_stream(imu.streams, imu.acc_ref, imu.mag_ref)[0]
        for staging in ("ldg", "tma", "tma_packed"):
            if wahba == "jacobi" and staging == "tma_packed":
                continue
            st, _, _ = B.replay(streams, imu.acc_ref, imu.mag_ref, dt=imu.dt, q=q, r=r, precise_state=precise, wahba=wahba,
                                staging=staging, innovation=True, allow_imprecise=True)
            got = st.innov.double().cpu().numpy()
            e = _err(got, *ref)
            worst = max(worst, e)
            assert e <= RTOL, (wahba, staging, e)
    # the low-pass stage (raw streams only)
    ref_l = _ref_sums(imu, q, r, alpha=0.3)
    for staging in ("ldg", "tma", "tma_packed"):
        st, _, _ = B.replay(imu.streams, imu.acc_ref, imu.mag_ref, dt=imu.dt, q=q, r=r, precise_state=precise, staging=staging,
                            lpf_alpha_acc=0.3, lpf_alpha_mag=0.3, innovation=True)
        got = st.innov.double().cpu().numpy()
        e = _err(got, *ref_l)
        worst = max(worst, e)
        assert e <= RTOL, ("lpf", staging, e)
    print(f"innovation sums, precise={precise}: max relative error {worst:.3e}")


def test_golden_trajectories(cuda, golden_traj):
    g = golden_traj
    for tag in ("clean", "noisy"):
        S = torch.from_numpy(g[tag + "_streams"]).to(cuda)
        ar = torch.from_numpy(g[tag + "_acc_ref"]).to(cuda); mr = torch.from_numpy(g[tag + "_mag_ref"]).to(cuda)
        T, _, N = S.shape
        for q, r, precise in ((1.0, 0.1, False), (1e-3, 1e3, True), (1e3, 1e-3, True)):
            S64 = g[tag + "_streams"].astype(np.float64)
            ref = IR.replay_innovation(np.full(T, float(np.float32(g["dt"])) * 1e9), S64[:, 0:3], S64[:, 3:6], S64[:, 6:9],
                                       g[tag + "_acc_ref"].T, g[tag + "_mag_ref"].T, float(np.float32(q)), float(np.float32(r)))
            for staging in ("ldg", "tma", "tma_packed"):
                st, _, _ = B.replay(S, ar, mr, dt=float(g["dt"]), q=q, r=r, staging=staging, innovation=True)
                got = st.innov.double().cpu().numpy()
                e = _err(got, ref["nis"].sum(0), ref["logdet"].sum(0))
                assert e <= RTOL, (tag, q, r, staging, e)
                if q / r < 1e4:        # where NIS is a sizeable part of the likelihood it also meets the bar on its own
                    assert float(np.max(np.abs(got[0] / ref["nis"].sum(0) - 1))) <= RTOL, (tag, q, r, staging)


def test_long_replay(cuda):
    N, T = 256, 20000
    imu = make_imu(N, T, seed=5, sigma=0.01, device=cuda)
    q = torch.logspace(-1, 1, N, device=cuda); r = torch.full((N,), 0.1, device=cuda)
    ref = _ref_sums(imu, q, r)
    st, _, _ = B.replay(imu.streams, imu.acc_ref, imu.mag_ref, dt=imu.dt, q=q, r=r, innovation=True)
    got = st.innov.double().cpu().numpy()
    e = _err(got, *ref)
    print(f"innovation sums, T={T}: max relative error {e:.3e}")
    assert e <= RTOL


@pytest.mark.parametrize("precise", [False, True])
def test_stagings_bitwise_and_statistic_does_not_perturb(cuda, precise):
    N, T = 1024, 101
    imu = make_imu(N, T, seed=8, sigma=0.01, device=cuda)
    q, r = _tunings(N, cuda, precise)
    outs = {}
    for staging in ("ldg", "tma", "tma_packed"):
        on, traj_on, fl_on = B.replay(imu.streams, imu.acc_ref, imu.mag_ref, dt=imu.dt, q=q, r=r, precise_state=precise,
                                      staging=staging, innovation=True, store_trajectory=True, store_flips=True)
        off, traj_off, fl_off = B.replay(imu.streams, imu.acc_ref, imu.mag_ref, dt=imu.dt, q=q, r=r, precise_state=precise,
                                         staging=staging, store_trajectory=True, store_flips=True)
        assert torch.equal(on.x, off.x) and torch.equal(on.p, off.p) and torch.equal(traj_on, traj_off) and torch.equal(fl_on, fl_off)
        # the packed kernel carries the statistic without per-step outputs (the sweep path)
        plain_on, _, _ = B.replay(imu.streams, imu.acc_ref, imu.mag_ref, dt=imu.dt, q=q, r=r, precise_state=precise,
                                  staging=staging, innovation=True)
        plain_off, _, _ = B.replay(imu.streams, imu.acc_ref, imu.mag_ref, dt=imu.dt, q=q, r=r, precise_state=precise, staging=staging)
        assert torch.equal(plain_on.x, plain_off.x) and torch.equal(plain_on.p, plain_off.p)
        assert torch.equal(plain_on.innov, on.innov)
        outs[staging] = on.innov
    assert torch.equal(outs["ldg"], outs["tma"]) and torch.equal(outs["tma"], outs["tma_packed"])


@pytest.mark.parametrize("staging", ["ldg", "tma_packed"])
def test_chunked_equals_unchunked(cuda, staging):
    N, T = 512, 100
    imu = make_imu(N, T, seed=9, sigma=0.01, device=cuda)
    q, r = _tunings(N, cuda, False)
    whole, _, _ = B.replay(imu.streams, imu.acc_ref, imu.mag_ref, dt=imu.dt, q=q, r=r, staging=staging, innovation=True)
    st = None
    for t0, t1 in ((0, 37), (37, 64), (64, 100)):
        st, _, _ = B.replay(imu.streams[t0:t1].contiguous(), imu.acc_ref, imu.mag_ref, dt=imu.dt, q=q, r=r, state=st,
                            staging=staging, keep_filter_frame=t1 < T, innovation=True if st is None else st.innov)
    assert torch.equal(st.x, whole.x) and torch.equal(st.innov, whole.innov)


def test_mixed_sweep_equals_groups_alone(cuda):
    w = WL.build_c3(cuda, grid=8, n_streams=256, n_steps=64, lo=-3.0, step=6.0 / 7)
    st = WL.run_c3(w, objective="innovation")
    idx_plain, idx_precise = B.sweep_partition(w.q, w.r, 256)
    assert idx_plain.numel() and idx_precise.numel()
    meas, _ = B.measurement_stream(w.streams, w.acc_ref, w.mag_ref)
    for idx, precise in ((idx_plain, False), (idx_precise, True)):
        alone, _, _ = B.replay(meas, w.acc_ref, w.mag_ref, dt=w.dt, q=w.q[idx].contiguous(), r=w.r[idx].contiguous(),
                               n_filters=idx.numel(), precise_state=precise, wahba="precomputed", innovation=True)
        assert torch.equal(st.innov[:, idx], alone.innov)
        assert torch.equal(st.x[:, idx], alone.x)


def test_small_sweep_picks_the_float64_minimum(cuda):
    # grid 3e-7 .. 1e-1 on both axes: it holds the Q that fits this data (the reference's P recursion forgets its prior,
    # P^- ~ q/4 (I - x x^T), and the attitude moves ~5e-3 per step).  In R the likelihood of the reference's model keeps
    # falling towards r ~ (|e|^2/2)^2: the direction of the state sees almost no innovation (DESIGN.md section 5), so its
    # minimum sits on the lowest R of any practical grid; the Q axis has an interior minimum.
    G, Ns, T = 8, 16, 500
    w = WL.build_c3(cuda, grid=G, n_streams=Ns, n_steps=T, lo=-6.5, step=0.75)
    st = WL.run_c3(w, objective="innovation")
    nll_dev, nis_dev = WL.innovation_surface(w, st)
    assert torch.isfinite(nll_dev).all() and (nis_dev > 0).all()
    reps = G * G
    S = w.streams.cpu().numpy().astype(np.float64)
    ref = IR.replay_innovation(np.full(T, float(np.float32(w.dt)) * 1e9), np.tile(S[:, 0:3], reps), np.tile(S[:, 3:6], reps),
                               np.tile(S[:, 6:9], reps), np.tile(w.acc_ref.cpu().numpy().T, (reps, 1)),
                               np.tile(w.mag_ref.cpu().numpy().T, (reps, 1)), w.q.cpu().numpy().astype(np.float64),
                               w.r.cpu().numpy().astype(np.float64))
    nll64 = IR.nll(ref["nis"].sum(0), ref["logdet"].sum(0), T).reshape(G, G, Ns).mean(2) / T
    best_dev = np.unravel_index(int(nll_dev.argmin()), (G, G))
    best64 = np.unravel_index(int(nll64.argmin()), (G, G))
    assert 0 < best64[0] < G - 1 and best64[1] == 0, best64          # interior in Q, lowest R (see above)
    assert abs(nll64[best_dev] - nll64.min()) <= 1e-4 * abs(nll64.min()), (best_dev, best64)
    err = np.abs(nll_dev.cpu().numpy() - nll64) / np.maximum(np.abs(nll64), 1.0)
    print(f"small sweep: NLL per step max error {err.max():.3e} (relative, or absolute below 1)")
    assert err.max() <= 1e-4


def test_no_out_of_bounds_writes_innovation(cuda):
    GUARD, POISON = 4096, -12345.0
    for N, T, staging in ((1000, 37, "tma"), (1000, 37, "tma_packed"), (1000, 37, "ldg"), (130, 9, "auto"), (516, 5, "tma_packed"),
                          (4, 1, "tma_packed"), (3, 2, "ldg")):
        imu = make_imu(N, T, seed=N + T, sigma=0.01, device=cuda)
        for precise in (False, True):
            for kw in (dict(), dict(store_trajectory=True, store_flips=True), dict(lpf_alpha_acc=0.2, lpf_alpha_mag=0.2)):
                buf = torch.full((2 * N + 2 * GUARD,), POISON, device=cuda)
                acc = buf[GUARD:GUARD + 2 * N].view(2, N)
                acc.zero_()
                st, _, _ = B.replay(imu.streams, imu.acc_ref, imu.mag_ref, dt=imu.dt, precise_state=precise, staging=staging,
                                    innovation=acc, **kw)
                torch.cuda.synchronize()
                assert bool((buf[:GUARD] == POISON).all() and (buf[GUARD + 2 * N:] == POISON).all()), (N, staging, precise, kw)
                assert torch.isfinite(acc).all() and (acc[0] > 0).all() and st.innov is acc
