"""Tangent-space innovation likelihood on the device (posekf_replay_innovation_ex_f32 with POSEKF_INNOV_TANGENT /
replay(innovation=..., innovation_model="tangent")): against the float64 definition on every path, bitwise properties
across stagings, chunking and the mixed-precision sweep, model 0 of the new entry point against the 4-D one, a small
tuning sweep whose argmin is interior in R, and guard bands around the accumulator."""
import numpy as np
import pytest
import torch

from poseestimationkf_b200 import _lib
from poseestimationkf_b200 import batched as B
from poseestimationkf_b200 import workloads as WL
from poseestimationkf_b200.synth import make_imu
from tests import innovation_tangent_ref as TR

pytestmark = pytest.mark.gpu

# Error bar of the per-filter sums, relative to the likelihood they form (|sum NIS3| + |sum ln det S3|), as for the 4-D
# objective (tests/test_gpu_innovation.py).  Measured maximum on B200: DESIGN.md section 5.
RTOL = 1e-4
TAN = dict(innovation=True, innovation_model="tangent")


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
    ref = TR.replay_tangent(np.full(T, float(np.float32(imu.dt)) * 1e9), S[:, 0:3], S[:, 3:6], S[:, 6:9],
                            imu.acc_ref.cpu().numpy().T, imu.mag_ref.cpu().numpy().T,
                            q.cpu().numpy().astype(np.float64), r.cpu().numpy().astype(np.float64))
    return ref["nis"].sum(0), ref["logdet"].sum(0)


def _err(got, nis, logdet):
    """max over filters and both sums of |error| / (|sum NIS3| + |sum ln det S3|)."""
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
def test_sums_match_definition_every_path(cuda, precise):
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
                                staging=staging, allow_imprecise=True, **TAN)
            assert st.innov_model == "tangent"
            e = _err(st.innov.double().cpu().numpy(), *ref)
            worst = max(worst, e)
            assert e <= RTOL, (wahba, staging, e)
    ref_l = _ref_sums(imu, q, r, alpha=0.3)
    for staging in ("ldg", "tma", "tma_packed"):
        st, _, _ = B.replay(imu.streams, imu.acc_ref, imu.mag_ref, dt=imu.dt, q=q, r=r, precise_state=precise, staging=staging,
                            lpf_alpha_acc=0.3, lpf_alpha_mag=0.3, **TAN)
        e = _err(st.innov.double().cpu().numpy(), *ref_l)
        worst = max(worst, e)
        assert e <= RTOL, ("lpf", staging, e)
    print(f"tangent innovation sums, precise={precise}: max relative error {worst:.3e}")


def test_golden_trajectories(cuda, golden_traj):
    g = golden_traj
    worst = 0.0
    for tag in ("clean", "noisy"):
        S = torch.from_numpy(g[tag + "_streams"]).to(cuda)
        ar = torch.from_numpy(g[tag + "_acc_ref"]).to(cuda); mr = torch.from_numpy(g[tag + "_mag_ref"]).to(cuda)
        T, _, N = S.shape
        S64 = g[tag + "_streams"].astype(np.float64)
        for q, r in ((1.0, 0.1), (1e-3, 1e3), (1e3, 1e-3)):
            ref = TR.replay_tangent(np.full(T, float(np.float32(g["dt"])) * 1e9), S64[:, 0:3], S64[:, 3:6], S64[:, 6:9],
                                    g[tag + "_acc_ref"].T, g[tag + "_mag_ref"].T, float(np.float32(q)), float(np.float32(r)))
            for staging in ("ldg", "tma", "tma_packed"):
                st, _, _ = B.replay(S, ar, mr, dt=float(g["dt"]), q=q, r=r, staging=staging, **TAN)
                e = _err(st.innov.double().cpu().numpy(), ref["nis"].sum(0), ref["logdet"].sum(0))
                worst = max(worst, e)
                assert e <= RTOL, (tag, q, r, staging, e)
    print(f"tangent innovation sums, golden trajectories: max relative error {worst:.3e}")


def test_long_replay(cuda):
    N, T = 256, 20000
    imu = make_imu(N, T, seed=5, sigma=0.01, device=cuda)
    q = torch.logspace(-1, 1, N, device=cuda); r = torch.full((N,), 0.1, device=cuda)
    ref = _ref_sums(imu, q, r)
    st, _, _ = B.replay(imu.streams, imu.acc_ref, imu.mag_ref, dt=imu.dt, q=q, r=r, **TAN)
    e = _err(st.innov.double().cpu().numpy(), *ref)
    print(f"tangent innovation sums, T={T}: max relative error {e:.3e}")
    assert e <= RTOL


@pytest.mark.parametrize("precise", [False, True])
def test_stagings_bitwise_and_statistic_does_not_perturb(cuda, precise):
    N, T = 1024, 101
    imu = make_imu(N, T, seed=8, sigma=0.01, device=cuda)
    q, r = _tunings(N, cuda, precise)
    outs = {}
    for staging in ("ldg", "tma", "tma_packed"):
        on, traj_on, fl_on = B.replay(imu.streams, imu.acc_ref, imu.mag_ref, dt=imu.dt, q=q, r=r, precise_state=precise,
                                      staging=staging, store_trajectory=True, store_flips=True, **TAN)
        off, traj_off, fl_off = B.replay(imu.streams, imu.acc_ref, imu.mag_ref, dt=imu.dt, q=q, r=r, precise_state=precise,
                                         staging=staging, store_trajectory=True, store_flips=True)
        assert torch.equal(on.x, off.x) and torch.equal(on.p, off.p) and torch.equal(traj_on, traj_off) and torch.equal(fl_on, fl_off)
        plain_on, _, _ = B.replay(imu.streams, imu.acc_ref, imu.mag_ref, dt=imu.dt, q=q, r=r, precise_state=precise,
                                  staging=staging, **TAN)
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
    whole, _, _ = B.replay(imu.streams, imu.acc_ref, imu.mag_ref, dt=imu.dt, q=q, r=r, staging=staging, **TAN)
    st = None
    for t0, t1 in ((0, 37), (37, 64), (64, 100)):
        st, _, _ = B.replay(imu.streams[t0:t1].contiguous(), imu.acc_ref, imu.mag_ref, dt=imu.dt, q=q, r=r, state=st,
                            staging=staging, keep_filter_frame=t1 < T, innovation=True if st is None else st.innov,
                            innovation_model="tangent")
    assert torch.equal(st.x, whole.x) and torch.equal(st.innov, whole.innov)
    # the state's accumulator holds tangent sums: continuing it under the other model is refused
    with pytest.raises(ValueError):
        B.replay(imu.streams[:5].contiguous(), imu.acc_ref, imu.mag_ref, dt=imu.dt, q=q, r=r, state=st, innovation=st.innov)


def _entry(fn, imu, q, r, st, innov, staging, *extra):
    T, _, Ns = imu.streams.shape
    dt = torch.full((1,), imu.dt, dtype=torch.float32, device=imu.streams.device)
    args = (st.x.shape[1], T, imu.streams.data_ptr(), Ns, dt.data_ptr(), 0, imu.acc_ref.data_ptr(), imu.mag_ref.data_ptr(),
            q.data_ptr(), r.data_ptr(), -1.0, -1.0, st.x.data_ptr(), None if st.x_lo is None else st.x_lo.data_ptr(),
            st.p.data_ptr(), None, None, None, None, None, innov.data_ptr())
    rc = fn(*args, *extra, _lib.WAHBA["qr2"], _lib.STAGING[staging], 0, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert rc == 0


@pytest.mark.parametrize("precise", [False, True])
def test_model_full_equals_the_4d_entry_point(cuda, precise):
    N, T = 512, 64
    imu = make_imu(N, T, seed=12, sigma=0.01, device=cuda)
    q, r = _tunings(N, cuda, precise)
    lib = _lib.load()
    for staging in ("ldg", "tma", "tma_packed"):
        outs = []
        for fn, extra in ((lib.posekf_replay_innovation_f32, ()), (lib.posekf_replay_innovation_ex_f32, (_lib.INNOV_MODEL["full"],)),
                          (lib.posekf_replay_innovation_ex_f32, (_lib.INNOV_MODEL["tangent"],))):
            st = B.ReplayState.initial(N, cuda, r=r)
            if precise:
                st.x_lo = torch.zeros((4, N), device=cuda)
            innov = torch.zeros((2, N), device=cuda)
            _entry(fn, imu, q, r, st, innov, staging, *extra)
            outs.append((st, innov))
        (a, ia), (b, ib), (c, ic) = outs
        assert torch.equal(ia, ib) and torch.equal(a.x, b.x) and torch.equal(a.p, b.p), staging
        assert torch.equal(a.x, c.x) and torch.equal(a.p, c.p) and not torch.equal(ia, ic), staging


def test_mixed_sweep_equals_groups_alone(cuda):
    w = WL.build_c3(cuda, grid=8, n_streams=256, n_steps=64, lo=-3.0, step=6.0 / 7)
    st = WL.run_c3(w, objective="innovation_tangent")
    assert st.innov_model == "tangent"
    idx_plain, idx_precise = B.sweep_partition(w.q, w.r, 256)
    assert idx_plain.numel() and idx_precise.numel()
    meas, _ = B.measurement_stream(w.streams, w.acc_ref, w.mag_ref)
    for idx, precise in ((idx_plain, False), (idx_precise, True)):
        alone, _, _ = B.replay(meas, w.acc_ref, w.mag_ref, dt=w.dt, q=w.q[idx].contiguous(), r=w.r[idx].contiguous(),
                               n_filters=idx.numel(), precise_state=precise, wahba="precomputed", **TAN)
        assert torch.equal(st.innov[:, idx], alone.innov)
        assert torch.equal(st.x[:, idx], alone.x)


def test_small_sweep_picks_the_float64_minimum_interior_in_r(cuda):
    # grid 1e-7 .. 1e-1 on both axes, one value per decade, on the config-3 data (sigma = 0.01): the tangent objective has
    # its minimum inside the grid on both axes (float64: q = 1e-5, r = 1e-4, mean NIS 3.3), unlike the 4-D one, whose
    # R axis keeps falling (tests/test_gpu_innovation.py)
    G, Ns, T = 7, 16, 500
    w = WL.build_c3(cuda, grid=G, n_streams=Ns, n_steps=T, lo=-7.0, step=1.0)
    st = WL.run_c3(w, objective="innovation_tangent")
    nll_dev, nis_dev = WL.innovation_surface(w, st)
    assert torch.isfinite(nll_dev).all() and (nis_dev > 0).all()
    reps = G * G
    S = w.streams.cpu().numpy().astype(np.float64)
    ref = TR.replay_tangent(np.full(T, float(np.float32(w.dt)) * 1e9), np.tile(S[:, 0:3], reps), np.tile(S[:, 3:6], reps),
                            np.tile(S[:, 6:9], reps), np.tile(w.acc_ref.cpu().numpy().T, (reps, 1)),
                            np.tile(w.mag_ref.cpu().numpy().T, (reps, 1)), w.q.cpu().numpy().astype(np.float64),
                            w.r.cpu().numpy().astype(np.float64))
    nll64 = TR.nll(ref["nis"].sum(0), ref["logdet"].sum(0), T).reshape(G, G, Ns).mean(2) / T
    best_dev = np.unravel_index(int(nll_dev.argmin()), (G, G))
    best64 = np.unravel_index(int(nll64.argmin()), (G, G))
    assert 0 < best64[0] < G - 1 and 0 < best64[1] < G - 1, best64
    assert best_dev == best64, (best_dev, best64)
    assert 2.0 <= float(nis_dev[best_dev]) <= 4.0
    err = np.abs(nll_dev.cpu().numpy() - nll64) / np.maximum(np.abs(nll64), 1.0)
    print(f"small tangent sweep: argmin {best64}, NLL per step max error {err.max():.3e} (relative, or absolute below 1)")
    assert err.max() <= 1e-4


def test_no_out_of_bounds_writes_tangent(cuda):
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
                                    innovation=acc, innovation_model="tangent", **kw)
                torch.cuda.synchronize()
                assert bool((buf[:GUARD] == POISON).all() and (buf[GUARD + 2 * N:] == POISON).all()), (N, staging, precise, kw)
                assert torch.isfinite(acc).all() and (acc[0] > 0).all() and st.innov is acc
