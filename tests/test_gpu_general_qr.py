"""General Q and R matrices on the device (posekf_replay_general_f32 / replay(q=<matrix>, r=<matrix>)): trajectories and
flip masks against the float64 definition (tests/general_qr_ref.py) on the golden trajectories and on 600 000 seeded
steps, every staging and Wahba mode with and without the low-pass; LDG against TMA, chunked against unchunked, ragged
batches against single recordings and shared against per-filter matrices bit for bit; the tuning loss against its
float64 recomputation; guard bands around every output; the host API's rules."""
import numpy as np
import pytest
import torch

from oracle import ekf_oracle as O
from poseestimationkf_b200 import batched as B
from poseestimationkf_b200.synth import make_imu
from tests import general_qr_ref as GR

pytestmark = pytest.mark.gpu


def _f32(M):
    """The float32 values the kernels see ([N,k,k] or [k,k]: upper triangle rounded, mirrored)."""
    M = np.asarray(M, dtype=np.float64)
    U = np.triu(M).astype(np.float32).astype(np.float64)
    return U + np.swapaxes(np.triu(U, 1), -1, -2)


def _matrices(kind, N, seed=0):
    rng = np.random.default_rng(seed)
    if kind == "full":             # full Q, full anisotropic R
        return GR.random_spd(rng, N, 3, 1e-4, 1e-2), GR.random_spd(rng, N, 4, 1e-3, 1e-1)
    if kind == "diag":
        return (np.einsum("nk,kj->nkj", np.exp(rng.uniform(np.log(1e-4), np.log(1e-2), (N, 3))), np.eye(3)),
                np.einsum("nk,kj->nkj", np.exp(rng.uniform(np.log(1e-3), np.log(1e-1), (N, 4))), np.eye(4)))
    if kind == "q_over_r_1e4":     # the edges of the plain variant's range
        return GR.random_spd(rng, N, 3, 1e-1, 1e0), GR.random_spd(rng, N, 4, 1e-5, 1e-4)
    if kind == "r_over_q_100":
        return GR.random_spd(rng, N, 3, 1e-3, 1e-2), GR.random_spd(rng, N, 4, 1e-1, 1e0)
    raise ValueError(kind)


def _lowpassed(S, alpha):
    out = S.copy()
    y = np.zeros_like(S[0, 3:9])
    for t in range(S.shape[0]):
        y = alpha * S[t, 3:9] + (1 - alpha) * y
        out[t, 3:9] = y
    return out


def _definition(S, ar, mr, dt, Q, R, alpha=None):
    """S [T,9,N], ar/mr [3,N] numpy float32; Q, R [N,k,k]."""
    S = S.astype(np.float64)
    if alpha is not None:
        S = _lowpassed(S, float(np.float32(alpha)))
    T = S.shape[0]
    return GR.replay_general(np.full(T, float(np.float32(dt)) * 1e9), S[:, 0:3], S[:, 3:6], S[:, 6:9],
                             ar.T.astype(np.float64), mr.T.astype(np.float64), _f32(Q), _f32(R))


def _run(S, ar, mr, dt, Q, R, wahba="qr2", **kw):
    st, traj, flips = B.replay(S, ar, mr, dt=dt, q=Q, r=R, wahba=wahba, store_trajectory=True, store_flips=True,
                               share_measurements=False, **kw)
    torch.cuda.synchronize()
    return st, traj, flips


def _check(st, traj, flips, ref, tag, exact_flips=True):
    """exact_flips: the launch settles float32 ties of the reference's sign rule in float64 (raw samples with the QR2
    solver, or a measurement stream); otherwise (low-pass, Jacobi; DESIGN.md section 8) a flip byte may differ from the
    definition only where the two largest squared vector components of its measurement are within 1e-5 |y|^2."""
    ang = O.quat_angle(traj.cpu().numpy().astype(np.float64), ref["X"])
    assert ang.max() <= 1e-5, (tag, ang.max())
    mism = flips.cpu().numpy().astype(bool) != ref["flips"]
    if exact_flips:
        assert not mism.any(), (tag, int(mism.sum()))
    else:
        sq = np.sort(ref["y"][..., 1:] ** 2, axis=-1)
        tie = sq[..., 2] - sq[..., 1] < 1e-5 * np.sum(ref["y"] ** 2, axis=-1)
        assert not (mism & ~tie).any(), (tag, int(mism.sum()), int(tie.sum()))
    P = st.covariance().cpu().numpy().astype(np.float64)
    assert np.abs(P - ref["P"]).max() <= 1e-4 * max(1.0, np.abs(ref["P"]).max()), tag
    return ang.max()


WAHBA_LPF = [("qr2", None), ("qr2", 0.3), ("jacobi", None), ("jacobi", 0.3), ("precomputed", None)]


@pytest.mark.parametrize("kind", ["full", "diag", "q_over_r_1e4", "r_over_q_100"])
@pytest.mark.parametrize("wahba,alpha", WAHBA_LPF)
def test_parity_seeded_600k_steps(cuda, kind, wahba, alpha):
    N, T = 600, 1000
    imu = make_imu(N, T, seed=41, sigma=0.01, device=cuda)
    Q, R = _matrices(kind, N)
    S, ar, mr = imu.streams, imu.acc_ref, imu.mag_ref
    Qd, Rd = torch.tensor(Q, device=cuda), torch.tensor(R, device=cuda)
    lpf = dict(lpf_alpha_acc=alpha, lpf_alpha_mag=alpha) if alpha is not None else {}
    Sm = B.measurement_stream(S, ar, mr)[0] if wahba == "precomputed" else S
    outs = {st: _run(Sm, ar, mr, imu.dt, Qd, Rd, wahba, staging=st, **lpf) for st in ("ldg", "tma")}
    a, b = outs["ldg"], outs["tma"]
    assert torch.equal(a[0].x, b[0].x) and torch.equal(a[0].p, b[0].p) and torch.equal(a[1], b[1]) and torch.equal(a[2], b[2])
    if alpha is not None:
        assert torch.equal(a[0].lpf, b[0].lpf)
    ref = _definition(S.cpu().numpy(), ar.cpu().numpy(), mr.cpu().numpy(), imu.dt, Q, R, alpha)
    _check(*b, ref, (kind, wahba, alpha), exact_flips=wahba != "jacobi" and alpha is None)


@pytest.mark.parametrize("tag", ["clean", "noisy"])
@pytest.mark.parametrize("kind", ["full", "diag"])
def test_parity_golden_trajectories(cuda, golden_traj, tag, kind):
    g = golden_traj
    S = torch.tensor(g[f"{tag}_streams"], dtype=torch.float32, device=cuda)
    ar = torch.tensor(g[f"{tag}_acc_ref"], dtype=torch.float32, device=cuda)
    mr = torch.tensor(g[f"{tag}_mag_ref"], dtype=torch.float32, device=cuda)
    N = S.shape[2]
    Q, R = _matrices(kind, N, seed=7)
    dt = float(g["dt"])
    ref = _definition(S.cpu().numpy(), ar.cpu().numpy(), mr.cpu().numpy(), dt, Q, R)
    for wahba in ("qr2", "jacobi"):
        for staging in ("ldg", "tma"):
            _check(*_run(S, ar, mr, dt, torch.tensor(Q, device=cuda), torch.tensor(R, device=cuda), wahba, staging=staging),
                   ref, (tag, kind, wahba, staging), exact_flips=wahba == "qr2")


def test_packed_staging_runs_the_scalar_tma_kernel(cuda):
    imu = make_imu(512, 200, seed=2, sigma=0.01, device=cuda)
    Q, R = (torch.tensor(m, device=cuda) for m in _matrices("full", 512))
    outs = [_run(imu.streams, imu.acc_ref, imu.mag_ref, imu.dt, Q, R, staging=s) for s in ("tma", "tma_packed", "auto")]
    for o in outs[1:]:
        assert torch.equal(o[0].x, outs[0][0].x) and torch.equal(o[0].p, outs[0][0].p) and torch.equal(o[1], outs[0][1])


def test_shared_matrices_equal_per_filter_copies(cuda):
    N = 384
    imu = make_imu(N, 300, seed=9, sigma=0.01, device=cuda)
    Q, R = _matrices("full", 1, seed=4)
    for staging in ("ldg", "tma"):
        for wahba in ("qr2", "precomputed"):
            S = B.measurement_stream(imu.streams, imu.acc_ref, imu.mag_ref)[0] if wahba == "precomputed" else imu.streams
            a = _run(S, imu.acc_ref, imu.mag_ref, imu.dt, Q[0], R[0], wahba, staging=staging)
            b = _run(S, imu.acc_ref, imu.mag_ref, imu.dt, torch.tensor(np.repeat(Q, N, 0), device=cuda),
                     torch.tensor(np.repeat(R, N, 0), device=cuda), wahba, staging=staging)
            assert torch.equal(a[0].x, b[0].x) and torch.equal(a[0].p, b[0].p) and torch.equal(a[1], b[1]) and torch.equal(a[2], b[2])
    # a scalar for one of the two is q I3 / r I4 as a matrix
    a = _run(imu.streams, imu.acc_ref, imu.mag_ref, imu.dt, Q[0], 0.05)
    b = _run(imu.streams, imu.acc_ref, imu.mag_ref, imu.dt, Q[0], 0.05 * np.eye(4))
    assert torch.equal(a[0].x, b[0].x) and torch.equal(a[0].p, b[0].p)


@pytest.mark.parametrize("wahba,alpha", WAHBA_LPF)
def test_chunked_equals_unchunked(cuda, wahba, alpha):
    N, T = 256, 300
    imu = make_imu(N, T, seed=12, sigma=0.01, device=cuda, keep_truth=True)
    truth = imu.q_true.permute(0, 2, 1).to(torch.float32).contiguous()
    Q, R = (torch.tensor(m, device=cuda) for m in _matrices("full", N))
    S = B.measurement_stream(imu.streams, imu.acc_ref, imu.mag_ref)[0] if wahba == "precomputed" else imu.streams
    lpf = dict(lpf_alpha_acc=alpha, lpf_alpha_mag=alpha) if alpha is not None else {}
    for staging in ("ldg", "tma"):
        full = _run(S, imu.acc_ref, imu.mag_ref, imu.dt, Q, R, wahba, staging=staging, truth=truth, **lpf)
        st, loss, trajs, flips = None, None, [], []
        for t0 in (0, 37, 160):
            t1 = {0: 37, 37: 160, 160: T}[t0]
            st, tr, fl = _run(S[t0:t1].contiguous(), imu.acc_ref, imu.mag_ref, imu.dt, Q, R, wahba, staging=staging, state=st,
                              truth=truth[t0:t1].contiguous(), loss=loss, keep_filter_frame=t1 < T, **lpf)
            loss = st.loss
            trajs.append(tr), flips.append(fl)
        assert torch.equal(st.x, full[0].x) and torch.equal(st.p, full[0].p) and torch.equal(st.loss, full[0].loss)
        assert torch.equal(torch.cat(trajs), full[1]) and torch.equal(torch.cat(flips), full[2])
        assert st.frame == "reference" and st.r == 1.0


def test_ragged_batch_equals_single_recordings(cuda):
    Ns, T = 128, 240
    imu = make_imu(Ns, T, seed=17, sigma=0.01, device=cuda)
    g = torch.Generator().manual_seed(5)
    lengths = torch.randint(0, T + 1, (Ns,), generator=g).int()
    dt = (0.005 + 0.01 * torch.rand((T, Ns), generator=g)).float()
    S = imu.streams.clone()
    for c in range(Ns):                           # samples and dt past a recording's end are never used
        S[int(lengths[c]):, :, c] = float("nan")
        dt[int(lengths[c]):, c] = float("nan")
    dt, lengths = dt.to(cuda), lengths.to(cuda)
    Q, R = (torch.tensor(m, device=cuda) for m in _matrices("full", Ns))
    for staging in ("ldg", "tma"):
        st, traj, flips = _run(S, imu.acc_ref, imu.mag_ref, dt, Q, R, staging=staging, lengths=lengths)
        for c in (0, 3, 64, 127):
            n = int(lengths[c])
            sl = slice(c, c + 1)
            one = B.replay(S[:n, :, sl].contiguous(), imu.acc_ref[:, sl].contiguous(), imu.mag_ref[:, sl].contiguous(),
                           dt=dt[:n, c].contiguous(), q=Q[sl], r=R[sl], staging="ldg", store_trajectory=True, store_flips=True)
            torch.cuda.synchronize()
            assert torch.equal(one[0].x, st.x[:, sl]) and torch.equal(one[0].p, st.p[:, sl])
            assert torch.equal(one[1], traj[:n, sl]) and torch.equal(one[2], flips[:n, sl])
            if n < T:                                 # held steps repeat the final state, flip byte 0
                assert torch.equal(traj[n:, c], st.x[:, c].expand(T - n, 4)) and int(flips[n:, c].sum()) == 0


def test_loss_matches_float64_recomputation(cuda):
    N, T = 256, 500
    imu = make_imu(N, T, seed=31, sigma=0.01, device=cuda, keep_truth=True)
    truth = imu.q_true.permute(0, 2, 1).to(torch.float32).contiguous()
    Q, R = _matrices("full", N)
    st, traj, _ = _run(imu.streams, imu.acc_ref, imu.mag_ref, imu.dt, torch.tensor(Q, device=cuda),
                       torch.tensor(R, device=cuda), truth=truth)
    ref = _definition(imu.streams.cpu().numpy(), imu.acc_ref.cpu().numpy(), imu.mag_ref.cpu().numpy(), imu.dt, Q, R)
    tq = truth.cpu().numpy().astype(np.float64)
    X = ref["X"]
    want = (np.sum(X * X, -1) * np.sum(tq * tq, -1) - np.sum(X * tq, -1) ** 2).sum(0)
    torch.testing.assert_close(st.loss.double().cpu(), torch.tensor(want), rtol=1e-3, atol=1e-9)


def test_guard_bands_untouched(cuda):
    GUARD, POISON = 4096, -12345.0

    def guarded(shape, dtype=torch.float32):
        n = int(np.prod(shape))
        buf = torch.full((n + 2 * GUARD,), POISON if dtype == torch.float32 else 77, dtype=dtype, device=cuda)
        return buf, buf[GUARD:GUARD + n].view(shape)

    def intact(buf, n):
        val = POISON if buf.dtype == torch.float32 else 77
        return bool((buf[:GUARD] == val).all() and (buf[GUARD + n:] == val).all())

    for N, T, staging in ((1000, 37, "tma"), (1000, 37, "ldg"), (130, 9, "auto"), (3, 2, "ldg"), (4, 1, "tma_packed")):
        imu = make_imu(N, T, seed=N + T, sigma=0.01, device=cuda, keep_truth=True)
        truth = imu.q_true.permute(0, 2, 1).to(torch.float32).contiguous()
        Q, R = (torch.tensor(m, device=cuda) for m in _matrices("full", N))
        bx, x = guarded((4, N)); bp, p = guarded((10, N)); bf, lpf = guarded((6, N))
        bt, traj = guarded((T, N, 4)); bloss, loss = guarded((N,))
        x.zero_(); x[0] = 1.0; p.zero_(); p[[0, 4, 7, 9]] = 1.0; lpf.zero_(); loss.zero_()
        st = B.ReplayState(x, p, 1.0, lpf)
        B.replay(imu.streams, imu.acc_ref, imu.mag_ref, dt=imu.dt, q=Q, r=R, state=st, out_traj=traj, truth=truth, loss=loss,
                 lpf_alpha_acc=0.2, lpf_alpha_mag=0.2, staging=staging)
        torch.cuda.synchronize()
        assert intact(bx, 4 * N) and intact(bp, 10 * N) and intact(bf, 6 * N) and intact(bt, T * N * 4) and intact(bloss, N)
        assert torch.isfinite(traj).all() and (traj != POISON).all() and (loss >= 0).all()


def test_host_rules(cuda):
    imu = make_imu(8, 4, seed=1, sigma=0.01, device=cuda)
    Q, R = _matrices("full", 8)
    Qd, Rd = torch.tensor(Q, device=cuda), torch.tensor(R, device=cuda)
    args = (imu.streams, imu.acc_ref, imu.mag_ref)
    with pytest.raises(ValueError, match="innovation"):
        B.replay(*args, dt=imu.dt, q=Qd, r=Rd, innovation=True)
    with pytest.raises(ValueError, match="gate"):
        B.replay(*args, dt=imu.dt, q=Qd, r=Rd, gate=16.0)
    with pytest.raises(ValueError, match="precise"):
        B.replay(*args, dt=imu.dt, q=Qd, r=Rd, precise_state=True)
    with pytest.raises(ValueError, match="positive definite"):
        B.replay(*args, dt=imu.dt, q=Qd, r=np.diag([1.0, 1.0, 1.0, -1.0]))
    # a state moves between the scaled (P/r) and the unscaled form as the calls need
    st, _, _ = B.replay(*args, dt=imu.dt, q=1e-2, r=0.1)
    P0 = st.covariance()
    B.replay(imu.streams[:0], imu.acc_ref, imu.mag_ref, dt=imu.dt, q=Qd, r=Rd, state=st)
    assert st.r == 1.0 and torch.allclose(st.covariance(), P0, rtol=1e-6, atol=0)
    B.replay(imu.streams[:0], imu.acc_ref, imu.mag_ref, dt=imu.dt, q=1e-2, r=0.1, state=st)
    assert st.r == 0.1 and torch.allclose(st.covariance(), P0, rtol=1e-6, atol=0)
