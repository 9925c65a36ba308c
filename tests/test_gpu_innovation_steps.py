"""Per-step innovation output on the device (posekf_replay_innovation_steps_f32 / replay(out_innovation=...)): the terms
against the float64 definitions along the same trajectory on every staging, the sum identity with innov_acc, every
other output bit-identical to the same launch without the output, bitwise agreement across stagings, chunks and the
recordings of a ragged batch, the gate's decisions against plane 0, and guard bands around the output."""
import math

import numpy as np
import pytest
import torch

from poseestimationkf_b200 import batched as B
from poseestimationkf_b200 import workloads as W
from poseestimationkf_b200.synth import add_disturbances, make_imu
from tests import gating_ref as GR
from tests import innovation_ref as IR
from tests import innovation_tangent_ref as TR

pytestmark = pytest.mark.gpu

GAMMA = B.GATE_CHI2_3_999
PATHS = [(w, s) for w in ("qr2", "jacobi", "precomputed") for s in ("ldg", "tma", "tma_packed")
         if not (w == "jacobi" and s == "tma_packed")]
# Per-step error bar (the f5/f6 bar of the sums, applied per step), relative to |NIS_t| + |ln det S~_t| + dof |ln r|:
# ln det S_t = dof ln r + ln det S~_t is a sum of terms of that size and can itself be near 0 (r < 1), where |NIS_t| +
# |ln det S_t| would measure float32 rounding of its parts against a vanishing total.  The NIS of the Q >> R filters
# (q/r > 1e4, the exception of the f5 sums) is reported apart; against this scale it needs no bar of its own.
RTOL = 1e-4


def _lowpassed(S, alpha):
    out = S.copy()
    y = np.zeros_like(S[0, 3:9])
    for t in range(S.shape[0]):
        y = alpha * S[t, 3:9] + (1 - alpha) * y
        out[t, 3:9] = y
    return out


def _tunings(N, device, precise):
    if not precise:
        q = torch.logspace(-1, 1, N, device=device); r = torch.logspace(0.5, -1.5, N, device=device)
    else:
        q = torch.where(torch.arange(N, device=device) % 2 == 0, 1e-3, 1e3).float()
        r = torch.where(torch.arange(N, device=device) % 2 == 0, 1e3, 1e-3).float()
    return q.contiguous(), r.contiguous()


def _ref_terms(imu, q, r, model, alpha=None):
    S = imu.streams.cpu().numpy().astype(np.float64)
    if alpha is not None:
        S = _lowpassed(S, float(np.float32(alpha)))
    T = S.shape[0]
    fn = IR.replay_innovation if model == "full" else TR.replay_tangent
    ref = fn(np.full(T, float(np.float32(imu.dt)) * 1e9), S[:, 0:3], S[:, 3:6], S[:, 6:9], imu.acc_ref.cpu().numpy().T,
             imu.mag_ref.cpu().numpy().T, q.cpu().numpy().astype(np.float64), r.cpu().numpy().astype(np.float64))
    return ref["nis"], ref["logdet"]


def _steps(streams, ar, mr, dt, n_filters=None, **kw):
    T, _, Ns = streams.shape
    out = torch.full((2, T, n_filters or Ns), float("nan"), device=streams.device)
    st, traj, flips = B.replay(streams, ar, mr, dt=dt, n_filters=n_filters, out_innovation=out, **kw)
    torch.cuda.synchronize()
    return st, traj, flips, out


def _scale(nis, logdet, r, dof):
    lr = dof * np.abs(np.log(np.asarray(r, dtype=np.float64)))
    return np.abs(nis) + np.abs(logdet - lr * np.sign(np.log(r))) + lr


def _errors(out, nis, logdet, q, r, dof):
    got = out.double().cpu().numpy()
    scale = _scale(nis, logdet, r.double().cpu().numpy()[None, :], dof)
    qr = (q / r).cpu().numpy()[None, :] > 1e4
    e_ld = np.abs(got[1] - logdet) / scale
    e_nis = np.abs(got[0] - nis) / scale
    return float(e_ld.max()), float(np.where(qr, 0.0, e_nis).max()), float(np.where(qr, e_nis, 0.0).max())


@pytest.mark.parametrize("precise", [False, True])
@pytest.mark.parametrize("model", ["full", "tangent"])
def test_terms_match_definition_every_path(cuda, precise, model):
    N, T = 256, 200
    imu = make_imu(N, T, seed=21, sigma=0.01, device=cuda)
    q, r = _tunings(N, cuda, precise)
    runs = [(w, s, None) for w, s in PATHS] + [(w, s, 0.3) for w in ("qr2", "jacobi") for s in ("ldg", "tma", "tma_packed")
                                              if not (w == "jacobi" and s == "tma_packed")]
    refs = {a: _ref_terms(imu, q, r, model, a) for a in (None, 0.3)}
    worst = [0.0, 0.0, 0.0]
    for wahba, staging, alpha in runs:
        streams = imu.streams if wahba != "precomputed" else B.measurement_stream(imu.streams, imu.acc_ref, imu.mag_ref)[0]
        lp = dict(lpf_alpha_acc=alpha, lpf_alpha_mag=alpha) if alpha is not None else {}
        _, _, _, out = _steps(streams, imu.acc_ref, imu.mag_ref, imu.dt, q=q, r=r, precise_state=precise, wahba=wahba,
                              staging=staging, allow_imprecise=True, innovation_model=model, **lp)
        e = _errors(out, *refs[alpha], q, r, 4 if model == "full" else 3)
        worst = [max(a, b) for a, b in zip(worst, e)]
        assert e[0] <= RTOL and e[1] <= RTOL and e[2] <= RTOL, (wahba, staging, alpha, e)
    print(f"per-step {model} terms, precise={precise}: max relative error ln det {worst[0]:.3e}, NIS {worst[1]:.3e}, "
          f"NIS at q/r > 1e4 {worst[2]:.3e}")


@pytest.mark.parametrize("precise", [False, True])
@pytest.mark.parametrize("model", ["full", "tangent"])
def test_sum_of_terms_is_innov_acc(cuda, precise, model):
    """sum_t out[k][t] (float64) against innov_acc[k] within the float32 recursive-summation bound
    (T - 1) u sum_t |term_t| (u = 2^-24), plus u |NIS_t| per step for the rounding of the fused NIS product."""
    N, T = 512, 1000
    imu = make_imu(N, T, seed=4, sigma=0.01, device=cuda)
    q, r = _tunings(N, cuda, precise)
    st, _, _, out = _steps(imu.streams, imu.acc_ref, imu.mag_ref, imu.dt, q=q, r=r, precise_state=precise,
                           allow_imprecise=True, innovation=True, innovation_model=model)
    o = out.double()
    u = 2.0 ** -24
    bound = T * u * o.abs().sum(1) + 1e-30
    err = (o.sum(1) - st.innov.double()).abs()
    assert (err <= bound).all(), float((err / bound).max())
    print(f"sum identity {model}, precise={precise}: max |error| / bound {float((err / bound).max()):.3f}")


def _all(st, traj, flips, og=None):
    return dict(x=st.x, p=st.p, x_lo=st.x_lo, lpf=st.lpf, innov=st.innov, loss=st.loss, traj=traj, flips=flips,
                gate_count=st.gate_count, gated=og)


def _bitwise(a, b):
    for k in a:
        if a[k] is None or b[k] is None:
            assert a[k] is None and b[k] is None, k
        else:
            assert torch.equal(a[k].contiguous().view(torch.uint8), b[k].contiguous().view(torch.uint8)), k


@pytest.mark.parametrize("wahba,staging", PATHS)
@pytest.mark.parametrize("precise", [False, True])
@pytest.mark.parametrize("gate", [None, GAMMA])
def test_other_outputs_bit_identical(cuda, wahba, staging, precise, gate):
    N, T = 512, 300
    imu = make_imu(N, T, seed=5, sigma=0.01, dt=0.01, keep_truth=True)
    add_disturbances(imu.streams, seed=1, n_mag=2, length=(20, 60), margin=(40, 60))
    S, ar, mr = imu.streams.to(cuda), imu.acc_ref.to(cuda), imu.mag_ref.to(cuda)
    if wahba == "precomputed":
        S = B.measurement_stream(S, ar, mr)[0]
    truth = imu.q_true.permute(0, 2, 1).float().contiguous().to(cuda)
    q, r = (7.9e-6, 1e-4) if not precise else (1e-3, 1e3)
    lpfs = [dict()] if wahba == "precomputed" else [dict(), dict(lpf_alpha_acc=0.3, lpf_alpha_mag=0.3)]
    for lp in lpfs:
        for model, innov in (("tangent", True), ("full", True), ("tangent", None)):
            kw = dict(dt=imu.dt, q=q, r=r, wahba=wahba, staging=staging, precise_state=precise, allow_imprecise=True,
                      store_trajectory=True, store_flips=True, truth=truth, innovation=innov, innovation_model=model,
                      gate=gate, **lp)
            og_a = torch.zeros((T, N), dtype=torch.uint8, device=cuda) if gate is not None else None
            og_b = torch.zeros((T, N), dtype=torch.uint8, device=cuda) if gate is not None else None
            a = B.replay(S, ar, mr, out_gated=og_a, **kw)
            st, traj, flips, out = _steps(S, ar, mr, out_gated=og_b, **kw)
            _bitwise(_all(*a, og_a), _all(st, traj, flips, og_b))
            assert torch.isfinite(out).all()


@pytest.mark.parametrize("wahba", ["qr2", "jacobi", "precomputed"])
def test_stagings_and_chunks_bitwise(cuda, wahba):
    N, T = 768, 300
    imu = make_imu(N, T, seed=8, sigma=0.01, device=cuda)
    S = imu.streams if wahba != "precomputed" else B.measurement_stream(imu.streams, imu.acc_ref, imu.mag_ref)[0]
    q, r = _tunings(N, cuda, False)
    outs = []
    for staging in ("ldg", "tma", "tma_packed"):
        if wahba == "jacobi" and staging == "tma_packed":
            continue
        outs.append(_steps(S, imu.acc_ref, imu.mag_ref, imu.dt, q=q, r=r, wahba=wahba, staging=staging,
                           innovation_model="tangent", gate=GAMMA)[3])
    for o in outs[1:]:
        assert torch.equal(o.view(torch.int32), outs[0].view(torch.int32))
    # chunked: each chunk writes its slice of one full-length buffer
    full = torch.full((2, T, N), float("nan"), device=cuda)
    st = None
    bounds = [(0, 64), (64, 65), (65, 200), (200, T)]
    for i, (t0, t1) in enumerate(bounds):
        st, _, _ = B.replay(S[t0:t1], imu.acc_ref, imu.mag_ref, dt=imu.dt, q=q, r=r, state=st, wahba=wahba,
                            innovation_model="tangent", gate=GAMMA, gate_count=None if st is None else st.gate_count,
                            keep_filter_frame=i + 1 < len(bounds), out_innovation=full[:, t0:t1])
    torch.cuda.synchronize()
    assert torch.equal(full.view(torch.int32), outs[0].view(torch.int32))


def test_ragged_batch_each_recording_alone_and_held_zero(cuda):
    Ns, T = 8, 240
    imu = make_imu(Ns, T, seed=12, sigma=0.01, device=cuda)
    lengths = torch.tensor([240, 17, 0, 100, 239, 1, 64, 128], dtype=torch.int32, device=cuda)
    g = torch.Generator(device=cuda).manual_seed(3)
    dt = (0.01 * (1 + 0.2 * torch.rand((T, Ns), generator=g, device=cuda))).float().contiguous()
    for model in ("full", "tangent"):
        st, _, _, out = _steps(imu.streams, imu.acc_ref, imu.mag_ref, dt, q=1.0, r=0.1, lengths=lengths,
                               innovation=True, innovation_model=model)
        for c in range(Ns):
            L = int(lengths[c])
            assert (out[:, L:, c] == 0).all() and not torch.signbit(out[:, L:, c]).any()
            if L == 0:
                continue
            sl = slice(c, c + 1)
            _, _, _, alone = _steps(imu.streams[:L, :, sl].contiguous(), imu.acc_ref[:, sl].contiguous(),
                                    imu.mag_ref[:, sl].contiguous(), dt[:L, c].contiguous(), q=1.0, r=0.1,
                                    innovation_model=model)
            assert torch.equal(out[:, :L, c].view(torch.int32), alone[:, :, 0].view(torch.int32)), c
        # windows: the whole of each recording is its innovation_nll
        bounds = torch.stack((torch.zeros_like(lengths), lengths), 1)
        nll, _ = W.window_innovation_nll(out, bounds, 3 if model == "tangent" else 4)
        want, _ = B.innovation_nll(st, lengths)
        assert torch.allclose(nll[0], want, rtol=1e-5, atol=1e-3)


@pytest.mark.parametrize("precise", [False, True])
def test_gate_decisions_follow_plane_zero(cuda, precise):
    N, T = 64, 1500
    imu = make_imu(N, T, seed=5, sigma=0.01, dt=0.01)
    add_disturbances(imu.streams, seed=1, n_mag=3, length=(100, 300), margin=(200, 300))
    S, ar, mr = imu.streams.to(cuda), imu.acc_ref.to(cuda), imu.mag_ref.to(cuda)
    q, r = (7.9e-6, 1e-4) if not precise else (1e-3, 1e3)
    og = torch.zeros((T, N), dtype=torch.uint8, device=cuda)
    st, _, _, out = _steps(S, ar, mr, imu.dt, q=q, r=r, precise_state=precise, allow_imprecise=True,
                           innovation_model="tangent", gate=GAMMA, out_gated=og)
    nis = out[0].double()
    tie = (nis / GAMMA - 1.0).abs() < 1e-6
    assert not ((og.bool() != (nis > GAMMA)) & ~tie).any()
    assert int(st.gate_count.sum()) == int(og.sum())
    if not precise:
        assert og.any()
    # and against the float64 definition along the same decisions
    Sd = imu.streams.numpy().astype(np.float64)
    ref = GR.replay_gated(np.full(T, float(np.float32(imu.dt)) * 1e9), Sd[:, 0:3], Sd[:, 3:6], Sd[:, 6:9],
                          imu.acc_ref.numpy().T.astype(np.float64), imu.mag_ref.numpy().T.astype(np.float64),
                          float(np.float32(q)), float(np.float32(r)), GAMMA, decisions=og.bool().cpu().numpy())
    got = out.double().cpu().numpy()
    scale = _scale(ref["nis"], ref["logdet"], float(np.float32(r)), 3)
    e = max(float((np.abs(got[0] - ref["nis"]) / scale).max()), float((np.abs(got[1] - ref["logdet"]) / scale).max()))
    assert e <= RTOL, e
    # gamma = +inf gives the ungated bits
    a = _steps(S, ar, mr, imu.dt, q=q, r=r, precise_state=precise, allow_imprecise=True, innovation_model="tangent",
               gate=math.inf, innovation=True)
    b = _steps(S, ar, mr, imu.dt, q=q, r=r, precise_state=precise, allow_imprecise=True, innovation_model="tangent",
               innovation=True)
    assert torch.equal(a[3].view(torch.int32), b[3].view(torch.int32))
    _bitwise(_all(*a[:3]), dict(_all(*b[:3]), gate_count=a[0].gate_count))


@pytest.mark.parametrize("staging", ["ldg", "tma", "tma_packed", "auto"])
def test_no_out_of_bounds_writes(cuda, staging):
    """A 300-filter launch (the last packed CTA of 256 has lanes past N) writes exactly its [2][T][N] slots of a buffer
    with guard bands before, between and after the planes."""
    N, T, pad, gap = 300, 70, 1024, 333
    imu = make_imu(N, T, seed=2, sigma=0.01, device=cuda)
    for lengths in (None, torch.randint(0, T + 1, (N,), dtype=torch.int32, device=cuda)):
        for kw in (dict(), dict(gate=GAMMA), dict(lpf_alpha_acc=0.2, lpf_alpha_mag=0.2)):
            canary = -12345.0
            buf = torch.full((pad + 2 * T * N + gap + pad,), canary, device=cuda)
            plane = T * N + gap
            out = buf[pad:pad + 2 * plane].view(2, plane)[:, :T * N].view(2, T, N)
            assert out.stride(0) == plane
            B.replay(imu.streams, imu.acc_ref, imu.mag_ref, dt=imu.dt, q=1.0, r=0.1, staging=staging, lengths=lengths,
                     innovation_model="tangent", out_innovation=out, **kw)
            torch.cuda.synchronize()
            assert (buf[:pad] == canary).all() and (buf[-pad:] == canary).all()
            assert (buf[pad + T * N:pad + plane] == canary).all()
            assert (out != canary).all() and torch.isfinite(out).all()


def test_empty_launch(cuda):
    imu = make_imu(8, 10, seed=2, sigma=0.01, device=cuda)
    st, _, _ = B.replay(imu.streams[:0], imu.acc_ref, imu.mag_ref, dt=imu.dt, innovation_model="tangent",
                        out_innovation=torch.empty((2, 0, 8), device=cuda))
    ref, _, _ = B.replay(imu.streams[:0], imu.acc_ref, imu.mag_ref, dt=imu.dt)
    assert torch.equal(st.x, ref.x) and torch.equal(st.p, ref.p)


def test_general_matrices_refused(cuda):
    imu = make_imu(8, 10, seed=2, sigma=0.01, device=cuda)
    with pytest.raises(ValueError, match="per-step innovation"):
        B.replay(imu.streams, imu.acc_ref, imu.mag_ref, dt=imu.dt, q=np.eye(3), r=0.1 * np.eye(4),
                 out_innovation=torch.zeros((2, 10, 8), device=cuda))
    with pytest.raises(ValueError):
        B.replay(imu.streams, imu.acc_ref, imu.mag_ref, dt=imu.dt, out_innovation=torch.zeros((2, 10, 8), device=cuda).double())
