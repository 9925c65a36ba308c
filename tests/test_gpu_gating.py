"""Innovation gate on the device (posekf_replay_gated_f32 / replay(gate=...)): the gate at +inf against the ungated
launch bit for bit, the gate decisions, trajectory and covariance against the float64 definition (tests/gating_ref.py) on
a disturbed scenario, pure prediction at gate 0, bitwise properties across stagings, chunks and batches, guard bands
around the new outputs, and the accuracy gain on disturbed data."""
import math

import numpy as np
import pytest
import torch

from poseestimationkf_b200 import batched as B
from poseestimationkf_b200.synth import add_disturbances, make_imu
from tests import gating_ref as GR

pytestmark = pytest.mark.gpu

GAMMA = B.GATE_CHI2_3_999
PATHS = [(w, s) for w in ("qr2", "jacobi", "precomputed") for s in ("ldg", "tma", "tma_packed")
         if not (w == "jacobi" and s == "tma_packed")]


def _scenario(cuda, N=16, T=1500, n_mag=3, seed=5):
    """The disturbed scenario: sigma = 0.01 data, 3 magnetometer disturbances per recording (100-300 steps each at
    T = 1500; shorter recordings get proportionally shorter ones)."""
    imu = make_imu(N, T, seed=seed, sigma=0.01, dt=0.01, keep_truth=True)
    f = min(1.0, T / 1500)
    mask = add_disturbances(imu.streams, seed=1, n_mag=n_mag, length=(int(100 * f), int(300 * f)),
                            margin=(int(200 * f), int(300 * f)))
    dev = torch.device(cuda)
    return imu, mask, imu.streams.to(dev), imu.acc_ref.to(dev), imu.mag_ref.to(dev)


def _lowpassed(S, alpha):
    out = S.copy()
    y = np.zeros_like(S[0, 3:9])
    for t in range(S.shape[0]):
        y = alpha * S[t, 3:9] + (1 - alpha) * y
        out[t, 3:9] = y
    return out


def _ref(imu, q, r, gamma, decisions=None, alpha=None):
    S = imu.streams.cpu().numpy().astype(np.float64)
    if alpha is not None:
        S = _lowpassed(S, float(np.float32(alpha)))
    T = S.shape[0]
    return GR.replay_gated(np.full(T, float(np.float32(imu.dt)) * 1e9), S[:, 0:3], S[:, 3:6], S[:, 6:9],
                           imu.acc_ref.cpu().numpy().T.astype(np.float64), imu.mag_ref.cpu().numpy().T.astype(np.float64),
                           float(np.float32(q)), float(np.float32(r)), gamma, decisions)


def _run(streams, ar, mr, dt, wahba="qr2", **kw):
    if wahba == "precomputed":
        streams = B.measurement_stream(streams, ar, mr)[0]
    T, _, N = streams.shape
    og = torch.full((T, kw.get("n_filters") or N), 7, dtype=torch.uint8, device=streams.device) if kw.pop("gated", True) else None
    if kw.get("gate") is None:
        og = None
    st, traj, flips = B.replay(streams, ar, mr, dt=dt, wahba=wahba, out_gated=og, **kw)
    torch.cuda.synchronize()
    return st, traj, flips, og


def _same(a, b):
    return a is None and b is None or torch.equal(a.view(torch.uint8) if a.dtype != torch.uint8 else a,
                                                  b.view(torch.uint8) if b.dtype != torch.uint8 else b)


def _outputs(st, traj, flips):
    return dict(x=st.x, p=st.p, x_lo=st.x_lo, lpf=st.lpf, innov=st.innov, loss=st.loss, traj=traj, flips=flips)


# ---- the gate at +inf is the ungated launch --------------------------------------------------------------------------
@pytest.mark.parametrize("wahba,staging", PATHS)
@pytest.mark.parametrize("precise", [False, True])
def test_infinite_gate_is_bit_identical(cuda, wahba, staging, precise):
    imu, _, S, ar, mr = _scenario(cuda, N=512, T=300)
    q, r = (7.9e-6, 1e-4) if not precise else (1e-3, 1e3)
    truth = imu.q_true.permute(0, 2, 1).float().contiguous().to(S.device)
    lpfs = [dict()] if wahba == "precomputed" else [dict(), dict(lpf_alpha_acc=0.3, lpf_alpha_mag=0.3)]
    for lpf in lpfs:
        for innov in (None, "full", "tangent"):
            kw = dict(q=q, r=r, precise_state=precise, staging=staging, store_trajectory=True, store_flips=True, truth=truth,
                      innovation=True if innov else None, innovation_model=innov or "full", allow_imprecise=True, **lpf)
            a = _run(S, ar, mr, imu.dt, wahba, gate=math.inf, **kw)
            b = _run(S, ar, mr, imu.dt, wahba, **kw)
            for k, v in _outputs(*a[:3]).items():
                assert _same(v, _outputs(*b[:3])[k]), (k, lpf, innov)
            assert int(a[0].gate_count.sum()) == 0 and int(a[3].sum()) == 0


def test_infinite_gate_ragged_batch_and_sweep(cuda):
    imu, _, S, ar, mr = _scenario(cuda, N=256, T=300)
    T, _, Ns = S.shape
    lengths = torch.randint(0, T + 1, (Ns,), generator=torch.Generator().manual_seed(3)).int().to(S.device)
    dt = torch.full((T, Ns), imu.dt, device=S.device)
    for staging in ("ldg", "tma", "tma_packed"):
        for innov in (None, "full", "tangent"):
            kw = dict(q=7.9e-6, r=1e-4, staging=staging, lengths=lengths, store_trajectory=True, store_flips=True,
                      innovation=True if innov else None, innovation_model=innov or "full")
            a = _run(S, ar, mr, dt, gate=math.inf, **kw)
            b = _run(S, ar, mr, dt, **kw)
            for k, v in _outputs(*a[:3]).items():
                assert _same(v, _outputs(*b[:3])[k]), (staging, innov, k)
    # the mixed plain / precise sweep
    N = 4 * Ns
    q = torch.logspace(-6, -2, N, device=S.device); r = torch.logspace(-4, 0, N, device=S.device).flip(0).contiguous()
    a = _run(S, ar, mr, imu.dt, gate=math.inf, q=q, r=r, n_filters=N, share_measurements=False, innovation=True,
             innovation_model="tangent", gated=False)
    b = _run(S, ar, mr, imu.dt, q=q, r=r, n_filters=N, share_measurements=False, innovation=True, innovation_model="tangent")
    assert torch.equal(a[0].x, b[0].x) and torch.equal(a[0].p, b[0].p) and torch.equal(a[0].innov, b[0].innov)


# ---- against the float64 definition ----------------------------------------------------------------------------------
def _check_against_definition(imu, st, traj, flips, og, q, r, gamma, alpha=None, tag=""):
    gated = og.cpu().numpy().astype(bool)
    ref = _ref(imu, q, r, gamma, decisions=gated, alpha=alpha)
    # the device's decisions are NIS3 > gamma of the definition along the same trajectory, except at threshold ties
    tie = np.abs(ref["nis"] / gamma - 1.0) < 1e-3
    wrong = (gated != (ref["nis"] > gamma)) & ~tie
    assert not wrong.any(), (tag, int(wrong.sum()))
    got = traj.cpu().numpy()
    ang = GR.angle(got, ref["X"])
    assert ang.max() <= 1e-5, (tag, ang.max())
    assert (np.sum(got * ref["X"], axis=-1) > 0).all(), tag
    assert np.array_equal(flips.cpu().numpy().astype(bool), ref["flips"]), tag
    Pd = ref["P"]
    P = st.covariance().cpu().numpy()
    rel = np.linalg.norm(P - Pd, axis=(1, 2)) / np.linalg.norm(Pd, axis=(1, 2))
    assert rel.max() <= 1e-4, (tag, rel.max())
    assert torch.equal(st.gate_count.cpu(), og.sum(0, dtype=torch.int32).cpu())
    return int(tie.sum()), float(gated.mean()), float(ang.max())


@pytest.mark.parametrize("wahba,staging", PATHS)
@pytest.mark.parametrize("precise", [False, True])
def test_decisions_trajectory_and_covariance_match_definition(cuda, wahba, staging, precise):
    imu, mask, S, ar, mr = _scenario(cuda)
    q, r = (7.9e-6, 1e-4) if not precise else (7.9e-6, 1e-3)
    st, traj, flips, og = _run(S, ar, mr, imu.dt, wahba, q=q, r=r, gate=GAMMA, precise_state=precise, staging=staging,
                               store_trajectory=True, store_flips=True)
    ties, frac, worst = _check_against_definition(imu, st, traj, flips, og, q, r, GAMMA, tag=(wahba, staging, precise))
    print(f"{wahba}/{staging}/precise={precise}: {frac:.1%} of steps gated, {ties} threshold ties excluded, "
          f"max angle {worst:.2e} rad")
    assert og.cpu().numpy().astype(bool)[mask.numpy()].mean() > 0.5


@pytest.mark.parametrize("wahba,staging", [p for p in PATHS if p[0] != "precomputed"])   # (a measurement stream has
@pytest.mark.parametrize("precise", [False, True])                                         #  no low-pass stage)
def test_lowpass_against_definition(cuda, wahba, staging, precise):
    imu, _, S, ar, mr = _scenario(cuda, T=800)
    q, r = (7.9e-6, 1e-4) if not precise else (7.9e-6, 1e-3)
    st, traj, flips, og = _run(S, ar, mr, imu.dt, wahba, q=q, r=r, gate=GAMMA, precise_state=precise, staging=staging,
                               store_trajectory=True, store_flips=True, lpf_alpha_acc=0.5, lpf_alpha_mag=0.5)
    ties, frac, worst = _check_against_definition(imu, st, traj, flips, og, q, r, GAMMA, alpha=0.5,
                                                  tag=(wahba, staging, precise))
    print(f"low-pass/{wahba}/{staging}/precise={precise}: {frac:.1%} gated, {ties} ties excluded, max angle {worst:.2e} rad")


@pytest.mark.parametrize("staging", ["ldg", "tma", "tma_packed"])
def test_zero_gate_is_pure_prediction(cuda, staging):
    imu, _, S, ar, mr = _scenario(cuda, N=64, T=500)
    q, r = 1e-3, 1e-2
    st, traj, flips, og = _run(S, ar, mr, imu.dt, q=q, r=r, gate=0.0, staging=staging, store_trajectory=True)
    ref = _ref(imu, q, r, 0.0)
    assert ref["gated"].all() and bool(og.bool().all())
    assert torch.equal(st.gate_count.cpu(), torch.full((64,), 500, dtype=torch.int32))
    assert GR.angle(traj.cpu().numpy(), ref["X"]).max() <= 1e-5


# ---- bitwise properties ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precise", [False, True])
def test_stagings_chunks_and_batches_bitwise(cuda, precise):
    imu, _, S, ar, mr = _scenario(cuda, N=512, T=700)
    T, _, Ns = S.shape
    q, r = (7.9e-6, 1e-4) if not precise else (7.9e-6, 1e-3)
    kw = dict(q=q, r=r, gate=GAMMA, precise_state=precise, store_trajectory=True, store_flips=True, innovation=True,
              innovation_model="tangent")
    runs = {s: _run(S, ar, mr, imu.dt, staging=s, **kw) for s in ("ldg", "tma", "tma_packed")}
    base = runs["tma_packed"]
    assert int(base[0].gate_count.sum()) > 0
    for s, run in runs.items():
        for k, v in _outputs(*run[:3]).items():
            assert _same(v, _outputs(*base[:3])[k]), (s, k)
        assert torch.equal(run[3], base[3]) and torch.equal(run[0].gate_count, base[0].gate_count), s
        assert torch.equal(run[0].gate_count, run[3].sum(0, dtype=torch.int32)), s
    # chunked (state in the filter frame between chunks, counts and sums carried) equals unchunked
    for staging in ("ldg", "tma_packed"):
        st = None
        trajs, gs = [], []
        for t0, t1 in ((0, 256), (256, 513), (513, T)):
            og = torch.empty((t1 - t0, Ns), dtype=torch.uint8, device=S.device)
            st, tr, _ = B.replay(S[t0:t1].contiguous(), ar, mr, dt=imu.dt, q=q, r=r, gate=GAMMA, precise_state=precise,
                                 staging=staging, state=st, keep_filter_frame=t1 < T, store_trajectory=True,
                                 innovation=True if st is None else st.innov, innovation_model="tangent",
                                 gate_count=None if st is None else st.gate_count, out_gated=og)
            trajs.append(tr); gs.append(og)
        assert torch.equal(torch.cat(trajs), base[1]) and torch.equal(torch.cat(gs), base[3]), staging
        assert torch.equal(st.x, base[0].x) and torch.equal(st.p, base[0].p) and torch.equal(st.innov, base[0].innov)
        assert torch.equal(st.gate_count, base[0].gate_count)
    # a ragged batch of recordings equals each recording replayed alone
    lengths = torch.randint(T // 2, T + 1, (Ns,), generator=torch.Generator().manual_seed(5)).int()
    dtc = torch.full((T, Ns), imu.dt)
    for c in range(Ns):
        dtc[lengths[c]:, c] = float("nan")
    Sn = S.clone()
    for c in range(Ns):
        Sn[lengths[c]:, :, c] = float("nan")
    for staging in ("ldg", "tma", "tma_packed"):
        stb, trb, _, ogb = _run(Sn, ar, mr, dtc.to(S.device), q=q, r=r, gate=GAMMA, precise_state=precise, staging=staging,
                                lengths=lengths.to(S.device), store_trajectory=True)
        assert torch.equal(stb.gate_count, ogb.sum(0, dtype=torch.int32))
        for c in range(0, Ns, 97):
            L = int(lengths[c])
            one = _run(S[:L, :, c:c + 1].contiguous(), ar[:, c:c + 1].contiguous(), mr[:, c:c + 1].contiguous(), imu.dt, q=q,
                       r=r, gate=GAMMA, precise_state=precise, staging="ldg", store_trajectory=True)
            assert torch.equal(stb.x[:, c], one[0].x[:, 0]) and torch.equal(stb.p[:, c], one[0].p[:, 0]), (staging, c)
            assert torch.equal(trb[:L, c], one[1][:, 0]) and torch.equal(ogb[:L, c], one[3][:, 0]), (staging, c)
            assert not ogb[L:, c].any() and int(stb.gate_count[c]) == int(one[0].gate_count[0]), (staging, c)


@pytest.mark.parametrize("staging", ["ldg", "tma", "tma_packed"])
@pytest.mark.parametrize("layout", ["aligned", "tail", "unaligned"])
def test_guard_bands(cuda, staging, layout):
    """gate_count and out_gated are written inside their bounds only.  "tail": N = 260, so the last packed CTA has lanes
    past N; "unaligned": gate_count only 4-byte and out_gated only 1-byte aligned, which the packed kernel cannot access
    (int2 / uchar2) -- such a launch runs the scalar TMA kernel, with the same results."""
    N = 256 if layout == "aligned" else 260
    imu, _, S, ar, mr = _scenario(cuda, N=N, T=400)
    T = S.shape[0]
    G = 64
    oc, of = (G + 1, G + N + 1) if layout == "unaligned" else (G, G + N)     # element offsets of the two views
    cnt = torch.full((N + 2 * G + 2,), -7, dtype=torch.int32, device=S.device)
    flags = torch.full(((T + 2) * N + 2 * G + 2,), 0xAB, dtype=torch.uint8, device=S.device)
    cnt[oc:oc + N] = 0
    og = flags[of:of + T * N].view(T, N)
    assert (og.data_ptr() % 2 == 1) == (layout == "unaligned") and (cnt[oc:].data_ptr() % 8 == 4) == (layout == "unaligned")
    st, _, _ = B.replay(S, ar, mr, dt=imu.dt, q=7.9e-6, r=1e-4, gate=GAMMA, staging=staging,
                        gate_count=cnt[oc:oc + N], out_gated=og)
    ref = _run(S, ar, mr, imu.dt, q=7.9e-6, r=1e-4, gate=GAMMA, staging="ldg")
    torch.cuda.synchronize()
    assert (cnt[:oc] == -7).all() and (cnt[oc + N:] == -7).all()
    assert (flags[:of] == 0xAB).all() and (flags[of + T * N:] == 0xAB).all()
    assert torch.equal(og, ref[3]) and torch.equal(cnt[oc:oc + N], ref[0].gate_count) and int(og.sum()) > 0
    assert torch.equal(st.x, ref[0].x) and torch.equal(st.p, ref[0].p)


# ---- accuracy on disturbed data --------------------------------------------------------------------------------------
def test_gate_cuts_the_error_on_disturbed_data(cuda):
    """The typical recording's error at least halves.  The RMS over all recordings need not: without a cap on consecutive
    rejections a recording whose prediction has drifted when a disturbance ends can stay locked out (DESIGN.md, f8), and
    a few such recordings dominate the RMS; it must not get worse."""
    imu, mask, S, ar, mr = _scenario(cuda, N=256)
    truth = imu.q_true.permute(0, 2, 1).numpy()          # [T,N,4]
    err = {}
    for gate in (None, GAMMA):
        st, traj, _, og = _run(S, ar, mr, imu.dt, q=7.9e-6, r=1e-4, gate=gate, store_trajectory=True)
        ang = np.degrees(GR.angle(traj.cpu().numpy(), truth))
        per_rec = np.sqrt(np.mean(ang ** 2, axis=0))
        err[gate] = (float(np.sqrt(np.mean(ang ** 2))), float(ang.max()), float(np.median(per_rec)))
    print(f"disturbed: ungated RMS {err[None][0]:.2f} deg / max {err[None][1]:.1f} deg / median recording "
          f"{err[None][2]:.2f} deg, gated RMS {err[GAMMA][0]:.2f} deg / max {err[GAMMA][1]:.1f} deg / median recording "
          f"{err[GAMMA][2]:.2f} deg")
    assert err[GAMMA][2] <= 0.5 * err[None][2]
    assert err[GAMMA][0] <= err[None][0]
