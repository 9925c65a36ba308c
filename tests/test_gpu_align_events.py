"""Alignment of raw event recordings on the device (posekf_align_events_f32 / logio.align_recordings): against the float64
definition (tests/align_ref.py) on asynchronous `make_events` batches, bit for bit against `B.preprocess` fed the
definition's brackets, every recording against its own one-recording alignment, stack_logs' padding, the replay of an
aligned batch end to end and in time chunks, and guard bands around every output."""
import numpy as np
import pytest
import torch

from oracle import ekf_oracle as O
from poseestimationkf_b200 import _lib, logio
from poseestimationkf_b200 import batched as B
from poseestimationkf_b200.synth import make_events, make_imu
from tests import align_ref as AR

pytestmark = pytest.mark.gpu


def _bits(t):
    return t.contiguous().view(torch.int32)


def _ragged_events(seed=5):
    # ragged durations, per-recording rates, one recording too short for the 100 initial events (length 0)
    dur = [6.0, 3.5, 5.0, 0.6, 4.2, 2.0, 5.5]
    rates = ([200.0, 150.0, 400.0, 200.0, 100.0, 250.0, 200.0], [100.0, 120.0, 50.0, 100.0, 200.0, 90.0, 100.0],
             [100.0, 60.0, 100.0, 100.0, 50.0, 110.0, 75.0])
    return make_events(len(dur), dur, rates=rates, jitter=0.3, sigma=0.01, seed=seed)


def test_matches_float64_definition(cuda):
    ev = _ragged_events()
    batch = logio.align_recordings(ev.recordings, device=cuda)
    ref = AR.align_events(ev.recordings)
    Ns = batch.streams.shape[2]
    assert batch.n_logs == len(ref) and Ns == 8
    L = batch.lengths.cpu().numpy()
    np.testing.assert_array_equal(L[:len(ref)], [a["length"] for a in ref])
    assert L[3] == 0 and L[len(ref):].sum() == 0 and L.max() == batch.streams.shape[0]
    S, dt = batch.streams.cpu().numpy(), batch.dt.cpu().numpy()
    ar, mr = batch.acc_ref.cpu().numpy(), batch.mag_ref.cpu().numpy()
    for c, a in enumerate(ref):
        n = a["length"]
        np.testing.assert_array_equal(dt[:n, c], a["dt"])                                  # bit-equal float32
        np.testing.assert_array_equal(S[:n, 0:3, c], a["streams"][:, 0:3].astype(np.float32))
        np.testing.assert_allclose(S[:n, 3:9, c], a["streams"][:, 3:9], atol=2e-6, rtol=0)
        np.testing.assert_allclose(ar[:, c], a["acc_ref"], atol=1e-7, rtol=0)
        np.testing.assert_allclose(mr[:, c], a["mag_ref"], atol=1e-7, rtol=0)


def test_references_equal_initial_values_and_streams_equal_preprocess(cuda):
    """The reference vectors are B.initial_values of the first 100 events and the streams B.preprocess of the
    definition's brackets, bit for bit: the alignment runs the same device functions."""
    ev = _ragged_events(seed=6)
    batch = logio.align_recordings(ev.recordings, device=cuda)
    for c, (rec, a) in enumerate(zip(ev.recordings, AR.align_events(ev.recordings))):
        n = a["length"]
        if n == 0:
            continue
        for e, got in ((rec.acc, batch.acc_ref), (rec.mag, batch.mag_ref)):
            m, _ = B.initial_values(torch.from_numpy(np.ascontiguousarray(e.v[:100, :, None])).to(cuda))
            assert torch.equal(_bits(got[:, c]), _bits(m[:, 0]))
        g = rec.gyro.v[a["first"]:a["first"] + n]
        prev = np.concatenate([rec.acc.v[a["j_acc"]], rec.mag.v[a["j_mag"]]], axis=1)
        nxt = np.concatenate([rec.acc.v[a["j_acc"] + 1], rec.mag.v[a["j_mag"] + 1]], axis=1)
        dev = lambda x: torch.from_numpy(np.ascontiguousarray(x[:, :, None], dtype=np.float32)).to(cuda)
        out, _ = B.preprocess(dev(g), dev(prev), dev(nxt), dev(AR.tspans(rec, a)))
        assert torch.equal(_bits(batch.streams[:n, :, c]), _bits(out[:, :, 0])), c


def test_each_recording_equals_its_own_alignment_and_padding(cuda):
    ev = _ragged_events(seed=7)
    batch = logio.align_recordings(ev.recordings, device=cuda)
    T = batch.streams.shape[0]
    for c, rec in enumerate(ev.recordings):
        one = logio.align_recordings([rec], device=cuda, pad_cols_to=1)
        n = int(one.lengths[0])
        assert n == int(batch.lengths[c])
        assert torch.equal(_bits(batch.streams[:n, :, c]), _bits(one.streams[:, :, 0]))
        assert torch.equal(_bits(batch.dt[:n, c]), _bits(one.dt[:, 0]))
        assert torch.equal(_bits(batch.acc_ref[:, c]), _bits(one.acc_ref[:, 0]))
        assert torch.equal(_bits(batch.mag_ref[:, c]), _bits(one.mag_ref[:, 0]))
    for c in range(batch.streams.shape[2]):
        n = int(batch.lengths[c])
        pad = batch.streams[n:, :, c]
        assert not batch.dt[n:, c].any()
        if n > 0:               # stack_logs: the last sample repeated
            assert torch.equal(_bits(pad), _bits(batch.streams[n - 1:n, :, c].expand(T - n, 9)))
        else:                   # stack_logs: gyro 0, the reference vectors as acc / mag
            assert not pad[:, 0:3].any()
            assert torch.equal(pad[:, 3:6], batch.acc_ref[:, c].expand(T, 3))
            assert torch.equal(pad[:, 6:9], batch.mag_ref[:, c].expand(T, 3))
    for c in (3, 7):            # too few events, and a padding column
        assert batch.acc_ref[:, c].tolist() == [0.0, 0.0, 1.0] and batch.mag_ref[:, c].tolist() == [1.0, 0.0, 0.0]


def _rms(x):
    return float(np.sqrt(np.mean(np.square(x))))


def test_end_to_end_replay_against_oracle(cuda):
    n_rec, dur = 16, 8.0
    ev = make_events(n_rec, dur, rates=(200.0, 100.0, 100.0), sigma=0.01, seed=11, keep_truth=True)
    batch = logio.align_recordings(ev.recordings, device=cuda)
    st, traj, _ = B.replay(batch.streams, batch.acc_ref, batch.mag_ref, dt=batch.dt, q=1.0, r=0.1, lengths=batch.lengths,
                           store_trajectory=True)
    traj = traj.cpu().numpy().astype(np.float64)
    err_gpu, err_ref, worst = [], [], 0.0
    for c, (rec, a) in enumerate(zip(ev.recordings, AR.align_events(ev.recordings))):
        n, f = a["length"], a["first"]
        S = a["streams"][:, :, None]                                             # [L,9,1]
        tg = rec.gyro.t_ns[f:f + n]
        dt_ns = np.diff(np.concatenate([[a["t_init"]], tg])).astype(np.float64)
        o = O.replay_batched(dt_ns, S[:, 0:3], S[:, 3:6], S[:, 6:9], a["acc_ref"][None], a["mag_ref"][None], 1.0,
                             float(np.float32(0.1)))
        worst = max(worst, float(O.quat_angle(traj[:n, c], o["X"][:, 0]).max()))
        truth = ev.truth[c][f:f + n]
        err_gpu.append(O.quat_angle(traj[:n, c], truth))
        err_ref.append(O.quat_angle(o["X"][:, 0], truth))
    assert worst < 1e-5, worst
    # sanity figure, not a bar: the same motion model sampled synchronously at 200 Hz
    imu = make_imu(n_rec, int(dur * 200), seed=11, sigma=0.01, dt=0.005, device=cuda, keep_truth=True)
    _, tr2, _ = B.replay(imu.streams, imu.acc_ref, imu.mag_ref, dt=imu.dt, q=1.0, r=0.1, store_trajectory=True)
    sync = O.quat_angle(tr2.cpu().numpy().astype(np.float64), imu.q_true.permute(0, 2, 1).cpu().numpy())
    print(f"\naligned events: RMS attitude error vs truth {_rms(np.concatenate(err_gpu)):.3e} rad (float64 oracle "
          f"{_rms(np.concatenate(err_ref)):.3e}); max |device - oracle| {worst:.2e} rad; synchronous make_imu "
          f"{_rms(sync):.3e} rad")


def test_window_chunks_replay_bit_identically(cuda):
    ev = make_events(12, [4.0, 3.0, 5.0, 2.5] * 3, rates=(200.0, 100.0, 100.0), sigma=0.01, seed=12)
    lb = logio.align_recordings(ev.recordings, device=cuda)
    T, chunk = lb.streams.shape[0], 128
    ref, traj, flips = B.replay(lb.streams, lb.acc_ref, lb.mag_ref, dt=lb.dt, q=1.0, r=0.1, lengths=lb.lengths,
                                store_trajectory=True, store_flips=True)
    st, trs, fls = None, [], []
    for t0 in range(0, T, chunk):
        w = lb.window(t0, t0 + chunk)
        st, tr, fl = B.replay(w.streams, w.acc_ref, w.mag_ref, dt=w.dt, q=1.0, r=0.1, lengths=w.lengths, state=st,
                              store_trajectory=True, store_flips=True, keep_filter_frame=t0 + chunk < T)
        trs.append(tr)
        fls.append(fl)
    assert torch.equal(_bits(st.x), _bits(ref.x)) and torch.equal(_bits(st.p), _bits(ref.p))
    assert torch.equal(_bits(torch.cat(trs)), _bits(traj)) and torch.equal(torch.cat(fls), flips)


@pytest.mark.parametrize("extra", [0, 37])
def test_guard_bands(cuda, extra):
    """Canaries around streams, dt, lengths and the references stay untouched, with T equal to the longest length and
    with T larger than every length (the extra rows then hold the padding)."""
    ev = _ragged_events(seed=8)
    ref = logio.align_recordings(ev.recordings, device=cuda)
    Ns, T = ref.streams.shape[2], ref.streams.shape[0] + extra
    recs = ev.recordings + [logio.RawRecording(*[logio.SensorEvents(np.zeros(0, np.int64), np.zeros((0, 3), np.float32))] * 3)]
    packed = []
    for name in ("gyro", "acc", "mag"):
        t, v, off = logio._pack_sensor([getattr(r, name) for r in recs], name)
        packed += [torch.from_numpy(a).to(cuda) for a in (t, v, off)]
    G = 64
    canary = -2.0 ** 100                # exact in float32

    def guarded(n, dtype=torch.float32):
        buf = torch.full((n + 2 * G,), canary if dtype == torch.float32 else -12345, dtype=dtype, device=cuda)
        return buf, buf[G:G + n]

    (sb, s), (db, d), (lb, ln), (ab, a), (mb, m) = (guarded(T * 9 * Ns), guarded(T * Ns), guarded(Ns, torch.int32),
                                                    guarded(3 * Ns), guarded(3 * Ns))
    with torch.cuda.device(cuda):
        rc = _lib.load().posekf_align_events_f32(Ns, 100, *[x.data_ptr() for x in packed], T, s.data_ptr(), d.data_ptr(),
                                                 ln.data_ptr(), a.data_ptr(), m.data_ptr(), B._stream())
    _lib.check(rc, "posekf_align_events_f32")
    torch.cuda.synchronize()
    for buf in (sb, db, lb, ab, mb):
        assert (buf[:G] == buf[0]).all() and (buf[-G:] == buf[0]).all() and float(buf[0]) in (canary, -12345)
    Tm = ref.streams.shape[0]
    s, d = s.view(T, 9, Ns), d.view(T, Ns)
    assert torch.equal(ln, ref.lengths)
    assert torch.equal(_bits(s[:Tm]), _bits(ref.streams)) and torch.equal(_bits(d[:Tm]), _bits(ref.dt))
    assert torch.equal(_bits(a.view(3, Ns)), _bits(ref.acc_ref)) and torch.equal(_bits(m.view(3, Ns)), _bits(ref.mag_ref))
    if extra:
        assert torch.equal(_bits(s[Tm:]), _bits(ref.streams[Tm - 1:Tm].expand(extra, 9, Ns))) and not d[Tm:].any()


def test_pooled_sweep_takes_an_aligned_batch(cuda):
    from poseestimationkf_b200 import workloads as WL
    ev = make_events(6, [3.0, 4.0, 2.0, 3.5, 2.5, 3.0], sigma=0.01, seed=13)
    b = logio.align_recordings(ev.recordings, device=cuda)
    w = WL.build_batch_sweep(b, grid=4, lo=-5.0, step=1.0)
    assert w.n_filters == 16 * b.streams.shape[2] and torch.equal(w.lengths, b.lengths)
    nll, nis = WL.pooled_innovation_surface(w, WL.run_c3(w, objective="innovation_tangent"))
    assert nll.shape == (4, 4) and torch.isfinite(nll).all() and torch.isfinite(nis).all()
