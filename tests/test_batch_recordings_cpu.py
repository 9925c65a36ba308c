"""A batch of recordings in one launch, the parts that need no GPU: `logio.stack_logs` and `LogBatch.window` on logs
written by `logio.write_log`, the argument rules of posekf_replay_batch_f32 and of `replay(lengths=...)`, the per-filter
step counts of `innovation_nll` and the pooled surface, and the per-lane time constants of the packed step (CPU build of
the header)."""
import atexit
import ctypes as C
import math
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest
import torch

from poseestimationkf_b200 import _lib
from poseestimationkf_b200 import batched as B
from poseestimationkf_b200 import logio
from poseestimationkf_b200 import workloads as WL

HERE = os.path.dirname(os.path.abspath(__file__))


def _unit(v):
    return v / np.linalg.norm(v, axis=-1, keepdims=True)


def write_recording(path, n_steps, seed, period_ns=10_000_000, jitter=0.2):
    """A log in the server's text format with `n_steps` samples and timestamps jittered by +-jitter of the period."""
    rng = np.random.default_rng(seed)
    t0 = 1_600_000_000_000_000_000 + int(rng.integers(0, 10**9))
    dts = np.rint(period_ns * (1.0 + jitter * rng.uniform(-1, 1, n_steps))).astype(np.int64)
    t_ns = t0 + np.cumsum(dts)
    gyro = rng.normal(0, 0.3, (n_steps, 3))
    acc = _unit(np.array([0.1, -0.2, 0.97]) + rng.normal(0, 0.01, (n_steps, 3)))
    mag = _unit(np.array([0.4, 0.0, -0.9165]) + rng.normal(0, 0.01, (n_steps, 3)))
    one = np.tile([1.0, 0.0, 0.0, 0.0], (n_steps, 1))
    logio.write_log(path, acc_0=acc[0], mag_0=mag[0], t0_ns=t0, t_ns=t_ns, gyro=gyro, mag_1=mag, acc_1=acc, x_k=one,
                    wahba_quart=one, q_gyro=one)
    return logio.read_log(path)


@pytest.fixture(scope="module")
def logs(tmp_path_factory):
    d = tmp_path_factory.mktemp("logs")
    return [write_recording(str(d / f"rec{k}.txt"), n, seed=k) for k, n in enumerate((37, 50, 12, 50, 1))]


def test_stack_logs_dt_is_each_recordings_own(logs):
    b = logio.stack_logs(logs, device="cpu")
    Tmax = max(lg.n_steps() for lg in logs)
    assert b.n_logs == 5 and b.streams.shape == (Tmax, 9, 8) and b.dt.shape == (Tmax, 8)
    assert b.acc_ref.shape == (3, 8) and b.mag_ref.shape == (3, 8)
    assert b.lengths.dtype == torch.int32 and b.lengths.tolist() == [37, 50, 12, 50, 1, 0, 0, 0]
    for c, lg in enumerate(logs):
        s, ar, mr, dt = lg.to_streams("cpu")
        T = lg.n_steps()
        assert torch.equal(b.dt[:T, c], dt)                        # bit for bit: same float64 differencing
        assert torch.equal(b.streams[:T, :, c], s[:, :, 0])
        assert torch.equal(b.acc_ref[:, c], ar[:, 0]) and torch.equal(b.mag_ref[:, c], mr[:, 0])
        # padding: the last sample repeated, dt = 0
        assert torch.equal(b.streams[T:, :, c], s[-1:, :, 0].expand(Tmax - T, 9))
        assert not b.dt[T:, c].any()
    assert len(set(b.dt[0, :5].tolist())) > 1                     # the recordings do not share a clock
    for c in range(5, 8):                                         # empty columns: finite, zero rate, zero dt
        assert torch.isfinite(b.streams[:, :, c]).all() and not b.streams[:, 0:3, c].any() and not b.dt[:, c].any()


def test_stack_logs_column_padding():
    d = tempfile.mkdtemp()
    try:
        lgs = [write_recording(os.path.join(d, f"r{k}.txt"), 5 + k, seed=10 + k) for k in range(4)]
        assert logio.stack_logs(lgs, device="cpu").streams.shape[2] == 4
        assert logio.stack_logs(lgs[:3], device="cpu", pad_cols_to=1).streams.shape[2] == 3
        assert logio.stack_logs(lgs[:3], device="cpu", pad_cols_to=8).lengths.tolist() == [5, 6, 7, 0, 0, 0, 0, 0]
    finally:
        shutil.rmtree(d)


def test_window_lengths_and_slices(logs):
    b = logio.stack_logs(logs, device="cpu")
    L = np.array(b.lengths.tolist())
    for t0, t1 in ((0, 12), (12, 37), (37, 50), (10, 11), (0, 50), (45, 50)):
        w = b.window(t0, t1)
        assert w.lengths.dtype == torch.int32
        assert w.lengths.tolist() == np.clip(L - t0, 0, t1 - t0).tolist()
        assert torch.equal(w.streams, b.streams[t0:t1]) and torch.equal(w.dt, b.dt[t0:t1])
        assert w.streams.is_contiguous() and w.dt.is_contiguous()
        assert w.acc_ref is b.acc_ref and w.n_logs == b.n_logs
    # chunk lengths add up to the recording lengths
    chunks = [b.window(t0, min(t0 + 16, 50)).lengths for t0 in range(0, 50, 16)]
    assert torch.equal(sum(chunks), b.lengths)


def _batch_call(lib, n=8, t=4, ns=8, model=0, wahba=0, staging=0, dt_cols=None, n_valid=None, streams=None, flags=0,
                innov=None, dt=None):
    return lib.posekf_replay_batch_f32(n, t, streams, ns, dt, 0, None, None, None, None, -1.0, -1.0, None, None, None, None,
                                       None, None, None, None, innov, model, wahba, staging, flags, None, dt_cols, n_valid)


def test_batch_entry_point_rejects_bad_arguments_without_gpu():
    lib = _lib.load()
    buf = np.zeros(64, dtype=np.float32)
    p = buf.ctypes.data
    assert _batch_call(lib, model=2) == _lib.EINVAL                      # unknown innovation model
    assert _batch_call(lib, model=-1, n=0) == _lib.EINVAL
    assert _batch_call(lib, n=-1) == _lib.EINVAL
    assert _batch_call(lib, t=-1) == _lib.EINVAL
    assert _batch_call(lib, ns=3) == _lib.EINVAL
    assert _batch_call(lib, flags=4) == _lib.EINVAL
    assert _batch_call(lib, dt_cols=p) == _lib.EINVAL                    # streams are still required
    assert _batch_call(lib, streams=p) == _lib.EINVAL                    # dt or dt_cols is required
    assert _batch_call(lib, streams=p, dt_cols=p) == _lib.EINVAL         # ... and the references, scales and state
    assert _batch_call(lib, n=0) == 0                                    # empty batch: no-op
    assert _batch_call(lib, n=0, innov=p, dt_cols=p, n_valid=p) == 0


def test_batch_entry_point_alignment_rules_without_gpu():
    lib = _lib.load()
    raw = np.zeros(4096, dtype=np.float32)
    base = raw.ctypes.data
    a = base + (-base) % 256                                             # a 256-byte aligned host address
    full = lambda **kw: lib.posekf_replay_batch_f32(
        256, 4, kw.get("streams", a), 256, kw.get("dt", a), 0, a, a, a, a, -1.0, -1.0, a, None, a, None, None, None, None,
        None, None, 0, 0, kw.get("staging", 0), 0, None, kw.get("dt_cols"), kw.get("n_valid"))
    assert full(n_valid=a + 2) == _lib.EALIGN                            # int32 lengths must be 4-byte aligned
    assert full(dt_cols=a + 2) == _lib.EALIGN                            # float32 columns must be 4-byte aligned
    # dt columns that TMA cannot read: an explicit TMA staging is refused (POSEKF_STAGE_AUTO runs the LDG kernel)
    assert full(dt_cols=a + 4, staging=_lib.STAGING["tma"]) == _lib.EALIGN
    assert full(dt_cols=a + 8, staging=_lib.STAGING["tma_packed"]) == _lib.EALIGN


def test_replay_checks_lengths_before_any_launch():
    with pytest.raises(ValueError):
        B._check_lengths(torch.tensor([3, 5, 11, 0], dtype=torch.int32), 4, 10)     # past the steps of the call
    with pytest.raises(ValueError):
        B._check_lengths(torch.tensor([3, -1, 1, 0], dtype=torch.int32), 4, 10)     # negative
    with pytest.raises(ValueError):
        B._check_lengths(torch.tensor([3, 5, 1, 0], dtype=torch.int64), 4, 10)      # not int32
    with pytest.raises(ValueError):
        B._check_lengths(torch.tensor([3, 5, 1], dtype=torch.int32), 4, 10)         # not [Ns]
    with pytest.raises(_lib.PosekfError):
        B._check_lengths(torch.tensor([3, 5, 10, 0], dtype=torch.int32), 4, 10)     # valid, but not on the device


def test_innovation_nll_per_filter_steps():
    sums = torch.tensor([[30.0, 8.0, 0.0], [-12.0, -5.0, 0.0]], dtype=torch.float32)
    n = torch.tensor([10, 4, 0])
    nll, nis = B.innovation_nll(sums, n, model="tangent")
    c = 1.5 * math.log(2 * math.pi)
    assert torch.allclose(nll, torch.tensor([9.0 + 10 * c, 1.5 + 4 * c, 0.0], dtype=torch.float64))
    assert nis[0].item() == 3.0 and nis[1].item() == 2.0 and math.isnan(nis[2].item())
    a, _ = B.innovation_nll(sums, 10)                                    # the scalar form is unchanged
    b, _ = B.innovation_nll(sums, torch.full((3,), 10))
    assert torch.equal(a, b)


def test_pooled_surface_is_the_joint_likelihood():
    G, Ns = 3, 4
    L = torch.tensor([7, 3, 5, 0], dtype=torch.int32)
    gen = torch.Generator().manual_seed(5)
    innov = torch.randn((2, G * G * Ns), generator=gen, dtype=torch.float32) * 10
    innov[:, 3::4] = 0                                                   # the empty column adds nothing
    st = B.ReplayState(torch.zeros((4, G * G * Ns)), torch.zeros((10, G * G * Ns)), innov=innov, innov_model="tangent")
    qs = torch.logspace(-3, -1, G)
    w = WL.SweepWorkload(torch.zeros((7, 9, Ns)), None, None, None, qs, qs, None, None, None, L)
    nll, nis = WL.pooled_innovation_surface(w, st)
    a = innov.double().reshape(2, G, G, Ns)
    Lf = L.double()
    ref_nll = (0.5 * (a[0] + a[1]) + 1.5 * Lf * math.log(2 * math.pi)).sum(-1) / Lf.sum()
    assert torch.allclose(nll, ref_nll, rtol=1e-12, atol=0) and nll.dtype == torch.float64
    assert torch.allclose(nis, a[0].sum(-1) / Lf.sum(), rtol=1e-12, atol=0)


_steph = None


def _steph_lib():
    global _steph
    if _steph is None:
        tmp = tempfile.mkdtemp(prefix="hostsim_steph_")
        atexit.register(shutil.rmtree, tmp, True)
        so = os.path.join(tmp, "libhostsim_steph.so")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-x", "c++", "-ffp-contract=off", "-fPIC", "-shared", "-o", so,
                               os.path.join(HERE, "hostsim", "steph.cpp")])
        _steph = C.CDLL(so)
    return _steph


def test_packed_step_constants_per_lane_equal_scalar_bitwise():
    rng = np.random.default_rng(3)
    n = 20000
    h0 = (0.01 * (1 + 0.2 * rng.uniform(-1, 1, n))).astype(np.float32)
    h1 = np.concatenate([(0.01 * (1 + 0.2 * rng.uniform(-1, 1, n - 6))), [0.0, 1e-30, 5.0, 0.0, 3e-3, 1e-7]]).astype(np.float32)
    out = np.empty(12 * n, dtype=np.float32)
    f = lambda a: a.ctypes.data_as(C.POINTER(C.c_float))
    assert _steph_lib().hostsim_steph(C.c_int64(n), f(h0), f(h1), f(out)) == 0
    scalar, packed = out[:6 * n].view(np.uint32), out[6 * n:].view(np.uint32)
    np.testing.assert_array_equal(scalar, packed)
    assert (out[:6 * n].reshape(n, 6)[:, 0] == h0).all()
