"""Reader / writer of the reference's text log (`KalmanFilter.txt`), SURVEY.md section 8(f-1).

The C++ server appends one `key : v,v,v` line per event (`Kalman Filter Server/PoseEstimator/
KalmanFilter.cpp:28,32,60-67,138,150-153,180-183,274,287,300`, numbers via `std::to_string`, i.e.
`%f`), and the Python replay parses it with substring tests in a fixed order
(`Python Kalman Filter/ReadFile.py:23-45`).  `read_log` follows those parse rules exactly (the order
matters: `'q_gyro'` is tested before `'gyro'`, and `'T'` is a bare substring test); `write_log`
emits the server's line sequence.  This is host-side text I/O, as in the reference; the arrays it
yields feed the device through `LogData.to_streams`.
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np


@dataclass
class LogData:
    """Same attribute names as the reference's `getData` (ReadFile.py:3-11)."""
    mag_0: list = field(default_factory=list)
    mag_1: list = field(default_factory=list)
    acc_0: list = field(default_factory=list)
    acc_1: list = field(default_factory=list)
    gyro: list = field(default_factory=list)
    timestamp: list = field(default_factory=list)
    quart_wahba: list = field(default_factory=list)
    quart_xk: list = field(default_factory=list)
    quart_gyro: list = field(default_factory=list)

    # ---- device hand-off ---------------------------------------------------------------------
    def n_steps(self) -> int:
        return len(self.acc_1)

    def to_streams(self, device="cuda"):
        """-> (streams [T,9,1] float32, acc_ref [3,1], mag_ref [3,1], dt [T] float32 seconds), the
        arguments of `batched.replay`.  Timestamps are differenced in integer/float64 ns on the host
        (the first one only seeds previousT: main_file.py:19,25)."""
        import torch
        T = self.n_steps()
        s = np.concatenate([np.asarray(self.gyro[:T], dtype=np.float64), np.asarray(self.acc_1, dtype=np.float64),
                            np.asarray(self.mag_1[:T], dtype=np.float64)], axis=1)           # [T, 9]
        t_ns = np.asarray(self.timestamp, dtype=np.float64)[:, 0]
        dt = np.diff(t_ns)[:T] * 1e-9
        dev = torch.device(device)
        f32 = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev)
        return (f32(s[:, :, None]), f32(np.asarray(self.acc_0, dtype=np.float64)[:, None]),
                f32(np.asarray(self.mag_0, dtype=np.float64)[:, None]), f32(dt))


@dataclass
class LogBatch:
    """Several recordings stacked for one `batched.replay` launch (`stack_logs`): column c is recording c.
    streams [T,9,Ns] float32, acc_ref / mag_ref [3,Ns], dt [T,Ns] float32 seconds, lengths [Ns] int32 (steps of each
    recording), n_logs: the number of real recordings (columns n_logs..Ns-1 are padding of length 0)."""
    streams: object
    acc_ref: object
    mag_ref: object
    dt: object
    lengths: object
    n_logs: int

    def window(self, t0: int, t1: int) -> "LogBatch":
        """Steps [t0, t1) for a time-chunked replay: the slices, and lengths counted from t0, clamped to [0, t1 - t0]
        (pass `keep_filter_frame=True` on every chunk but the last)."""
        import torch
        lengths = torch.clamp(self.lengths - t0, 0, t1 - t0).to(torch.int32)
        return LogBatch(self.streams[t0:t1], self.acc_ref, self.mag_ref, self.dt[t0:t1], lengths, self.n_logs)


def stack_logs(logs, device="cuda", pad_cols_to: int = 4) -> LogBatch:
    """Stack recordings (`LogData`) of different lengths and timestamps into one batch.  Each recording's dt is its own
    timestamps differenced in float64 ns on the host, bit for bit the dt of its `to_streams` (main_file.py:25: every
    recording keeps its own previousT).  The steps past a recording's end repeat its last sample with dt = 0 (a
    recording without samples repeats its reference vectors with zero rate); the number of columns is rounded up to a
    multiple of `pad_cols_to` (4 keeps the TMA staging) with empty recordings of length 0."""
    import torch
    K = len(logs)
    Tmax = max([lg.n_steps() for lg in logs], default=0)
    Ns = -(-K // pad_cols_to) * pad_cols_to if pad_cols_to > 1 else K
    streams = np.zeros((Tmax, 9, Ns), dtype=np.float32)
    acc_ref = np.zeros((3, Ns), dtype=np.float32)
    mag_ref = np.zeros((3, Ns), dtype=np.float32)
    acc_ref[2] = 1.0
    mag_ref[0] = 1.0
    dt = np.zeros((Tmax, Ns), dtype=np.float32)
    lengths = np.zeros((Ns,), dtype=np.int32)
    for c, lg in enumerate(logs):
        T = lg.n_steps()
        acc_ref[:, c] = np.asarray(lg.acc_0, dtype=np.float64)
        mag_ref[:, c] = np.asarray(lg.mag_0, dtype=np.float64)
        lengths[c] = T
        if T == 0:
            continue
        # the arithmetic of to_streams, one recording at a time
        s = np.concatenate([np.asarray(lg.gyro[:T], dtype=np.float64), np.asarray(lg.acc_1, dtype=np.float64),
                            np.asarray(lg.mag_1[:T], dtype=np.float64)], axis=1)
        t_ns = np.asarray(lg.timestamp, dtype=np.float64)[:, 0]
        streams[:T, :, c] = s.astype(np.float32)
        streams[T:, :, c] = streams[T - 1, :, c]
        dt[:T, c] = np.ascontiguousarray(np.diff(t_ns)[:T] * 1e-9, dtype=np.float32)
    for c in range(Ns):
        if lengths[c] == 0:
            streams[:, 3:6, c] = acc_ref[:, c]
            streams[:, 6:9, c] = mag_ref[:, c]
    dev = torch.device(device)
    t = lambda a: torch.from_numpy(a).to(dev)
    return LogBatch(t(streams), t(acc_ref), t(mag_ref), t(dt), t(lengths), K)


@dataclass
class SensorEvents:
    """One sensor's event stream: t_ns [M] int64 timestamps in ns (strictly increasing), v [M,3] float32 values."""
    t_ns: np.ndarray
    v: np.ndarray


@dataclass
class RawRecording:
    """A raw recording as a phone sends it: each sensor's events at its own rate and with its own timestamps."""
    gyro: SensorEvents
    acc: SensorEvents
    mag: SensorEvents


def _pack_sensor(events, name: str):
    """Concatenate one sensor of every recording: (t [M] int64, v [3,M] float32, off [len+1] int64), host arrays."""
    ts, vs = [], []
    for c, e in enumerate(events):
        t = np.asarray(e.t_ns)
        v = np.asarray(e.v)
        if t.dtype.kind not in "iu":
            raise TypeError(f"recording {c}: {name} timestamps must be integer ns")
        if t.ndim != 1 or v.shape != (t.shape[0], 3):
            raise ValueError(f"recording {c}: {name} needs t_ns [M] and v [M,3], got {t.shape} and {v.shape}")
        t = t.astype(np.int64)
        if t.size > 1 and not (np.diff(t) > 0).all():
            raise ValueError(f"recording {c}: {name} timestamps are not strictly increasing")
        ts.append(t)
        vs.append(np.asarray(v, dtype=np.float32))
    off = np.zeros(len(ts) + 1, dtype=np.int64)
    off[1:] = np.cumsum([t.size for t in ts])
    t = np.concatenate(ts) if ts else np.zeros(0, dtype=np.int64)
    v = np.concatenate(vs).T if vs else np.zeros((3, 0), dtype=np.float32)
    return t, np.ascontiguousarray(v), off


def align_recordings(recs, device="cuda", k_init: int = 100, pad_cols_to: int = 4) -> LogBatch:
    """Raw event recordings (`RawRecording`) -> the `LogBatch` that `stack_logs` returns, aligned to each recording's
    gyro clock on the device in one call (`batched.align_events`; the rules are `posekf_align_events_f32`'s in
    include/posekf.h): reference vectors from the first `k_init` acc / mag events, one step per gyro event after them
    that both sensors bracket, acc / mag interpolated to the gyro timestamp and normalised, dt from the gyro timestamps.
    The number of columns is rounded up to a multiple of `pad_cols_to` with empty recordings, as in `stack_logs`.  The
    replay's own low-pass (`lpf_alpha_acc/mag`) is not applied here."""
    import torch
    from . import batched as B
    if int(k_init) < 1:
        raise ValueError("k_init must be >= 1")
    recs = list(recs)
    K = len(recs)
    Ns = -(-K // pad_cols_to) * pad_cols_to if pad_cols_to > 1 else K
    empty = SensorEvents(np.zeros(0, dtype=np.int64), np.zeros((0, 3), dtype=np.float32))
    packed = []
    for name in ("gyro", "acc", "mag"):
        t, v, off = _pack_sensor([getattr(r, name) for r in recs] + [empty] * (Ns - K), name)
        if name == "gyro" and off.size > 1 and int(np.diff(off).max()) >= 2 ** 31:
            raise ValueError("a recording has 2^31 gyro events or more")
        dev = torch.device(device)
        packed += [torch.from_numpy(t).to(dev), torch.from_numpy(v).to(dev), torch.from_numpy(off).to(dev)]
    streams, dt, lengths, acc_ref, mag_ref = B.align_events(*packed, k_init=int(k_init))
    return LogBatch(streams, acc_ref, mag_ref, dt, lengths, K)


def _values(line: str):
    """ReadFile.py:14-21 (`getArray`): text after the first ':' split on ','."""
    return [float(v) for v in line.split(":")[1].split(",")]


def parse_lines(lines) -> LogData:
    d = LogData()
    for line in lines:                                   # ReadFile.py:27-45, same test order
        if "mag_0" in line:
            d.mag_0 = _values(line)
        elif "acc_0" in line:
            d.acc_0 = _values(line)
        elif "Acc_1" in line:
            d.acc_1.append(_values(line))
        elif "Mag_1" in line:
            d.mag_1.append(_values(line))
        elif "q_gyro" in line:
            d.quart_gyro.append(_values(line))
        elif "gyro" in line:
            d.gyro.append(_values(line))
        elif "T" in line:
            d.timestamp.append(_values(line))
        elif "Wahba_quart" in line:
            d.quart_wahba.append(_values(line))
        elif "X_k" in line:
            d.quart_xk.append(_values(line))
    return d


def read_log(path: str) -> LogData:
    with open(path) as fh:
        return parse_lines(fh.readlines())


def _f(v) -> str:
    return "%f" % float(v)          # std::to_string(double)


def _vec(key: str, v) -> str:
    return key + " : " + ",".join(_f(x) for x in v)


def format_log(acc_0, mag_0, t0_ns: int, t_ns, gyro, mag_1, acc_1, x_k, wahba_quart, q_gyro) -> list[str]:
    """The server's line sequence: header (`set_mag_0`, `set_acc_0`, `compute_initial_params`:
    KalmanFilter.cpp:26-33,56-67), the first `T` line (`Prediction` :136-141), then per sample
    gyro (:274), T, q_gyro (:150-153), Mag_1 (:287), Acc_1 (:300), X_k, Wahba_quart (:180-183)."""
    out = [_vec("mag_0", mag_0), _vec("acc_0", acc_0), "q_gyro : 1.0, 0.0, 0.0, 0.0", "X_k : 1.0, 0.0, 0.0, 0.0",
           "Wahba_quart : 1.0, 0.0, 0.0, 0.0"]
    for i in range(len(gyro)):
        out.append(_vec("gyro", gyro[i]))
        if i == 0:
            out.append("T : %d" % int(t0_ns))
        out.append("T : %d" % int(t_ns[i]))
        out.append(_vec("q_gyro", q_gyro[i]))
        out.append(_vec("Mag_1", mag_1[i]))
        out.append(_vec("Acc_1", acc_1[i]))
        out.append(_vec("X_k", x_k[i]))
        out.append(_vec("Wahba_quart", wahba_quart[i]))
    return out


def write_log(path: str, **kw) -> None:
    with open(path, "w") as fh:
        fh.write("\n".join(format_log(**kw)) + "\n")
