"""Synthetic IMU sequence generator (SURVEY.md section 8d).

The recorded dataset of the reference is not in its repository (`Python Kalman Filter/ReadFile.py:24`
opens an un-shipped file), so every parity and throughput input is synthetic.  The generator is
plain torch (it runs on the CPU for the tests and on the GPU for the benchmark) and is *plumbing*:
it produces the `[T, 9, N]` float32 stream tensor the replay kernel consumes, it is never timed.

Conventions (validated against the reference by tests/test_synth.py): scalar-first quaternion
[w,x,y,z]; q maps body -> initial frame; omega is the body rate, q_dot = 0.5*q (x) (0,omega);
measurements are `meas = R(q)^T ref`, so that Wahba's `ref ~= R meas` recovers R(q).
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import torch

GYRO, ACC, MAG = slice(0, 3), slice(3, 6), slice(6, 9)
N_CHANNELS = 9


@dataclass
class SyntheticIMU:
    """streams  : [T, 9, N] float32   rows 0-2 gyro (rad/s, body), 3-5 acc, 6-8 mag (unit vectors, body)
    acc_ref  : [3, N] float32      sample 0 of acc  (the log's acc_0)
    mag_ref  : [3, N] float32      sample 0 of mag  (the log's mag_0)
    q_true   : [T, 4, N] float64 or None   ground-truth attitude after each step
    dt       : float               seconds between samples"""
    streams: torch.Tensor
    acc_ref: torch.Tensor
    mag_ref: torch.Tensor
    q_true: torch.Tensor | None
    dt: float


def _quat_mul(a, b):
    """Hamilton product of [4,N] tensors (scalar first)."""
    aw, ax, ay, az = a[0], a[1], a[2], a[3]
    bw, bx, by, bz = b[0], b[1], b[2], b[3]
    return torch.stack((aw * bw - ax * bx - ay * by - az * bz,
                        aw * bx + ax * bw + ay * bz - az * by,
                        aw * by - ax * bz + ay * bw + az * bx,
                        aw * bz + ax * by - ay * bx + az * bw))


def _rotate_inverse(q, v):
    """R(q)^T v for q [4,N], v [3,N]."""
    w, x, y, z = q[0], q[1], q[2], q[3]
    vx, vy, vz = v[0], v[1], v[2]
    # rows of R(q)^T are the columns of R(q)
    r00 = 1 - 2 * (y * y + z * z); r01 = 2 * (x * y - w * z); r02 = 2 * (x * z + w * y)
    r10 = 2 * (x * y + w * z); r11 = 1 - 2 * (x * x + z * z); r12 = 2 * (y * z - w * x)
    r20 = 2 * (x * z - w * y); r21 = 2 * (y * z + w * x); r22 = 1 - 2 * (x * x + y * y)
    return torch.stack((r00 * vx + r10 * vy + r20 * vz,
                        r01 * vx + r11 * vy + r21 * vz,
                        r02 * vx + r12 * vy + r22 * vz))


def _unit(v):
    return v / torch.linalg.vector_norm(v, dim=0, keepdim=True)


def _reference_pair(U, N, az_range, f64):
    """Gravity and field in the body frame at the start (float64 [3,N] each), drawn with the uniform sampler U."""
    # initial tilt: gravity in the body frame has |z| = cos(tilt) in az_range, random azimuth
    az = U(az_range[0] + 0.03, az_range[1] - 0.03, N) * torch.where(U(0, 1, N) < 0.5, -1.0, 1.0)
    psi = U(0.0, 2 * math.pi, N)
    s = torch.sqrt(1 - az * az)
    acc0 = torch.stack((s * torch.cos(psi), s * torch.sin(psi), az))
    # field: fixed angle to gravity (world: g=(0,0,1), m=normalize(0.4,0,-0.9165)); pick the
    # horizontal direction at a random heading around gravity
    mw = torch.tensor([0.4, 0.0, -0.9165], **f64)
    mw = mw / torch.linalg.vector_norm(mw)
    hdg = U(0.0, 2 * math.pi, N)
    helper = torch.where((acc0[2].abs() < 0.9).unsqueeze(0),
                         torch.tensor([0.0, 0.0, 1.0], **f64).unsqueeze(1).expand(3, N),
                         torch.tensor([1.0, 0.0, 0.0], **f64).unsqueeze(1).expand(3, N))
    e1 = _unit(torch.linalg.cross(acc0, helper, dim=0))
    e2 = torch.linalg.cross(acc0, e1, dim=0)
    horiz = torch.cos(hdg) * e1 + torch.sin(hdg) * e2
    return acc0, _unit(mw[2] * acc0 + mw[0] * horiz)


def make_imu(n_filters: int, n_steps: int, *, seed: int = 0, sigma: float = 0.0, dt: float = 0.01,
             device="cpu", keep_truth: bool = False, out: torch.Tensor | None = None,
             az_range=(0.02, 0.98), gyro_sigma=None) -> SyntheticIMU:
    """Generate `n_filters` independent trajectories of `n_steps` samples.

    Body rate: omega_i(t) = sum_{j<3} A_ij sin(2 pi f_ij t + phi_ij), A~U(0.2,1) rad/s,
    f~U(0.05,0.5) Hz, phi~U(0,2pi).  True attitude: per-sample exact exponential of the mid-point
    rate.  Reference vectors: gravity (0,0,1) and field normalize(0.4,0,-0.9165) seen through a
    random initial tilt drawn so that |acc_z| starts inside `az_range`.  Noise sigma is added to
    all three sensors, acc/mag are renormalised afterwards.  Everything is computed in float64 and
    rounded to float32 once; the oracle consumes exactly those float32 values.
    `gyro_sigma`: (sx, sy, sz) per-body-axis gyro noise std that replaces `sigma` on the gyro (an anisotropic process
    noise, e.g. a noisier yaw gyro); None keeps `sigma` and draws exactly the numbers it always did.
    """
    dev = torch.device(device)
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    f64 = dict(dtype=torch.float64, device=dev)
    N, T = n_filters, n_steps

    def U(lo, hi, *shape):
        return lo + (hi - lo) * torch.rand(*shape, generator=g, **f64)

    amp, freq, phase = U(0.2, 1.0, 3, 3, N), U(0.05, 0.5, 3, 3, N), U(0.0, 2 * math.pi, 3, 3, N)
    acc0, mag0 = _reference_pair(U, N, az_range, f64)

    if out is None:
        out = torch.empty((T, N_CHANNELS, N), dtype=torch.float32, device=dev)
    assert out.shape == (T, N_CHANNELS, N) and out.dtype == torch.float32
    q_true = torch.empty((T, 4, N), **f64) if keep_truth else None

    def add_noise(v):
        if sigma == 0.0:
            return v
        return v + sigma * torch.randn(v.shape, generator=g, **f64)

    gyro_std = None if gyro_sigma is None else torch.as_tensor(gyro_sigma, **f64).reshape(3, 1)

    def add_gyro_noise(v):
        if gyro_std is None:
            return add_noise(v)
        return v + gyro_std * torch.randn(v.shape, generator=g, **f64)

    if sigma != 0.0:   # the references themselves are noisy samples, like a real log's sample 0
        acc0_meas, mag0_meas = _unit(add_noise(acc0)), _unit(add_noise(mag0))
    else:
        acc0_meas, mag0_meas = acc0, mag0

    q = torch.zeros((4, N), **f64)
    q[0] = 1.0
    two_pi_f = 2 * math.pi * freq
    for i in range(T):
        t_mid = (i + 0.5) * dt
        t_end = (i + 1.0) * dt
        w_mid = (amp * torch.sin(two_pi_f * t_mid + phase)).sum(dim=1)        # [3,N]
        w_end = (amp * torch.sin(two_pi_f * t_end + phase)).sum(dim=1)
        ang = torch.linalg.vector_norm(w_mid, dim=0) * dt
        half = 0.5 * ang
        sinc = torch.where(ang > 1e-12, torch.sin(half) / ang.clamp_min(1e-300), torch.full_like(ang, 0.5))
        dq = torch.cat((torch.cos(half).unsqueeze(0), w_mid * dt * sinc), dim=0)
        q = _quat_mul(q, dq)
        q = q / torch.linalg.vector_norm(q, dim=0, keepdim=True)
        # the gyro sample logged with step i is the body rate at that sample's timestamp
        out[i, GYRO] = add_gyro_noise(w_end).to(torch.float32)
        out[i, ACC] = _unit(add_noise(_rotate_inverse(q, acc0))).to(torch.float32)
        out[i, MAG] = _unit(add_noise(_rotate_inverse(q, mag0))).to(torch.float32)
        if keep_truth:
            q_true[i] = q
    return SyntheticIMU(out, acc0_meas.to(torch.float32), mag0_meas.to(torch.float32), q_true, dt)


def add_disturbances(streams: torch.Tensor, *, seed: int = 1, n_mag: int = 3, n_acc: int = 0,
                     mag_strength=(0.15, 0.5), acc_strength=(0.15, 0.5), length=(100, 300),
                     margin=(200, 300)) -> torch.Tensor:
    """Inject sensor disturbances into a `[T, 9, N]` stream IN PLACE and return the disturbed-step mask `[T, N]` (bool).

    Every recording (column) gets `n_mag` magnetometer disturbances (a magnetic field distortion near metal) and
    `n_acc` accelerometer ones (a burst of linear acceleration).  Each starts at a uniform step in
    [margin[0], T - margin[1]), lasts a uniform number of steps in [length[0], length[1]] and adds u * d to the unit
    sample, with u ~ U(strength) and d a random unit vector fixed for the disturbance; the sample is then renormalised.
    Overlapping disturbances add up.  The draws come from a CPU generator seeded with `seed`, so the result does not
    depend on the device.  Sample 0 (the reference vectors of `make_imu`) is outside every disturbance."""
    T, C, N = streams.shape
    if C != N_CHANNELS:
        raise ValueError("streams must be [T, 9, N]")
    if T - margin[1] <= margin[0]:
        raise ValueError(f"T = {T} leaves no room for a disturbance between the margins {margin}")
    dev = streams.device
    g = torch.Generator(device="cpu")
    g.manual_seed(seed)
    f64 = dict(dtype=torch.float64)
    t = torch.arange(T, device=dev)[:, None]
    mask = torch.zeros((T, N), dtype=torch.bool, device=dev)
    for rows, count, (lo, hi) in ((MAG, n_mag, mag_strength), (ACC, n_acc, acc_strength)):
        for _ in range(count):
            start = torch.randint(margin[0], T - margin[1], (N,), generator=g).to(dev)
            dur = torch.randint(length[0], length[1] + 1, (N,), generator=g).to(dev)
            u = (lo + (hi - lo) * torch.rand(N, generator=g, **f64)).to(dev)
            d = _unit(torch.randn(3, N, generator=g, **f64)).to(dev)
            on = (t >= start[None]) & (t < (start + dur)[None])                       # [T,N]
            v = streams[:, rows].to(torch.float64) + (u * d)[None] * on[:, None].to(torch.float64)
            v = v / torch.linalg.vector_norm(v, dim=1, keepdim=True)
            streams[:, rows] = torch.where(on[:, None], v.to(torch.float32), streams[:, rows])
            mask |= on
    return mask


@dataclass
class SyntheticEvents:
    """recordings : list of `logio.RawRecording` (int64 ns timestamps, float32 values)
    truth      : list of [Mg, 4] float64 true attitudes at each gyro timestamp, or None
    acc0, mag0 : [3, n_rec] float64 noise-free gravity and field in the body frame at rest"""
    recordings: list
    truth: list | None
    acc0: torch.Tensor
    mag0: torch.Tensor


def make_events(n_rec: int, duration_s, *, rates=(200.0, 100.0, 100.0), jitter: float = 0.2, sigma: float = 0.0,
                seed: int = 0, keep_truth: bool = False, still_s: float = 1.5, t0_ns: int = 1_700_000_000_000_000_000,
                az_range=(0.02, 0.98)) -> SyntheticEvents:
    """Asynchronous raw event recordings from `make_imu`'s motion model: the same body-rate model and reference
    geometry, with the device at rest for the first `still_s` seconds (the phase whose first 100 acc / mag events make
    the reference vectors) and the rate model running from then on.  Each sensor has its own sample clock: event k of
    a sensor at rate f is at t0_ns + (phase + k + jitter * u_k) / f seconds, phase ~ U(0,1), u_k ~ U(-1/2,1/2), rounded
    to integer ns; jitter < 1 keeps the timestamps strictly increasing.  `duration_s` and each entry of `rates` are
    scalars or one value per recording.  Gyro events are the body rate at their timestamp, acc / mag the reference
    vectors rotated into the body frame; noise sigma on all three, acc / mag renormalised; float64, rounded to float32
    once.  The true attitude (body -> rest frame, identity at rest) is integrated with `make_imu`'s exact exponential of
    the mid-point rate over the merged event times of each recording and kept at every gyro timestamp."""
    from .logio import RawRecording, SensorEvents
    if not 0.0 <= jitter < 1.0:
        raise ValueError("jitter must be in [0, 1)")
    g = torch.Generator(device="cpu")
    g.manual_seed(seed)
    f64 = dict(dtype=torch.float64)
    N = n_rec

    def U(lo, hi, *shape):
        return lo + (hi - lo) * torch.rand(*shape, generator=g, **f64)

    amp, freq, phase = U(0.2, 1.0, 3, 3, N), U(0.05, 0.5, 3, 3, N), U(0.0, 2 * math.pi, 3, 3, N)
    acc0, mag0 = _reference_pair(U, N, az_range, f64)
    per_rec = lambda x: torch.as_tensor(x, **f64).expand(N).clone()
    dur = per_rec(duration_s)
    rate = [per_rec(r) for r in rates]

    def omega(c, t):
        """body rate [3, n] of recording c at times t [n] (seconds since t0)"""
        tm = (t - still_s).clamp_min(0.0)
        w = (amp[:, :, c, None] * torch.sin(2 * math.pi * freq[:, :, c, None] * tm + phase[:, :, c, None])).sum(dim=1)
        return torch.where(t >= still_s, w, torch.zeros_like(w))

    def noisy(v):
        return v if sigma == 0.0 else v + sigma * torch.randn(v.shape, generator=g, **f64)

    recs, truth = [], [] if keep_truth else None
    for c in range(N):
        times = []
        for f in rate:
            fc = float(f[c])
            n = int(math.floor(float(dur[c]) * fc))
            k = torch.arange(n, **f64)
            t = (U(0.0, 1.0, 1) + k + jitter * (U(0.0, 1.0, n) - 0.5)) / fc
            times.append(torch.round(t * 1e9).to(torch.int64))                    # ns since t0
        # attitude at the merged event times: the exact exponential of the mid-point rate over each interval
        u = torch.unique(torch.cat(times))
        us = u.to(torch.float64) * 1e-9
        h = torch.diff(torch.cat((torch.zeros(1, **f64), us)))
        w_mid = omega(c, us - 0.5 * h)
        ang = torch.linalg.vector_norm(w_mid, dim=0) * h
        half = 0.5 * ang
        sinc = torch.where(ang > 1e-12, torch.sin(half) / ang.clamp_min(1e-300), torch.full_like(ang, 0.5))
        dq = torch.cat((torch.cos(half)[None], w_mid * h * sinc), dim=0)          # [4, n]
        q = torch.empty_like(dq)
        cur = torch.tensor([1.0, 0.0, 0.0, 0.0], **f64)[:, None]
        for i in range(dq.shape[1]):
            cur = _quat_mul(cur, dq[:, i:i + 1])
            cur = cur / torch.linalg.vector_norm(cur, dim=0, keepdim=True)
            q[:, i] = cur[:, 0]
        at = lambda t_ns: q[:, torch.searchsorted(u, t_ns)]
        tg, ta, tm = times
        qa, qm = at(ta), at(tm)
        gyro = noisy(omega(c, tg.to(torch.float64) * 1e-9))
        acc = _unit(noisy(_rotate_inverse(qa, acc0[:, c, None].expand(3, qa.shape[1]))))
        mag = _unit(noisy(_rotate_inverse(qm, mag0[:, c, None].expand(3, qm.shape[1]))))
        ev = lambda t, v: SensorEvents((t + t0_ns).numpy(), v.t().to(torch.float32).numpy())
        recs.append(RawRecording(ev(tg, gyro), ev(ta, acc), ev(tm, mag)))
        if keep_truth:
            truth.append(at(tg).t().numpy())
    return SyntheticEvents(recs, truth, acc0, mag0)
