"""Float64 definition of the replay with general Q and R matrices -- TEST INFRASTRUCTURE.

`replay_kf` drives the oracle's own `KalmanFilter` (`oracle.ekf_oracle.OracleEKF`, PKF/ExtendedKalmanFilter.py:5-80) with
its Q and R attributes assigned, one filter at a time: that is the definition of include/posekf.h
(posekf_replay_general_f32).  `replay_general` is the same recursion vectorised over filters (the arithmetic of
`tests.gating_ref.replay_gated` with per-filter matrices), pinned to `replay_kf` by tests/test_general_qr_cpu.py, and
used where many filters or steps are checked.
"""
from __future__ import annotations

import numpy as np

from oracle import ekf_oracle as O


def _mats(M, n, k):
    M = np.asarray(M, dtype=np.float64)
    return np.broadcast_to(M, (n, k, k)) if M.ndim == 2 else M


def replay_kf(dt_ns, gyro, acc, mag, acc_ref, mag_ref, Q, R):
    """One filter: dt_ns [T]; gyro/acc/mag [T,3]; acc_ref/mag_ref [3]; Q [3,3]; R [4,4].
    Returns dict(X [T,4], flips [T] bool, P [4,4] final covariance)."""
    t_ns = np.concatenate([[0.0], np.cumsum(np.asarray(dt_ns, dtype=np.float64))])
    kf = O.OracleEKF(t_ns[0], np.asarray(mag_ref, dtype=np.float64), np.asarray(acc_ref, dtype=np.float64), 0.5)
    kf.Q = np.array(Q, dtype=np.float64)
    kf.R = np.array(R, dtype=np.float64)
    X, P = np.asarray([1.0, 0.0, 0.0, 0.0]), np.identity(4)
    T = len(gyro)
    out = dict(X=np.empty((T, 4)), flips=np.zeros(T, dtype=bool))
    for i in range(T):
        z, P, K = kf.predict(np.asarray(gyro[i], dtype=np.float64), t_ns[i + 1], X, P)
        X, P, out["flips"][i], _ = kf.correct_ex(np.asarray(mag[i], dtype=np.float64), np.asarray(acc[i], dtype=np.float64),
                                                 z, P, K)
        out["X"][i] = X
    out["P"] = P
    return out


def replay_general(dt_ns, gyro, acc, mag, acc_ref, mag_ref, Q, R):
    """dt_ns [T] or [T,N]; gyro/acc/mag [T,3,N]; acc_ref/mag_ref [N,3]; Q [3,3] or [N,3,3]; R [4,4] or [N,4,4].
    Returns dict(X [T,N,4], flips [T,N] bool, y [T,N,4] the Wahba quaternions before the comparator, P [N,4,4] final
    covariance)."""
    T, _, N = gyro.shape
    Q, R = _mats(Q, N, 3), _mats(R, N, 4)
    X = np.tile(np.asarray([1.0, 0.0, 0.0, 0.0]), (N, 1))
    P = np.tile(np.identity(4), (N, 1, 1))
    acc_ref = np.asarray(acc_ref, dtype=np.float64)
    mag_ref = np.asarray(mag_ref, dtype=np.float64)
    dt_ns = np.asarray(dt_ns, dtype=np.float64)
    out = dict(X=np.empty((T, N, 4)), flips=np.zeros((T, N), dtype=bool), y=np.empty((T, N, 4)))
    for i in range(T):
        w = np.ascontiguousarray(gyro[i].T, dtype=np.float64)
        A = O._half_omega_b(w)
        Bn = O._jacobian_b_b(X)
        P = A @ P @ A.transpose(0, 2, 1) + Bn @ Q @ Bn.transpose(0, 2, 1)
        h = dt_ns[i] * (10 ** -9)
        h = h[:, None] if np.ndim(h) else h
        k1 = np.einsum("nij,nj->ni", A, X)
        k2 = np.einsum("nij,nj->ni", A, X + h / 2 * k1)
        k3 = np.einsum("nij,nj->ni", A, X + h / 2 * k2)
        k4 = np.einsum("nij,nj->ni", A, X + h * k3)
        z = X + 1 / 6 * h * (k1 + 2 * k2 + 2 * k3 + k4)
        z = z / O._norm_b(z)[:, None]
        S = P + R
        K = P @ np.linalg.inv(S)
        a = np.ascontiguousarray(acc[i].T, dtype=np.float64)
        m = np.ascontiguousarray(mag[i].T, dtype=np.float64)
        ka = np.abs(a[:, 2])
        y = O.wahba_batched(acc_ref, mag_ref, a, m, ka, 1 - ka)
        out["y"][i] = y
        flip = np.einsum("ni,ni->n", y, z) < 0.0
        y = np.where(flip[:, None], -y, y)
        X = z + np.einsum("nij,nj->ni", K, y - z)
        P = P - K @ P
        X = X / O._norm_b(X)[:, None]
        out["X"][i], out["flips"][i] = X, flip
    out["P"] = P
    return out


def random_spd(rng, n, k, lo, hi):
    """[n,k,k] symmetric positive definite matrices with eigenvalues log-uniform in [lo, hi] and random eigenvectors."""
    V = np.linalg.qr(rng.standard_normal((n, k, k)))[0]
    lam = np.exp(rng.uniform(np.log(lo), np.log(hi), (n, k)))
    return np.einsum("nij,nj,nkj->nik", V, lam, V)
