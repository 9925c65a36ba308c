"""Float64 definition of the innovation likelihood -- TEST INFRASTRUCTURE.

`replay_innovation` is `oracle.ekf_oracle.replay_batched` (the reference's recursion, PKF/ExtendedKalmanFilter.py:58-80,
same numpy building blocks) that also records, per step and filter, the two terms of the filter's Gaussian model of its
innovations, literally from its own S = P + R (:63) and innovation e = y - z (:76):
    nis [T,N] = e^T S^-1 e  (np.linalg.solve),    logdet [T,N] = ln det S  (np.linalg.slogdet).
The per-filter NLL is 1/2 sum_t (nis + logdet) + 2 T ln 2 pi.
"""
from __future__ import annotations

import math

import numpy as np

from oracle import ekf_oracle as O


def replay_innovation(dt_ns, gyro, acc, mag, acc_ref, mag_ref, q_scale, r_scale):
    """dt_ns [T] or [T,N]; gyro/acc/mag [T,3,N]; acc_ref/mag_ref [N,3]; q_scale/r_scale scalar or [N].
    Returns dict(X [T,N,4], flips [T,N], nis [T,N], logdet [T,N])."""
    T, _, N = gyro.shape
    qs = np.broadcast_to(np.asarray(q_scale, dtype=np.float64), (N,))
    rs = np.broadcast_to(np.asarray(r_scale, dtype=np.float64), (N,))
    Q = qs[:, None, None] * np.identity(3)[None]
    R = rs[:, None, None] * np.identity(4)[None]
    X = np.tile(np.asarray([1.0, 0.0, 0.0, 0.0]), (N, 1))
    P = np.tile(np.identity(4), (N, 1, 1))
    acc_ref = np.asarray(acc_ref, dtype=np.float64)
    mag_ref = np.asarray(mag_ref, dtype=np.float64)
    dt_ns = np.asarray(dt_ns, dtype=np.float64)
    traj = np.empty((T, N, 4))
    flips = np.zeros((T, N), dtype=bool)
    nis = np.empty((T, N))
    logdet = np.empty((T, N))
    for i in range(T):
        w = np.ascontiguousarray(gyro[i].T, dtype=np.float64)
        a = np.ascontiguousarray(acc[i].T, dtype=np.float64)
        m = np.ascontiguousarray(mag[i].T, dtype=np.float64)
        A = O._half_omega_b(w)
        Bn = O._jacobian_b_b(X)
        P = A @ P @ A.transpose(0, 2, 1) + Bn @ Q @ Bn.transpose(0, 2, 1)
        h = (dt_ns[i] * (10 ** -9))
        h = h[:, None] if np.ndim(h) else h
        k1 = np.einsum("nij,nj->ni", A, X)
        k2 = np.einsum("nij,nj->ni", A, X + h / 2 * k1)
        k3 = np.einsum("nij,nj->ni", A, X + h / 2 * k2)
        k4 = np.einsum("nij,nj->ni", A, X + h * k3)
        z = X + 1 / 6 * h * (k1 + 2 * k2 + 2 * k3 + k4)
        z = z / O._norm_b(z)[:, None]
        S = P + R
        K = P @ np.linalg.inv(S)
        ka = np.abs(a[:, 2])
        y = O.wahba_batched(acc_ref, mag_ref, a, m, ka, 1 - ka)
        flip = np.einsum("ni,ni->n", y, z) < 0.0
        y = np.where(flip[:, None], -y, y)
        e = y - z
        nis[i] = np.einsum("ni,ni->n", e, np.linalg.solve(S, e[:, :, None])[:, :, 0])
        logdet[i] = np.linalg.slogdet(S)[1]
        X = z + np.einsum("nij,nj->ni", K, e)
        P = P - K @ P
        X = X / O._norm_b(X)[:, None]
        flips[i] = flip
        traj[i] = X
    return dict(X=traj, flips=flips, nis=nis, logdet=logdet)


def nll(nis_sum, logdet_sum, n_steps):
    """Per-filter innovation NLL from the two sums (natural log)."""
    return 0.5 * (np.asarray(nis_sum) + np.asarray(logdet_sum)) + 2.0 * n_steps * math.log(2.0 * math.pi)
