"""Float64 definition of the innovation gate -- TEST INFRASTRUCTURE.

`replay_gated` is the recursion of `tests.innovation_tangent_ref.replay_tangent` (the reference's
PKF/ExtendedKalmanFilter.py:58-80 in float64) with the gate of include/posekf.h (posekf_replay_gated_f32):
    NIS3_t = e3^T S3^-1 e3   (explicit tangent basis, `innovation_tangent_ref.tangent_terms`)
    gated_t = NIS3_t > gamma   (strict; NaN is not gated), or decisions[t] when forced
    gated:   X_t = z_t / |z_t|  (the prediction),   P_t = P^-_t  (the propagated covariance)
    else:    the reference's update.
The innovation terms are recorded on every step, gated or not.  `decisions` [T,N] forces the gate, so that a device run
can be followed step for step without a threshold tie sending the two recursions apart.
"""
from __future__ import annotations

import numpy as np

from oracle import ekf_oracle as O
from tests import innovation_tangent_ref as TR


def replay_gated(dt_ns, gyro, acc, mag, acc_ref, mag_ref, q_scale, r_scale, gamma=np.inf, decisions=None):
    """dt_ns [T] or [T,N]; gyro/acc/mag [T,3,N]; acc_ref/mag_ref [N,3]; q_scale/r_scale scalar or [N]; gamma the NIS3
    threshold; decisions [T,N] bool or None.  Returns dict(X [T,N,4], flips [T,N], nis [T,N], logdet [T,N],
    gated [T,N] bool, P [N,4,4] final covariance)."""
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
    out = dict(X=np.empty((T, N, 4)), flips=np.zeros((T, N), dtype=bool), nis=np.empty((T, N)), logdet=np.empty((T, N)),
               gated=np.zeros((T, N), dtype=bool))
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
        nis, logdet = TR.tangent_terms(S, e, z)
        g = (nis > gamma) if decisions is None else np.asarray(decisions[i], dtype=bool)
        Xu = z + np.einsum("nij,nj->ni", K, e)
        Pu = P - K @ P
        X = np.where(g[:, None], z, Xu)
        P = np.where(g[:, None, None], P, Pu)
        X = X / O._norm_b(X)[:, None]
        out["X"][i], out["flips"][i], out["nis"][i], out["logdet"][i], out["gated"][i] = X, flip, nis, logdet, g
    out["P"] = P
    return out


def angle(a, b):
    """Angle [rad] between quaternions a, b [..., 4], sign-insensitive (as `oracle.ekf_oracle.quat_angle`)."""
    return O.quat_angle(a, b)
