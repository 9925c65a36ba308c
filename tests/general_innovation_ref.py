"""Float64 definition of the innovation terms and the gate with general Q and R matrices -- TEST INFRASTRUCTURE.

`replay` is the recursion of `tests.general_qr_ref.replay_general` (the reference's KalmanFilter with Q and R assigned,
per-filter matrices) with, per step and filter:
    S = P^- + R,  e = y - z  (y sign-fixed by the comparator)
    4-D:      nis4 = e^T S^-1 e (np.linalg.solve),   logdet4 = ln det S (np.linalg.slogdet)
    tangent:  nis3, logdet3 = `innovation_tangent_ref.tangent_terms` (an explicit orthonormal basis of z-perp)
    gated_t = nis3 > gamma (strict; NaN is not gated), or decisions[t] when forced
    gated:   X_t = z_t / |z_t|,  P_t = P^-_t;   else the reference's update.
That is the definition of include/posekf.h (posekf_replay_general_innovation_f32).  The terms are recorded on every step,
gated or not.  `decisions` [T,N] forces the gate, so that a device run can be followed step for step.  `parts4` /
`parts3` = sum_k |ln lambda_k(S)| (resp. S3): the size of the terms ln det S is a sum of, the scale a per-step
log-determinant is compared on (it can pass near 0 while its parts are not small).
"""
from __future__ import annotations

import numpy as np

from oracle import ekf_oracle as O
from tests import innovation_tangent_ref as TR
from tests.general_qr_ref import _mats


def replay(dt_ns, gyro, acc, mag, acc_ref, mag_ref, Q, R, gamma=np.inf, decisions=None, basis="householder"):
    """dt_ns [T] or [T,N]; gyro/acc/mag [T,3,N]; acc_ref/mag_ref [N,3]; Q [3,3] or [N,3,3]; R [4,4] or [N,4,4]; gamma the
    NIS3 threshold; decisions [T,N] bool or None.  Returns dict(X [T,N,4], flips [T,N], nis4, logdet4, nis3, logdet3,
    parts4, parts3 [T,N], gated [T,N] bool, P [N,4,4] final covariance)."""
    T, _, N = gyro.shape
    Q, R = _mats(Q, N, 3), _mats(R, N, 4)
    X = np.tile(np.asarray([1.0, 0.0, 0.0, 0.0]), (N, 1))
    P = np.tile(np.identity(4), (N, 1, 1))
    acc_ref = np.asarray(acc_ref, dtype=np.float64)
    mag_ref = np.asarray(mag_ref, dtype=np.float64)
    dt_ns = np.asarray(dt_ns, dtype=np.float64)
    out = dict(X=np.empty((T, N, 4)), flips=np.zeros((T, N), dtype=bool), gated=np.zeros((T, N), dtype=bool),
               **{k: np.empty((T, N)) for k in ("nis4", "logdet4", "nis3", "logdet3", "parts4", "parts3")})
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
        flip = np.einsum("ni,ni->n", y, z) < 0.0
        y = np.where(flip[:, None], -y, y)
        e = y - z
        out["nis4"][i] = np.einsum("ni,ni->n", e, np.linalg.solve(S, e[:, :, None])[:, :, 0])
        out["logdet4"][i] = np.linalg.slogdet(S)[1]
        out["nis3"][i], out["logdet3"][i] = TR.tangent_terms(S, e, z, basis)
        E = TR.BASES[basis](z / np.linalg.norm(z, axis=1)[:, None])
        out["parts4"][i] = np.abs(np.log(np.linalg.eigvalsh(S))).sum(1)
        out["parts3"][i] = np.abs(np.log(np.linalg.eigvalsh(E.transpose(0, 2, 1) @ S @ E))).sum(1)
        g = (out["nis3"][i] > gamma) if decisions is None else np.asarray(decisions[i], dtype=bool)
        Xu = z + np.einsum("nij,nj->ni", K, e)
        Pu = P - K @ P
        X = np.where(g[:, None], z, Xu)
        P = np.where(g[:, None, None], P, Pu)
        X = X / O._norm_b(X)[:, None]
        out["X"][i], out["flips"][i], out["gated"][i] = X, flip, g
    out["P"] = P
    return out


def terms(out, model):
    """(nis [T,N], logdet [T,N]) of `replay`'s output for the model "full" or "tangent"."""
    return (out["nis4"], out["logdet4"]) if model == "full" else (out["nis3"], out["logdet3"])


def step_scale(out, model):
    """[T,N] |NIS_t| + sum_k |ln lambda_k|: the scale of a per-step error (see the module docstring)."""
    nis = out["nis4"] if model == "full" else out["nis3"]
    return np.abs(nis) + (out["parts4"] if model == "full" else out["parts3"])


def pooled_nll(nis, logdet, lengths, dof):
    """Per-filter NLL (float64) from per-step terms [T,N] over the first lengths[n] steps of each filter."""
    T, N = nis.shape
    live = np.arange(T)[:, None] < np.asarray(lengths)[None, :]
    s = np.where(live, nis + logdet, 0.0).sum(0)
    return 0.5 * s + 0.5 * dof * np.asarray(lengths, dtype=np.float64) * np.log(2.0 * np.pi)
