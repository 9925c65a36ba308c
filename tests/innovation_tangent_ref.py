"""Float64 definition of the tangent-space innovation likelihood -- TEST INFRASTRUCTURE.

`replay_tangent` runs the reference's recursion (PKF/ExtendedKalmanFilter.py:58-80, the building blocks of
`oracle.ekf_oracle.replay_batched`, as `tests/innovation_ref.py` does) and records, per step and filter, the two terms of
the filter's Gaussian model of its innovation restricted to the tangent space of the prediction u = z/|z|:
    E [N,4,3]  an explicit orthonormal basis of u-perp,   e3 = E^T e,   S3 = E^T S E   (S = P + R :63, e = y - z :76),
    nis [T,N] = e3^T S3^-1 e3  (np.linalg.solve),    logdet [T,N] = ln det S3  (np.linalg.slogdet).
The per-filter NLL is 1/2 sum_t (nis + logdet) + 3/2 T ln 2 pi.  The result does not depend on the basis: `basis`
picks one of two constructions so that tests can check that.

`schur` instead gives the basis-free algebra the kernels use (c = z^T S^-1 z, b = z^T S^-1 e, s = e^T S^-1 e from a
Cholesky factor of S; NIS3 = s - b^2/c, ln det S3 = ln det S + ln(c/|z|^2)) -- a check of that algebra, not a definition:
at extreme Q/R its difference of near-equal terms loses float64 digits that the basis form keeps.
"""
from __future__ import annotations

import math

import numpy as np

from oracle import ekf_oracle as O


def householder_basis(u):
    """[N,4,3]: the last three columns of the reflector H = I - 2 v v^T / v^T v, v = u + sign(u_0) e_1, which maps the
    unit vector u to -sign(u_0) e_1; they are orthonormal and orthogonal to u."""
    N = u.shape[0]
    sg = np.where(u[:, 0] >= 0.0, 1.0, -1.0)
    v = u.copy()
    v[:, 0] += sg
    H = np.tile(np.identity(4), (N, 1, 1)) - 2.0 * v[:, :, None] * v[:, None, :] / np.einsum("ni,ni->n", v, v)[:, None, None]
    return H[:, :, 1:]


def qr_basis(u):
    """[N,4,3]: a second construction -- the complete QR factor of [u | I4] (first column +-u), columns 2..4."""
    M = np.concatenate([u[:, :, None], np.tile(np.identity(4), (u.shape[0], 1, 1))], axis=2)
    Q, _ = np.linalg.qr(M, mode="complete")
    return Q[:, :, 1:]


BASES = {"householder": householder_basis, "qr": qr_basis}


def tangent_terms(S, e, z, basis="householder"):
    """(nis [N], logdet [N]) of one step: S [N,4,4], e [N,4], z [N,4]."""
    E = BASES[basis](z / np.linalg.norm(z, axis=1)[:, None])
    e3 = np.einsum("nij,ni->nj", E, e)
    S3 = E.transpose(0, 2, 1) @ S @ E
    nis = np.einsum("ni,ni->n", e3, np.linalg.solve(S3, e3[:, :, None])[:, :, 0])
    return nis, np.linalg.slogdet(S3)[1]


def schur_terms(S, e, z):
    """The basis-free form of `tangent_terms` (see the module docstring)."""
    L = np.linalg.cholesky(S)
    lz = np.linalg.solve(L, z[:, :, None])[:, :, 0]
    le = np.linalg.solve(L, e[:, :, None])[:, :, 0]
    c, b, s = (np.einsum("ni,ni->n", lz, lz), np.einsum("ni,ni->n", lz, le), np.einsum("ni,ni->n", le, le))
    logdet_s = 2.0 * np.log(np.abs(np.diagonal(L, axis1=1, axis2=2))).sum(1)
    return s - b * b / c, logdet_s + np.log(c / np.einsum("ni,ni->n", z, z))


def replay_tangent(dt_ns, gyro, acc, mag, acc_ref, mag_ref, q_scale, r_scale, basis="householder", form="basis"):
    """dt_ns [T] or [T,N]; gyro/acc/mag [T,3,N]; acc_ref/mag_ref [N,3]; q_scale/r_scale scalar or [N].
    form "basis" (the definition, with `basis`) or "schur".  Returns dict(X [T,N,4], flips [T,N], nis [T,N], logdet [T,N])."""
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
        nis[i], logdet[i] = tangent_terms(S, e, z, basis) if form == "basis" else schur_terms(S, e, z)
        X = z + np.einsum("nij,nj->ni", K, e)
        P = P - K @ P
        X = X / O._norm_b(X)[:, None]
        flips[i] = flip
        traj[i] = X
    return dict(X=traj, flips=flips, nis=nis, logdet=logdet)


def nll(nis_sum, logdet_sum, n_steps):
    """Per-filter tangent-space innovation NLL from the two sums (natural log)."""
    return 0.5 * (np.asarray(nis_sum) + np.asarray(logdet_sum)) + 1.5 * n_steps * math.log(2.0 * math.pi)
