"""The oracle (oracle/ekf_oracle.py) against the frozen outputs of the unmodified reference and the
reference's own known answers.  CPU only."""
import numpy as np

from oracle import ekf_oracle as O


def test_wahba_hand_check(golden_wahba):
    # Python Kalman Filter/WahbaProblem_singularValue.py:4-26: acc (0,0,1)->(0,0,1), mag (-1,0,0)->(1,0,0),
    # weights .5/.5  =>  R = diag(-1,-1,1), and R.mag_init = (1,0,0)
    w = O.OracleWahba(np.asarray([0.0, 0.0, 1.0]), np.asarray([-1.0, 0.0, 0.0]))
    R = w.rotation(np.asarray([0.0, 0.0, 1.0]), np.asarray([1.0, 0.0, 0.0]), 0.5, 0.5)
    np.testing.assert_allclose(R, np.diag([-1.0, -1.0, 1.0]), atol=1e-15)
    np.testing.assert_allclose(golden_wahba["hand_check_R"], np.diag([-1.0, -1.0, 1.0]), atol=1e-15)
    np.testing.assert_allclose(R @ np.asarray([-1.0, 0.0, 0.0]), [1.0, 0.0, 0.0], atol=1e-15)


def test_rk4_known_answer(golden_rk4):
    # Quarternions.py:19-41,99-112: omega=[3pi/2,pi,pi/2] for 1 s in 10^j steps
    w = golden_rk4["omega"]
    for n_it in (1, 10, 100, 1000):
        q = np.asarray([1.0, 0.0, 0.0, 0.0])
        for _ in range(n_it):
            q = O.rk4_seconds(q, 1.0 / n_it, w)
        np.testing.assert_array_equal(q, golden_rk4[f"steps_{n_it}"])
    # the converged value is the analytic exponential
    a = np.linalg.norm(w)
    exact = np.concatenate([[np.cos(a / 2)], np.sin(a / 2) * w / a])
    np.testing.assert_allclose(golden_rk4["steps_1000"], exact, atol=1e-12)
    # the ns-based form used by the filter gives the same step
    q1 = O.rk4(np.asarray([1.0, 0.0, 0.0, 0.0]), 10 ** 8, w)
    np.testing.assert_allclose(q1, O.rk4_seconds(np.asarray([1.0, 0.0, 0.0, 0.0]), 0.1, w), atol=1e-15)


def test_replay_scalar_equals_reference(golden_traj):
    g = golden_traj
    for tag in ("clean", "noisy"):
        S = g[f"{tag}_streams"].astype(np.float64)
        T = S.shape[0]
        t_ns = np.arange(T + 1, dtype=np.int64) * 10 ** 7
        for n in (0, 3, 6, 7):
            X, P, flips, ys = O.replay_scalar(t_ns, S[:, 0:3, n], S[:, 3:6, n], S[:, 6:9, n],
                                              g[f"{tag}_acc_ref"][:, n].astype(np.float64),
                                              g[f"{tag}_mag_ref"][:, n].astype(np.float64),
                                              g[f"{tag}_q"][n], g[f"{tag}_r"][n], return_aux=True)
            # same operations in the same order: bit-for-bit
            np.testing.assert_array_equal(X, g[f"{tag}_X"][:, n])
            np.testing.assert_array_equal(P, g[f"{tag}_P"][n])
            np.testing.assert_array_equal(flips, g[f"{tag}_flips"][:, n])
            np.testing.assert_array_equal(ys, g[f"{tag}_y"][:, n])


def test_replay_batched_matches_reference(golden_traj):
    g = golden_traj
    for tag in ("clean", "noisy"):
        S = g[f"{tag}_streams"].astype(np.float64)
        T = S.shape[0]
        out = O.replay_batched(np.full(T, 1e7), S[:, 0:3], S[:, 3:6], S[:, 6:9], g[f"{tag}_acc_ref"].T,
                               g[f"{tag}_mag_ref"].T, g[f"{tag}_q"], g[f"{tag}_r"])
        assert O.quat_angle(out["X"], g[f"{tag}_X"]).max() < 1e-9
        np.testing.assert_allclose(out["P_final"], g[f"{tag}_P"], rtol=1e-6, atol=1e-12)
        assert (out["flips"] == g[f"{tag}_flips"]).all()


def test_stepwise_functions(golden_step):
    g = golden_step
    for n in range(0, 64, 7):
        k = O.OracleEKF(1000, g["mag0"][n].astype(np.float64), g["acc0"][n].astype(np.float64))
        k.set_q(2.0); k.set_q(1.5); k.set_r(float(g["r_scale"]))
        assert k.Q[0, 0] == 3.0                       # cumulative setQ  (ExtendedKalmanFilter.py:12-13)
        x, P, w = g["x"][n].astype(np.float64), g["P"][n].astype(np.float64), g["gyro"][n].astype(np.float64)
        z, Pp, K = k.predict(w, 1000 + int(g["dt_ns"][n]), x, P)
        np.testing.assert_array_equal(z, g["z"][n])
        np.testing.assert_array_equal(Pp, g["P_pred"][n])
        np.testing.assert_array_equal(K, g["K"][n])
        X, Pc = k.correct(g["mag"][n].astype(np.float64), g["acc"][n].astype(np.float64), z, Pp, K)
        np.testing.assert_array_equal(X, g["X"][n])
        np.testing.assert_array_equal(Pc, g["P_corr"][n])
        np.testing.assert_array_equal(O.half_omega(w), g["JA"][n])
        np.testing.assert_array_equal(O.jacobian_b(x), g["JB"][n])
        np.testing.assert_array_equal(O.comparator(x, z), g["comparator"][n])
        assert O.comparator(x, z)[0] == np.dot(np.asarray([x[0], x[1], x[2], x[3]]), z) or \
            abs(O.comparator(x, z)[0] - np.dot(x, z)) < 1e-15
        np.testing.assert_array_equal(O.rk4(x, int(g["dt_ns"][n]), w), g["rk4"][n])
        np.testing.assert_array_equal(O.quat_to_rpy_deg(x), g["rpy"][n])
        assert O.norm(P[0]) == g["norm"][n]
    assert O.dimensional_split(g["split_in"].tolist()) == g["split_out"].tolist()


def test_wahba_and_rot2quat(golden_wahba):
    g = golden_wahba
    for tag in ("half", "refw"):
        for n in range(0, 1500, 97):
            w = O.OracleWahba(g["acc_ref"][n].astype(np.float64), g["mag_ref"][n].astype(np.float64))
            R = w.rotation(g["acc"][n].astype(np.float64), g["mag"][n].astype(np.float64), g[f"{tag}_ka"][n], g[f"{tag}_km"][n])
            np.testing.assert_array_equal(R, g[f"{tag}_R"][n])
            np.testing.assert_array_equal(O.rotation_to_quat(R), g[f"{tag}_q"][n])
        qb = O.wahba_batched(g["acc_ref"].astype(np.float64), g["mag_ref"].astype(np.float64), g["acc"].astype(np.float64),
                             g["mag"].astype(np.float64), g[f"{tag}_ka"], g[f"{tag}_km"])
        np.testing.assert_allclose(qb, g[f"{tag}_q"], atol=1e-9)
    with np.errstate(all="ignore"):
        out = np.array([O.rotation_to_quat(m) for m in g["r2q_in"]])
        outb = O.rotation_to_quat_batched(g["r2q_in"])
    np.testing.assert_array_equal(out, g["r2q_out"])
    np.testing.assert_array_equal(outb, g["r2q_out"])
    # exact identity -> [nan, nan, nan, 0]  (SURVEY.md section 0.4)
    ident = out[64]
    assert np.isnan(ident[:3]).all() and ident[3] == 0.0


def test_lowpass_closed_form():
    # y <- a x + (1-a) y from 0 with constant input x: y_t = x (1 - (1-a)^t)   (Test.py:27-33)
    x = np.tile(np.asarray([0.3, -1.2, 2.0]), (50, 1))
    y = O.lowpass_scalar(x, 0.1)
    t = np.arange(1, 51)[:, None]
    np.testing.assert_allclose(y, x * (1 - 0.9 ** t), rtol=1e-12)


def test_oracle_equals_reference_on_edge_cases(golden_edge):
    """Caller-supplied non-unit X0 with a full P0, and un-normalised sensors (|a_z| > 1: negative magnetometer
    weight), frozen from the unmodified reference (tests/golden/make_golden.py edge_cases): bit-for-bit."""
    g = golden_edge
    T = g["state_streams"].shape[0]
    t_ns = np.arange(T + 1, dtype=np.int64) * 10 ** 7
    for tag, use_x0 in (("state", True), ("sensors", False), ("both", True)):
        S = g[f"{tag}_streams"].astype(np.float64)
        if tag != "state":
            az = np.abs(S[:, 5])
            assert (az > 1).mean() > 0.1 and (az < 1).mean() > 0.1
        for n in range(S.shape[2]):
            X, P, flips, _ = O.replay_scalar(t_ns, S[:, 0:3, n], S[:, 3:6, n], S[:, 6:9, n], g["acc_ref"][:, n].astype(np.float64),
                                             g["mag_ref"][:, n].astype(np.float64), float(g["q"]), float(g["r"]),
                                             x0=g["x0"][n].astype(np.float64) if use_x0 else None,
                                             P0=g["P0"][n].astype(np.float64) if use_x0 else None, return_aux=True)
            np.testing.assert_array_equal(X, g[f"{tag}_X"][:, n])
            np.testing.assert_array_equal(P, g[f"{tag}_P"][n])
            np.testing.assert_array_equal(flips, g[f"{tag}_flips"][:, n])


def test_preprocessing_restatements_equal_the_reference_cpp():
    """SURVEY 8f-2 / f-2b: the oracle's interpolate / normalise / initial-values restatements against fixtures frozen
    from the reference's OWN C++ (oracle/_ref: InitialValues.cpp compiled as is, Parser.cpp:221-228,259-267 extracted at
    build time; tests/golden/make_golden_cpp.py): bit for bit."""
    import os
    from tests.conftest import GOLDEN
    g = np.load(os.path.join(GOLDEN, "preprocess_ref.npz"))
    np.testing.assert_array_equal(O.interpolate_sensor(g["y1"], g["y2"], g["t1"], g["t2"], g["t3"]), g["interpolated"])
    np.testing.assert_array_equal(O.interpolate_normalise(g["y1"], g["y2"], g["t1"], g["t2"], g["t3"]), g["normalised"])
    assert (g["t3"] == g["t1"]).sum() >= 64 and (g["t3"] > g["t2"]).sum() >= 64        # end points and extrapolation covered
    h = np.load(os.path.join(GOLDEN, "initial_values_ref.npz"))
    mean, var = O.initial_values(h["samples"])
    np.testing.assert_array_equal(mean, h["avg"])
    np.testing.assert_array_equal(var, h["var"])
    np.testing.assert_array_equal(O.normalize_values(mean), h["avg_unit"])
