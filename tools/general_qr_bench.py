#!/usr/bin/env python
"""Cost and accuracy of the replay with general Q and R matrices (replay(q=<3x3>, r=<4x4>), one GPU, CUDA events, variants
alternated, medians):

  * the config-2 shape (1 Mi filters x 1000 steps, streams resident in HBM) with one full Q and one anisotropic full R
    (eigenvalues 0.5-2 and 0.05-0.2 around the default q = 1, r = 0.1), against the isotropic scalar TMA kernel (the
    like-for-like baseline: the general kernel is a scalar TMA kernel) and against the default (packed) launch, both at
    q = 1, r = 0.1;
  * the measured error against the float64 definition (tests/general_qr_ref.py) inside and outside the plain variant's
    range of eigenvalue ratios (lambda(R)/lambda(Q) <= 100, lambda(Q)/lambda(R) <= 1e4).

  python tools/general_qr_bench.py [--reps 7] [--out profiles/r07_general_qr.json]
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from batch_bench import alternate, card  # noqa: E402


def _spd(rng, k, eig):
    import numpy as np
    V = np.linalg.qr(rng.standard_normal((k, k)))[0]
    return V @ np.diag(eig) @ V.T


def accuracy(dev, N=256, T=1000):
    """Max angle [rad] to the float64 definition over N filters x T steps, QR2 Wahba, TMA staging, for eigenvalue
    ratios inside and outside the plain variant's range (random eigenvectors, one pair of matrices per filter)."""
    import numpy as np
    import torch
    from oracle import ekf_oracle as O
    from poseestimationkf_b200 import batched as B
    from poseestimationkf_b200.synth import make_imu
    from tests import general_qr_ref as GR
    imu = make_imu(N, T, seed=41, sigma=0.01, device=dev)
    S = imu.streams.cpu().numpy().astype(np.float64)
    ar, mr = imu.acc_ref.cpu().numpy().T.astype(np.float64), imu.mag_ref.cpu().numpy().T.astype(np.float64)
    out = {}
    # (Q eigenvalue range, R eigenvalue range): the largest ratio of the two spectra is the one named
    cases = {"R/Q=1e1": ((1e-3, 1e-2), (1e-2, 1e-1)), "R/Q=1e2": ((1e-3, 1e-3), (1e-1, 1e-1)),
             "R/Q=1e3": ((1e-4, 1e-4), (1e-1, 1e-1)), "R/Q=1e4": ((1e-5, 1e-5), (1e-1, 1e-1)),
             "Q/R=1e4": ((1e-1, 1e-1), (1e-5, 1e-5)), "Q/R=1e5": ((1e0, 1e0), (1e-5, 1e-5)),
             "Q/R=1e6": ((1e0, 1e0), (1e-6, 1e-6))}
    rng = np.random.default_rng(0)
    for name, (ql, rl) in cases.items():
        Q = GR.random_spd(rng, N, 3, *ql) if ql[0] != ql[1] else np.stack([_spd(rng, 3, np.full(3, ql[0]) * [1, 1.5, 2]) for _ in range(N)])
        R = GR.random_spd(rng, N, 4, *rl) if rl[0] != rl[1] else np.stack([_spd(rng, 4, np.full(4, rl[0]) * [0.5, 0.75, 1, 1]) for _ in range(N)])
        st, traj, flips = B.replay(imu.streams, imu.acc_ref, imu.mag_ref, dt=imu.dt, q=torch.tensor(Q, device=dev),
                                   r=torch.tensor(R, device=dev), staging="tma", store_trajectory=True, store_flips=True)
        U = lambda M: np.triu(M).astype(np.float32).astype(np.float64)
        f32 = lambda M: U(M) + np.swapaxes(np.triu(U(M), 1), -1, -2)
        ref = GR.replay_general(np.full(T, float(np.float32(imu.dt)) * 1e9), S[:, 0:3], S[:, 3:6], S[:, 6:9], ar, mr,
                                f32(Q), f32(R))
        ang = O.quat_angle(traj.cpu().numpy().astype(np.float64), ref["X"])
        lq, lr = np.linalg.eigvalsh(f32(Q)), np.linalg.eigvalsh(f32(R))
        out[name] = {"max_rad": float(ang.max()), "flip_mismatches": int((flips.cpu().numpy().astype(bool) != ref["flips"]).sum()),
                     "max_lambdaR_over_lambdaQ": float((lr.max(1) / lq.min(1)).max()),
                     "max_lambdaQ_over_lambdaR": float((lq.max(1) / lr.min(1)).max())}
    return {"workload": f"{N} filters x {T} steps, sigma = 0.01, QR2 Wahba, TMA staging", "cases": out}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--filters", type=int, default=1 << 20)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_general_qr.json"))
    a = ap.parse_args()
    import numpy as np
    import torch
    from poseestimationkf_b200 import batched as B
    from poseestimationkf_b200 import workloads as WL
    assert torch.cuda.is_available(), "needs a GPU"
    dev = torch.device("cuda:0")
    res = {"card": card(), "torch": torch.__version__,
           "timing": "CUDA events around each call, one warm-up per variant, variants alternated, medians"}

    N, T = a.filters, a.steps
    w = WL.build_c2(N, T, dev)
    rng = np.random.default_rng(1)
    Q = torch.tensor(_spd(rng, 3, [0.5, 1.0, 2.0]), device=dev)
    R = torch.tensor(_spd(rng, 4, [0.05, 0.08, 0.12, 0.2]), device=dev)

    def run(general, staging):
        q, r = (Q, R) if general else (w.q, w.r)
        return lambda: B.replay(w.streams, w.acc_ref, w.mag_ref, dt=0.01, q=q, r=r, staging=staging,
                                state=B.ReplayState.initial(N, dev, r=1.0 if general else w.r))
    c2 = alternate({"isotropic_tma": run(False, "tma"), "general_tma": run(True, "tma"),
                    "isotropic_packed_default": run(False, "auto")}, a.reps)
    for k in list(c2):
        c2[k]["gsteps_per_s"] = N * T / (c2[k]["ms_median"] * 1e-3) / 1e9
    c2["general_over_isotropic_tma"] = c2["general_tma"]["ms_median"] / c2["isotropic_tma"]["ms_median"]
    c2["general_over_packed_default"] = c2["general_tma"]["ms_median"] / c2["isotropic_packed_default"]["ms_median"]
    c2["workload"] = (f"{N} filters x {T} steps, 16384 distinct trajectories (replicated, own noise), streams resident "
                      f"({N * T * 36 / 1e9:.0f} GB); general: one full Q (eigenvalues 0.5, 1, 2) and one full R (eigenvalues "
                      f"0.05, 0.08, 0.12, 0.2) shared by the launch; isotropic: q = 1, r = 0.1 per filter; state set-up "
                      f"included in every variant")
    c2["Q"], c2["R"] = Q.tolist(), R.tolist()
    res["c2"] = c2
    del w
    torch.cuda.empty_cache()
    res["accuracy"] = accuracy(dev)

    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({"card": res["card"],
                      "c2": {k: (v["ms_median"] if isinstance(v, dict) else v) for k, v in c2.items()
                             if k not in ("workload", "Q", "R")},
                      "accuracy": {k: v["max_rad"] for k, v in res["accuracy"]["cases"].items()}}, indent=1))


if __name__ == "__main__":
    main()
