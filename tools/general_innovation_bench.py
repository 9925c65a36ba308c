#!/usr/bin/env python
"""Cost of the innovation terms and the gate with general Q and R matrices (B.replay_general; one GPU, CUDA events,
variants alternated, medians):

  * the config-2 shape (1 Mi filters x 1000 steps, 16 Ki distinct trajectories, resident in HBM) with one full Q and one
    full anisotropic R: the general replay, + tangent sums, + tangent sums and the gate, + per-step output;
  * one recording x 30 000 steps under 16^3 diagonal-Q candidates (4096 filters, one matrix sweep), beside the isotropic
    64x64 tangent (Q,R) sweep of the same recording (4096 cells).

  python tools/general_innovation_bench.py [--reps 7] [--out profiles/r10_general_innovation.json]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from batch_bench import alternate, card  # noqa: E402
from general_qr_bench import _spd  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--filters", type=int, default=1 << 20)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--sweep-steps", type=int, default=30000)
    ap.add_argument("--grid", type=int, default=16)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r10_general_innovation.json"))
    a = ap.parse_args()
    import numpy as np
    import torch
    from poseestimationkf_b200 import batched as B
    from poseestimationkf_b200 import workloads as WL
    from poseestimationkf_b200.synth import make_imu
    assert torch.cuda.is_available(), "needs a GPU"
    dev = torch.device("cuda:0")
    res = {"card": card(), "torch": torch.__version__,
           "timing": "CUDA events around each call, one warm-up per variant, variants alternated, medians"}

    # ---- config-2 shape ------------------------------------------------------------------------
    N, T = a.filters, a.steps
    w = WL.build_c2(N, T, dev)
    rng = np.random.default_rng(1)
    Q = torch.tensor(_spd(rng, 3, [0.5, 1.0, 2.0]), device=dev)
    R = torch.tensor(_spd(rng, 4, [0.05, 0.08, 0.12, 0.2]), device=dev)
    out = torch.empty((2, T, N), dtype=torch.float32, device=dev)

    def run(sums=False, gate=None, steps=False):
        return lambda: B.replay_general(w.streams, w.acc_ref, w.mag_ref, dt=0.01, q=Q, r=R,
                                        innovation=True if sums else None, innovation_model="tangent", gate=gate,
                                        out_innovation=out if steps else None, state=B.ReplayState.initial(N, dev, r=1.0))
    c2 = alternate({"general": run(), "tangent_sums": run(sums=True),
                    "tangent_sums_gate": run(sums=True, gate=B.GATE_CHI2_3_999),
                    "tangent_sums_steps": run(sums=True, steps=True)}, a.reps)
    for k in list(c2):
        c2[k]["gsteps_per_s"] = N * T / (c2[k]["ms_median"] * 1e-3) / 1e9
    base = c2["general"]["ms_median"]
    for k in ("tangent_sums", "tangent_sums_gate", "tangent_sums_steps"):
        c2[f"{k}_over_general"] = c2[k]["ms_median"] / base
    c2["target_tangent_sums_over_general"] = 1.3
    c2["workload"] = (f"{N} filters x {T} steps, 16384 distinct trajectories (replicated, own noise), streams resident "
                      f"({N * T * 36 / 1e9:.0f} GB); one full Q (eigenvalues 0.5, 1, 2) and one full R (eigenvalues 0.05, "
                      f"0.08, 0.12, 0.2) shared by the launch, automatic staging (the scalar TMA kernel); gate at the "
                      f"chi^2_3 0.999 quantile; steps writes [2,T,N] ({N * T * 8 / 1e9:.0f} GB) into one preallocated "
                      f"tensor; state set-up included in every variant")
    c2["Q"], c2["R"] = Q.tolist(), R.tolist()
    res["c2"] = c2
    del w, out
    torch.cuda.empty_cache()

    # ---- one recording x 30 000 steps: 16^3 diagonal-Q candidates against the isotropic 64x64 sweep ------------
    Ts, G, G3 = a.sweep_steps, WL.C3_GRID, a.grid
    imu = make_imu(1, Ts, seed=9, sigma=0.01, dt=0.01, device=dev)
    b = types.SimpleNamespace(streams=imu.streams, acc_ref=imu.acc_ref, mag_ref=imu.mag_ref, dt=imu.dt, lengths=None)
    g = np.logspace(-7, -7 + 0.2 * (G3 - 1), G3)
    Qs = np.stack([np.diag([x, y, z]) for x in g for y in g for z in g])
    mw = WL.build_matrix_sweep(b, Qs, np.eye(4) * 1e-4)
    qs = torch.logspace(-7, -7 + 0.1 * (G - 1), G, device=dev)
    iw = WL.SweepWorkload(imu.streams, imu.acc_ref, imu.mag_ref, None, qs, qs, qs.repeat_interleave(G).contiguous(),
                          qs.repeat(G).contiguous(), imu.dt)
    B.general_qr_tri(mw.q, mw.r, mw.n_filters, dev)          # (the one-time matrix checks, cached per tensor)
    sw = alternate({"matrix_sweep_16x16x16": lambda: WL.run_matrix_sweep(mw, "innovation_tangent"),
                    "isotropic_sweep_64x64": lambda: WL.run_c3(iw, objective="innovation_tangent")}, a.reps)
    sw["matrix_over_isotropic"] = sw["matrix_sweep_16x16x16"]["ms_median"] / sw["isotropic_sweep_64x64"]["ms_median"]
    nll, nis = WL.matrix_innovation_surface(mw, WL.run_matrix_sweep(mw, "innovation_tangent"))
    k = int(torch.argmin(nll))
    sw["argmin_diag_q"] = [float(v) for v in np.diag(Qs[k])]
    sw["nll_at_argmin"], sw["mean_nis_at_argmin"] = float(nll[k]), float(nis[k])
    sw["workload"] = (f"1 recording (sigma = 0.01) x {Ts} steps; matrix sweep: {G3}^3 diagonal Q (log-spaced from 1e-7 in "
                      f"0.2 decades per axis) with R = 1e-4 I, {len(Qs)} filters with per-filter matrices, tangent sums; "
                      f"isotropic: {G}x{G} (Q,R) grid (log-spaced from 1e-7 in 0.1 decades), {G * G} filters, tangent "
                      f"sums, automatic precision")
    res["sweep"] = sw

    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({"card": res["card"],
                      "c2": {k: (v["ms_median"] if isinstance(v, dict) else v) for k, v in c2.items()
                             if k not in ("workload", "Q", "R")},
                      "sweep": {k: (v["ms_median"] if isinstance(v, dict) else v) for k, v in sw.items() if k != "workload"}},
                     indent=1))


if __name__ == "__main__":
    main()
