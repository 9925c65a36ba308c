#!/usr/bin/env python
"""Cost of the per-step innovation output (replay(out_innovation=...), one GPU, CUDA events, variants alternated,
medians):

  * the config-2 shape (1 Mi filters x 1000 steps, 16 Ki distinct trajectories, resident in HBM): the replay that
    stores the trajectory (the per-step output it is compared with), the tangent-model replay with the per-step
    output, with and without the trajectory, and the tangent-model sums alone;
  * one recording under a 64x64 (Q,R) sweep x 30 000 steps with the per-step output, and the windowed surfaces
    (`workloads.window_innovation_nll`, 10 windows of 3000 steps) from it.

  python tools/innovation_steps_bench.py [--reps 7] [--out profiles/r09_innovation_steps.json]
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--filters", type=int, default=1 << 20)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--sweep-steps", type=int, default=30000)
    ap.add_argument("--windows", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r09_innovation_steps.json"))
    a = ap.parse_args()
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
    traj = torch.empty((T, N, 4), dtype=torch.float32, device=dev)
    out = torch.empty((2, T, N), dtype=torch.float32, device=dev)

    def run(with_traj, steps, sums=False):
        return lambda: B.replay(w.streams, w.acc_ref, w.mag_ref, dt=0.01, q=w.q, r=w.r,
                                out_traj=traj if with_traj else None, out_innovation=out if steps else None,
                                innovation=True if sums else None, innovation_model="tangent",
                                state=B.ReplayState.initial(N, dev, r=w.r))
    c2 = alternate({"traj": run(True, False), "steps": run(False, True), "steps_traj": run(True, True),
                    "sums_only": run(False, False, sums=True)}, a.reps)
    for k in list(c2):
        c2[k]["gsteps_per_s"] = N * T / (c2[k]["ms_median"] * 1e-3) / 1e9
    c2["steps_over_traj"] = c2["steps"]["ms_median"] / c2["traj"]["ms_median"]
    c2["steps_traj_over_traj"] = c2["steps_traj"]["ms_median"] / c2["traj"]["ms_median"]
    c2["target_steps_over_traj"] = 1.15
    c2["workload"] = (f"{N} filters x {T} steps, 16384 distinct trajectories (replicated, own noise), streams resident "
                      f"({N * T * 36 / 1e9:.0f} GB), q = 1, r = 0.1, tangent model; state set-up included in every "
                      f"variant; traj writes [T,N,4] ({N * T * 16 / 1e9:.0f} GB), steps writes [2,T,N] "
                      f"({N * T * 8 / 1e9:.0f} GB), each into one preallocated tensor; sums_only accumulates innov_acc "
                      f"and writes no per-step output")
    res["c2"] = c2
    del w, traj, out
    torch.cuda.empty_cache()

    # ---- one recording, 64x64 (Q,R) sweep x 30 000 steps, per-step output ------------------------------
    Ts, G = a.sweep_steps, WL.C3_GRID
    imu = make_imu(1, Ts, seed=9, sigma=0.01, dt=0.01, device=dev)
    qs = torch.logspace(-7, -7 + 0.1 * (G - 1), G, device=dev)
    q = qs.repeat_interleave(G).contiguous()
    r = qs.repeat(G).contiguous()
    Nw = G * G
    outs = torch.empty((2, Ts, Nw), dtype=torch.float32, device=dev)
    Wn = a.windows
    edges = torch.linspace(0, Ts, Wn + 1, device=dev).round().long()
    bounds = torch.stack((edges[:-1], edges[1:]), 1)[:, None, :]            # [W, 1, 2]

    def sweep():
        return B.replay(imu.streams, imu.acc_ref, imu.mag_ref, dt=imu.dt, q=q, r=r, n_filters=Nw,
                        innovation_model="tangent", out_innovation=outs)

    def surfaces():
        return WL.window_innovation_nll(outs, bounds, 3)
    sw = alternate({"sweep_with_steps": sweep, "window_surfaces": surfaces}, a.reps)
    nll, nis = surfaces()
    per_step = nll / (bounds[..., 1] - bounds[..., 0]).double()
    argmin = per_step.view(Wn, G, G).flatten(1).argmin(1)
    sw["windows"] = [{"steps": [int(bounds[k, 0, 0]), int(bounds[k, 0, 1])],
                      "argmin_q": float(qs[argmin[k] // G]), "argmin_r": float(qs[argmin[k] % G]),
                      "mean_nis_at_argmin": float(nis[k, argmin[k]])} for k in range(Wn)]
    sw["workload"] = (f"1 recording (sigma = 0.01) x {Ts} steps under a {G}x{G} (Q,R) grid (log-spaced from 1e-7 in "
                      f"0.1 decades) = {Nw} filters, tangent model, per-step output [2,{Ts},{Nw}] "
                      f"({2 * Ts * Nw * 4 / 1e9:.2f} GB); automatic precision (whole batch); window_surfaces: "
                      f"{Wn} windows of {Ts // Wn} steps, float64 prefix sums on the device")
    res["sweep"] = sw

    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({"card": res["card"],
                      "c2": {k: (v["ms_median"] if isinstance(v, dict) else v) for k, v in c2.items() if k != "workload"},
                      "sweep": {k: sw[k]["ms_median"] for k in ("sweep_with_steps", "window_surfaces")}}, indent=1))


if __name__ == "__main__":
    main()
