#!/usr/bin/env python
"""Cost and effect of the innovation gate (replay(gate=...), one GPU, CUDA events, variants alternated, medians):

  * the config-2 shape (1 Mi filters x 1000 steps, 16 Ki distinct trajectories, resident in HBM), gated against
    ungated, without and with the trajectory output;
  * the config-3 sweep (64x64 (Q,R) grid x 16 trajectories x 5000 steps), gated against ungated, with the truth
    objective (`run_c3` default) and with no objective;
  * the disturbed scenario (sigma = 0.01 data, 3 magnetometer disturbances of 100-300 steps per recording, (q, r) =
    (7.9e-6, 1e-4), gate 16.27 = the 0.999 quantile of chi^2_3) at GPU scale: RMS / max angle to the ground truth,
    gated against ungated.

  python tools/gate_bench.py [--reps 7] [--out profiles/r06_gating.json]
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
    ap.add_argument("--scenario-filters", type=int, default=1 << 16)
    ap.add_argument("--scenario-steps", type=int, default=1500)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_gating.json"))
    a = ap.parse_args()
    import torch
    from poseestimationkf_b200 import batched as B
    from poseestimationkf_b200 import workloads as WL
    from poseestimationkf_b200.synth import add_disturbances, make_imu
    assert torch.cuda.is_available(), "needs a GPU"
    dev = torch.device("cuda:0")
    gamma = B.GATE_CHI2_3_999
    res = {"card": card(), "torch": torch.__version__, "gate": gamma,
           "timing": "CUDA events around each call, one warm-up per variant, variants alternated, medians"}

    # ---- config-2 shape ------------------------------------------------------------------------
    N, T = a.filters, a.steps
    w = WL.build_c2(N, T, dev)
    traj = torch.empty((T, N, 4), dtype=torch.float32, device=dev)

    def run(gate, with_traj):
        return lambda: B.replay(w.streams, w.acc_ref, w.mag_ref, dt=0.01, q=w.q, r=w.r, gate=gate,
                                out_traj=traj if with_traj else None, state=B.ReplayState.initial(N, dev, r=w.r))
    st = run(gamma, False)()[0]
    torch.cuda.synchronize()
    c2 = alternate({"ungated": run(None, False), "gated": run(gamma, False)}, a.reps)
    c2t = alternate({"ungated_traj": run(None, True), "gated_traj": run(gamma, True)}, a.reps)
    c2.update(c2t)
    for k in list(c2):
        c2[k]["gsteps_per_s"] = N * T / (c2[k]["ms_median"] * 1e-3) / 1e9
    c2["gated_over_ungated"] = c2["gated"]["ms_median"] / c2["ungated"]["ms_median"]
    c2["gated_over_ungated_traj"] = c2["gated_traj"]["ms_median"] / c2["ungated_traj"]["ms_median"]
    c2["gated_fraction"] = float(st.gate_count.double().sum()) / (N * T)
    c2["workload"] = (f"{N} filters x {T} steps, 16384 distinct trajectories (replicated, own noise), streams resident "
                      f"({N * T * 36 / 1e9:.0f} GB), q = {w.q}, r = {w.r}; state set-up included in every variant; the "
                      f"trajectory variants write [T,N,4] ({N * T * 16 / 1e9:.0f} GB) into one preallocated tensor")
    res["c2"] = c2
    del w, traj, st
    torch.cuda.empty_cache()

    # ---- config-3 sweep --------------------------------------------------------------------------
    w3 = WL.build_c3(dev)
    c3 = {}
    for obj in ("truth", "none"):
        r = alternate({"ungated": lambda: WL.run_c3(w3, objective=obj),
                       "gated": lambda: WL.run_c3(w3, objective=obj, gate=gamma)}, a.reps)
        r["gated_over_ungated"] = r["gated"]["ms_median"] / r["ungated"]["ms_median"]
        c3[obj] = r
    c3["workload"] = (f"{w3.n_filters} filters ({w3.qs.numel()}x{w3.rs.numel()} (Q,R) cells x {w3.streams.shape[2]} "
                      f"trajectories) x {w3.streams.shape[0]} steps, automatic precision (mixed plain / precise cells)")
    res["c3"] = c3
    del w3
    torch.cuda.empty_cache()

    # ---- disturbed scenario at GPU scale -----------------------------------------------------------
    Ns, Ts = a.scenario_filters, a.scenario_steps
    imu = make_imu(Ns, Ts, seed=5, sigma=0.01, dt=0.01, device=dev, keep_truth=True)
    mask = add_disturbances(imu.streams, seed=1, n_mag=3)
    truth = imu.q_true.permute(0, 2, 1)                       # [T,N,4] float64
    sc = {"workload": f"{Ns} recordings x {Ts} steps, sigma = 0.01, 3 magnetometer disturbances each "
                      f"(u ~ U(0.15, 0.5), 100-300 steps, start in [200, T-300)), q = 7.9e-6, r = 1e-4",
          "disturbed_fraction": float(mask.double().mean())}
    for name, gate in (("ungated", None), ("gated", gamma)):
        og = torch.empty((Ts, Ns), dtype=torch.uint8, device=dev) if gate is not None else None
        st, tr, _ = B.replay(imu.streams, imu.acc_ref, imu.mag_ref, dt=imu.dt, q=7.9e-6, r=1e-4, gate=gate,
                             store_trajectory=True, out_gated=og)
        d = (tr.double() * truth).sum(-1).abs().clamp(max=1.0)
        ang = torch.rad2deg(2 * torch.acos(d))
        sc[name] = {"rms_deg": float(ang.pow(2).mean().sqrt()), "max_deg": float(ang.max()),
                    "median_recording_rms_deg": float(ang.pow(2).mean(0).sqrt().median()),
                    "recordings_rms_over_10_deg": float((ang.pow(2).mean(0).sqrt() > 10).double().mean())}
        if og is not None:
            g = og.bool()
            sc[name]["gated_of_disturbed"] = float(g[mask].double().mean())
            sc[name]["gated_of_clean"] = float(g[~mask].double().mean())
    sc["rms_ratio"] = sc["ungated"]["rms_deg"] / sc["gated"]["rms_deg"]
    sc["median_recording_ratio"] = sc["ungated"]["median_recording_rms_deg"] / sc["gated"]["median_recording_rms_deg"]
    res["disturbed"] = sc

    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({"card": res["card"],
                      "c2": {k: (v["ms_median"] if isinstance(v, dict) else v) for k, v in c2.items() if k != "workload"},
                      "c3": {o: {k: (v["ms_median"] if isinstance(v, dict) else v) for k, v in c3[o].items()}
                             for o in ("truth", "none")},
                      "disturbed": sc}, indent=1))


if __name__ == "__main__":
    main()
