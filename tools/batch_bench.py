#!/usr/bin/env python
"""Cost of replaying a batch of recordings, each with its own time steps and length, in one launch (one GPU, CUDA
events, variants alternated, medians):

  * the config-2 shape (1 Mi filters x 1000 steps, 16 Ki distinct trajectories, resident in HBM) with one scalar dt
    (the existing launch), with per-stream dt [T, N] and full lengths, and with per-stream dt and lengths uniform in
    [T/2, T];
  * a pooled (Q,R) sweep: 64 recordings x a 64x64 grid x 5000 steps in one `run_c3` call (tangent innovation
    objective), against the 64 single-recording sweeps of the same recordings run back to back.

  python tools/batch_bench.py [--reps 7] [--out profiles/r05_batch_recordings.json]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else None
    except Exception:
        return None


def timed(fn):
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def median(v):
    return sorted(v)[len(v) // 2]


def alternate(fns: dict, reps: int) -> dict:
    """Each variant once as a warm-up, then `reps` rounds that run every variant once in turn."""
    import torch
    for f in fns.values():
        f()
    torch.cuda.synchronize()
    ms = {k: [] for k in fns}
    for _ in range(reps):
        for k, f in fns.items():
            ms[k].append(timed(f))
    return {k: {"ms": v, "ms_median": median(v)} for k, v in ms.items()}


def synthetic_logs(K, T, seed, device):
    """K recordings of T samples (LogData) with timestamps jittered by +-20 % around 100 Hz."""
    import numpy as np
    from poseestimationkf_b200.logio import LogData
    from poseestimationkf_b200.synth import make_imu
    imu = make_imu(K, T, seed=seed, sigma=0.01, device=device)
    S = imu.streams.double().cpu().numpy()
    ar, mr = imu.acc_ref.double().cpu().numpy(), imu.mag_ref.double().cpu().numpy()
    rng = np.random.default_rng(seed)
    logs = []
    for k in range(K):
        t = np.concatenate([[0], np.cumsum(np.rint(1e7 * (1 + 0.2 * rng.uniform(-1, 1, T))))]).astype(np.int64)
        logs.append(LogData(mag_0=mr[:, k], acc_0=ar[:, k], gyro=S[:, 0:3, k], acc_1=S[:, 3:6, k], mag_1=S[:, 6:9, k],
                            timestamp=t[:, None]))
    return logs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--filters", type=int, default=1 << 20)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--recordings", type=int, default=64)
    ap.add_argument("--sweep-steps", type=int, default=5000)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_batch_recordings.json"))
    a = ap.parse_args()
    import torch
    from poseestimationkf_b200 import batched as B
    from poseestimationkf_b200 import workloads as WL
    assert torch.cuda.is_available(), "needs a GPU"
    dev = torch.device("cuda:0")
    res = {"card": card(), "torch": torch.__version__,
           "timing": "CUDA events around each call, one warm-up per variant, variants alternated, medians"}

    # ---- config-2 shape ------------------------------------------------------------------------
    N, T, base = a.filters, a.steps, 1 << 14
    w = WL.build_c2(N, T, dev)
    g = torch.Generator(device=dev).manual_seed(5)
    # one jittered dt column per distinct trajectory, shared by its replicas (they are one recording with its own noise)
    d = (0.01 * (1 + 0.2 * (2 * torch.rand((T, base), generator=g, device=dev) - 1))).float()
    dt_cols = d.repeat(1, N // base).contiguous()
    full = torch.full((N,), T, dtype=torch.int32, device=dev)
    ragged = torch.randint(T // 2, T + 1, (base,), generator=g, device=dev).to(torch.int32).repeat(N // base).contiguous()

    def run(dt, lengths):
        return lambda: B.replay(w.streams, w.acc_ref, w.mag_ref, dt=dt, q=w.q, r=w.r, lengths=lengths,
                                state=B.ReplayState.initial(N, dev, r=w.r))
    st0, st1 = run(0.01, None)()[0], run(dt_cols, full)()[0]
    torch.cuda.synchronize()
    c2 = alternate({"scalar_dt": run(0.01, None), "per_stream_dt": run(dt_cols, full),
                    "per_stream_dt_ragged": run(dt_cols, ragged)}, a.reps)
    for k in c2:
        c2[k]["gsteps_per_s"] = N * T / (c2[k]["ms_median"] * 1e-3) / 1e9
    c2["per_stream_over_scalar"] = c2["per_stream_dt"]["ms_median"] / c2["scalar_dt"]["ms_median"]
    c2["ragged_over_scalar"] = c2["per_stream_dt_ragged"]["ms_median"] / c2["scalar_dt"]["ms_median"]
    c2["ragged_live_fraction"] = float(ragged.double().sum()) / (N * T)
    c2["finite"] = bool(torch.isfinite(st1.x).all())
    c2["workload"] = (f"{N} filters x {T} steps, {base} distinct trajectories (replicated, own noise), streams resident "
                      f"({N * T * 36 / 1e9:.0f} GB + {N * T * 4 / 1e9:.0f} GB of dt columns); state set-up included, as in "
                      f"every variant")
    res["c2"] = c2
    del w, dt_cols, st0, st1
    torch.cuda.empty_cache()

    # ---- pooled sweep against single-recording sweeps -----------------------------------------------
    K, Ts = a.recordings, a.sweep_steps
    logs = synthetic_logs(K, Ts, 55, dev)
    multi = WL.build_multi_recording_sweep(logs, dev)
    singles = [WL.build_recording_sweep(lg, dev, lo=-7.0) for lg in logs]

    def run_singles():
        for s in singles:
            WL.run_c3(s, objective="innovation_tangent")
    sw = alternate({"pooled": lambda: WL.run_c3(multi, objective="innovation_tangent"), "singles_back_to_back": run_singles},
                   max(3, a.reps // 2))
    fsteps = multi.n_filters * Ts
    for k in ("pooled", "singles_back_to_back"):
        sw[k]["gsteps_per_s"] = fsteps / (sw[k]["ms_median"] * 1e-3) / 1e9
    sw["speedup"] = sw["singles_back_to_back"]["ms_median"] / sw["pooled"]["ms_median"]
    nll, nis = WL.pooled_innovation_surface(multi, WL.run_c3(multi, objective="innovation_tangent"))
    bi, G = int(nll.argmin()), multi.qs.numel()
    sw["argmin"] = {"q": float(multi.qs[bi // G]), "r": float(multi.rs[bi % G]), "mean_nis": float(nis.view(-1)[bi])}
    sw["workload"] = (f"{K} recordings x {Ts} steps (dt jittered +-20 %), 64x64 grid from 1e-7 in steps of 0.1 decade, "
                      f"tangent innovation objective: {multi.n_filters} filters in one call against {K} calls of 4096")
    res["pooled_sweep"] = sw
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({"card": res["card"],
                      "c2": {k: (v["ms_median"] if isinstance(v, dict) else v) for k, v in c2.items() if k != "workload"},
                      "pooled": {k: (v["ms_median"] if isinstance(v, dict) and "ms_median" in v else v)
                                 for k, v in sw.items() if k != "workload"}}, indent=1))


if __name__ == "__main__":
    main()
