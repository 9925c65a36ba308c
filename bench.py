#!/usr/bin/env python
"""bench.py -- EKF filter-steps/s of the batched replay on N B200s (contract in the task prompt).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload auto|c2|c3|c4|c5]        our arm
  python bench.py --impl reference ...                the reference's own CPU implementation of the path
  python bench.py ... --dump-outputs DIR              also write what the last timed step computed as DIR/<name>.npy

Workloads (BASELINE.json `configs`, built by poseestimationkf_b200/workloads.py):
  c2  1 Mi independent filters x 1000 steps per GPU, inputs resident in HBM      (configs[1]; the default on 1 GPU)
  c5  16 Mi filters x 2000 steps SHARDED over the ranks, time-chunked with carried state, inputs generated per
      chunk on the device, final states gathered afterwards                      (configs[4]; the default on 2+ GPUs)
  c3  64x64 (Q,R) sweep x 256 trajectories x 5000 steps, loss surface on device  (configs[2])
  c4  Wahba-only, 100 M (acc, mag) pairs                                          (configs[3])

A "step" of the contract = one full pass of the hot path over the workload.  `value` = filter-steps/s with inputs
resident in HBM (device time, CUDA events, MAX over ranks); `e2e` = the same metric through posekf_replay_host_f32
with pinned HOST buffers (H2D of the stream and D2H of the final state inside the timed region).  Filters are
independent: there is no collective on the path; the only communication is the MAX of the timings and, for c5, the
gather of the final states, which is timed apart (`gather_ms`).
"""
from __future__ import annotations

import argparse
import glob
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "ekf_filter_steps_per_s"
UNIT = "filter-steps/s"
# algorithmic work per filter-step (DESIGN.md "Roofline"): bytes streamed and flops executed
BYTES_PER_STEP = 36            # 9 float32 inputs (final-state-only replay)
# Executed arithmetic of the shipped packed kernel, from the dynamic opcode census of its ncu capture
# (profiles/r02_replay_packed_opcode_census.json): FMA / MUL / ADD lane operations + MUFU per filter-step.
# (SURVEY.md's 1570 flops is the un-restructured reference algorithm.)
CENSUS = os.path.join(ROOT, "profiles", "r02_replay_packed_opcode_census.json")
NCU_FULL = os.path.join(ROOT, "profiles", "r02_replay_packed_ncu_full.json")
FLOPS_FALLBACK = {"qr2": 364.0, "jacobi": 1292.0}
LANE_OPS_FALLBACK = {"qr2": 237.0}
FLOPS_COMPENSATED_EXTRA = 32      # two-sum folding of the state
DUMP_BYTES = 64 * 10**6           # --dump-outputs: bound on all arrays together


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="auto", choices=["auto", "c2", "c3", "c4", "c5"],
                    help="auto: c2 on one GPU, c5 (the sharded scaling run) on 2+ GPUs")
    ap.add_argument("--filters", type=int, default=None, help="c2: filters per GPU (1 Mi); c5: filters in total (16 Mi)")
    ap.add_argument("--timesteps", type=int, default=None, help="c2: 1000; c5: 2000")
    ap.add_argument("--wahba", default="qr2", choices=["qr2", "jacobi"])
    ap.add_argument("--staging", default="auto", choices=["auto", "ldg", "tma", "tma_packed"])
    ap.add_argument("--e2e-timesteps", type=int, default=None,
                    help="timesteps of the host-buffer (e2e) replay; default: the workload's own where host memory allows")
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="target wall time of the CPU baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-numa-bind", action="store_true", help="do not pin the process to the CPUs local to its GPU")
    ap.add_argument("--no-variants", action="store_true", help="skip the context measurements of the other kernels")
    ap.add_argument("--precise-state", action="store_true",
                    help="compensated two-float state (needed for R >> Q sweeps, not for the Q=1, R=0.1 headline config)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the arrays the last one returned as DIR/<name>.npy (float32, rank 0, "
                         f"at most {DUMP_BYTES // 10**6} MB: a seeded sample of the filters beyond that); the inputs are "
                         "seeded, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to our arm only (the reference arm returns no arrays)")
    return args


def kernel_source_sha() -> str:
    """Hash of the device sources (comments and white space stripped): profiles are stamped with it, and a profile taken
    from other sources is not quoted."""
    import re
    h = hashlib.sha256()
    for f in ("ekf_math.cuh", "device_util.cuh", "replay_kernels.cuh"):
        src = open(os.path.join(ROOT, "poseestimationkf_b200", "csrc", f), encoding="utf-8").read()
        src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
        src = re.sub(r"//[^\n]*", "", src)
        h.update(re.sub(r"\s+", "", src).encode())
    return h.hexdigest()[:16]


def state_arrays(st) -> dict:
    """What `replay` hands its caller in a ReplayState: x [4,N], p [10,N] (packed P/r) and, where present, the
    compensated low part x_lo [4,N] and the tuning objective loss [N]."""
    out = {"state_x": st.x, "state_p": st.p}
    for name in ("x_lo", "loss"):
        if getattr(st, name) is not None:
            out["state_" + name] = getattr(st, name)
    return out


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Writes {name: tensor [..., N]} (one N for all) as out_dir/<name>.npy in float32.  Where all N columns would
    exceed DUMP_BYTES, every array keeps the same sample of columns, drawn with a fixed seed and kept in order."""
    import numpy as np
    import torch
    n = next(iter(arrays.values())).shape[-1]
    col_bytes = sum(4 * a.numel() // max(n, 1) for a in arrays.values())
    keep = min(n, DUMP_BYTES // col_bytes)
    idx = None if keep == n else torch.randperm(n, generator=torch.Generator().manual_seed(0))[:keep].sort().values
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        if idx is not None:
            a = a[..., idx.to(a.device)]
        np.save(os.path.join(out_dir, name + ".npy"), a.detach().float().cpu().numpy())


def executed_arithmetic(wahba: str):
    """(flops, FP32 lane operations, source) per filter-step of the kernel the bench times."""
    if wahba == "qr2":
        try:
            c = json.load(open(CENSUS))
            lo = c["fp32_lane_ops_per_filter_step"]
            lane = lo["fma"] + lo["mul"] + lo["add"]
            fsel = c["thread_inst_per_filter_step"].get("FSEL", 0.0)
            return c["flops_per_filter_step_executed"], lane + fsel, os.path.relpath(CENSUS, ROOT)
        except Exception:
            pass
    return FLOPS_FALLBACK[wahba], LANE_OPS_FALLBACK.get(wahba), "static estimate (no census for this kernel)"


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's own Python classes where its tree is present, else the oracle's port of them; one
# independent trajectory per worker process, all host cores, driven exactly as PKF/main_file.py:19-47.
# ------------------------------------------------------------------------------------------------
_BARRIER = None


def find_reference():
    """Directory holding the reference's ExtendedKalmanFilter.py / Wahba.py / UtilityFunctions.py, or None."""
    cands = [os.environ.get("POSEKF_REF"), "/root/reference/Python Kalman Filter"]
    cands += glob.glob(os.path.join(ROOT, "baseline", "_ref", "**", "Python Kalman Filter"), recursive=True)
    for c in cands:
        if c and os.path.exists(os.path.join(c, "ExtendedKalmanFilter.py")) and os.path.exists(os.path.join(c, "Wahba.py")):
            return c
    return None


def _cpu_init(barrier):
    global _BARRIER
    _BARRIER = barrier
    for var in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[var] = "1"


def _cpu_worker(args):
    """One independent trajectory through the reference loop (main_file.py:38-47).  Input synthesis is untimed; all
    workers start the timed replay together (barrier) so the rate is a genuine all-cores figure."""
    seed, n_steps, use_barrier, ref_dir = args
    for var in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[var] = "1"
    import numpy as np
    import torch
    torch.set_num_threads(1)
    from poseestimationkf_b200.synth import make_imu
    imu = make_imu(1, n_steps, seed=seed, sigma=0.01)
    S = imu.streams.numpy().astype(np.float64)
    gyro, acc, mag = S[:, 0:3, 0].copy(), S[:, 3:6, 0].copy(), S[:, 6:9, 0].copy()
    t_ns = np.arange(n_steps + 1, dtype=np.int64) * 10 ** 7
    a0, m0 = imu.acc_ref[:, 0].numpy().astype(np.float64), imu.mag_ref[:, 0].numpy().astype(np.float64)
    if ref_dir:
        if ref_dir not in sys.path:
            sys.path.insert(0, ref_dir)
        from ExtendedKalmanFilter import KalmanFilter       # the unmodified reference class
        ekf = KalmanFilter(t_ns[0], m0, a0, 0.5)            # main_file.py:19 (argument order T0, mag_0, acc_0, eps)
        ekf.setQ(1.0); ekf.setR(0.1)                        # :21-22
        predict, correct = ekf.Prediction, ekf.Correction
    else:
        from oracle import ekf_oracle as O                  # the port: same numpy call sequence per step
        ekf = O.OracleEKF(t_ns[0], m0, a0, 0.5)
        ekf.set_q(1.0); ekf.set_r(0.1)
        predict, correct = ekf.predict, ekf.correct
    P = np.identity(4)                                      # :23
    X = np.asarray([1.0, 0.0, 0.0, 0.0])                    # :26
    traj = []
    if use_barrier and _BARRIER is not None:
        _BARRIER.wait()
    t0 = time.perf_counter()
    for i in range(n_steps):                                # :38
        z, P, K = predict(gyro[i], t_ns[i + 1], X, P)       # :39
        X, P = correct(mag[i], acc[i], z, P, K)             # :43
        traj.append(X)                                      # :44
    return time.perf_counter() - t0, float(traj[-1][0])


def cpu_baseline(target_seconds: float, cores: int | None = None):
    """Times the reference path on `cores` processes; returns the cpu_baseline object.  Sample: one independent 100 Hz
    trajectory per core."""
    import multiprocessing as mp
    cores = cores or len(os.sched_getaffinity(0)) or 1
    ref_dir = find_reference()
    dt1, _ = _cpu_worker((0, 300, False, ref_dir))          # calibrate on one short run in this process
    per_step = dt1 / 300
    n_steps = int(max(500, min(20000, target_seconds / per_step)))
    ctx = mp.get_context("spawn")
    barrier = ctx.Barrier(cores)
    with ctx.Pool(cores, initializer=_cpu_init, initargs=(barrier,)) as pool:
        pool.map(_cpu_worker, [(i, 50, False, ref_dir) for i in range(cores)], chunksize=1)          # warm the workers (imports)
        res = pool.map(_cpu_worker, [(100 + i, n_steps, True, ref_dir) for i in range(cores)], chunksize=1)
    wall = max(r[0] for r in res)
    single = 1.0 / per_step
    what = ("the UNMODIFIED reference classes (ExtendedKalmanFilter.KalmanFilter / Wahba from " + ref_dir + ")") if ref_dir else \
        "the float64 numpy oracle port of the reference classes (reference tree not on this box)"
    return {"value": cores * n_steps / wall, "unit": UNIT, "cores": cores, "kind": "reference" if ref_dir else "port",
            "sample": f"{cores} independent synthetic 100 Hz trajectories x {n_steps} steps, Q=1 R=0.1, float64: {what}, driven as "
                      f"main_file.py:38-47, one process per core, started together; single-core rate {single:.0f} steps/s. "
                      f"A bounded SAMPLE of the GPU arm's workload (same per-step work, {cores * n_steps} of its filter-steps)",
            "single_core_value": single, "seconds": wall}


def cpu_baseline_compiled(n_filters: int = 16384, n_steps: int = 500):
    """The same path as an optimised CPU program would run it: oracle/ekf_oracle.c (float64, dense 4x4 algebra + Jacobi
    SVD as the reference's numpy calls do, gcc -O2), one pthread per host core.  Context beside `cpu_baseline`."""
    from oracle import c_oracle as CO
    from poseestimationkf_b200.synth import make_imu
    cores = len(os.sched_getaffinity(0)) or 1
    imu = make_imu(n_filters, n_steps, seed=5, sigma=0.01)
    S = imu.streams.numpy()
    ar, mr = imu.acc_ref.numpy(), imu.mag_ref.numpy()
    CO.replay(S[:50], 1e7, ar, mr, 1.0, 0.1, store=False, flips=False, threads=cores)
    t0 = time.perf_counter()
    CO.replay(S, 1e7, ar, mr, 1.0, 0.1, store=False, flips=False, threads=cores)
    wall = time.perf_counter() - t0
    return {"value": n_filters * n_steps / wall, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{n_filters} filters x {n_steps} steps, float64 C restatement (oracle/ekf_oracle.c), {cores} pthreads"}


def workload_text(name, world, filters, timesteps):
    if name == "c5":
        return (f"sharded long replay: {filters} independent filters x {timesteps} steps in total, filter-sharded over {world} GPU(s), "
                "time-chunked with carried state, inputs generated per chunk on the device, Q=1, R=0.1, dt=0.01 (BASELINE.json configs[4])")
    if name == "c3":
        return "Q/R tuning sweep: 64x64 (Q,R) grid x 256 trajectories x 5000 steps, loss surface on device (BASELINE.json configs[2])"
    if name == "c4":
        return "Wahba-only: 100 M (acc, mag) pairs -> quaternion (BASELINE.json configs[3])"
    return (f"batched EKF replay: {filters} independent filters x {timesteps} steps per GPU, Q=1, R=0.1, dt=0.01 "
            "(BASELINE.json configs[1])")


def resolve_workload(args, world):
    name = args.workload if args.workload != "auto" else ("c2" if world == 1 else "c5")
    if name == "c5":
        return name, args.filters or (1 << 24), args.timesteps or 2000
    return name, args.filters or (1 << 20), args.timesteps or 1000


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    name, filters, timesteps = resolve_workload(args, world)
    base = cpu_baseline(max(5.0, args.cpu_seconds))
    # K steps = K repetitions of the bounded sample; report the mean rate
    vals = [base["value"]]
    for _ in range(args.steps - 1):
        vals.append(cpu_baseline(max(5.0, args.cpu_seconds))["value"])
    v = sum(vals) / len(vals)
    base["value"] = v
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * base["seconds"], "higher_is_better": True,
            "scaling": "strong" if name == "c5" else "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_text(name, world, filters, timesteps) + "; reference arm = the reference's Python EKF on "
                                   "all host cores, each step a bounded sample of that workload (one independent trajectory per core)",
                       "filters": filters, "timesteps": timesteps, "sample": base["sample"], "same_config": False,
                       "same_config_note": "the CPU arm cannot finish the full workload (1e9+ filter-steps at ~1e5/s): it times a "
                                           "bounded sample with identical per-step work"},
            "cpu_baseline": base,
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi, during the timed region)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "20"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for t, r in self.rows if t0 <= t <= t1] or [r for _, r in self.rows[-3:]]
        sm = sorted(int(float(r[0])) for r in rows if r and r[0].replace(".", "").isdigit())
        reasons = []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            for name, val in zip(names, r[3:7]):
                if val.lower().startswith("active") and name not in reasons:
                    reasons.append(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None,
                "sm_max_mhz": int(float(rows[0][1])) if rows else None,
                "power_w_max": max((float(r[2]) for r in rows if r[2].replace(".", "").isdigit()), default=None),
                "samples": len(rows), "reasons": reasons}


def host_memory_available() -> int:
    """Bytes this process may still take: MemAvailable, capped by the container's cgroup limit minus its usage."""
    avail = 0
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable:"):
                avail = int(line.split()[1]) * 1024
    except Exception:
        pass
    for lim_f, use_f in (("/sys/fs/cgroup/memory.max", "/sys/fs/cgroup/memory.current"),
                         ("/sys/fs/cgroup/memory/memory.limit_in_bytes", "/sys/fs/cgroup/memory/memory.usage_in_bytes")):
        try:
            lim = open(lim_f).read().strip()
            if lim != "max" and int(lim) < (1 << 60):
                left = int(lim) - int(open(use_f).read().strip())
                avail = min(avail, left) if avail else left
        except Exception:
            pass
    return max(avail, 0)


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
class Ctx:
    """Process-wide plumbing of one rank."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        from poseestimationkf_b200 import sharding as SH
        self.torch, self.dist, self.SH = torch, dist, SH
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        # one process per GPU: keep this rank's pinned staging memory (e2e) on the socket its GPU hangs off
        self.all_cpus = os.sched_getaffinity(0)
        self.affinity = None if args.no_numa_bind else SH.bind_host_to_gpu(self.local)
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=self.dev)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, v: float) -> float:
        return self.SH.max_over_ranks(v, self.dev) if self.world > 1 else v

    def gather_floats(self, v: float) -> list:
        if self.world == 1:
            return [v]
        t = self.torch.tensor([v], dtype=self.torch.float64, device=self.dev)
        parts = [self.torch.empty_like(t) for _ in range(self.world)]
        self.dist.all_gather(parts, t)
        return [float(p.item()) for p in parts]

    def gather_objects(self, obj) -> list:
        if self.world == 1:
            return [obj]
        out = [None] * self.world
        self.dist.all_gather_object(out, obj)
        return out

    def finish(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def measure_e2e(ctx, args, streams, acc_ref, mag_ref, q, r, timesteps_total, note_prefix=""):
    """The same metric end to end through posekf_replay_host_f32: pinned host [Te,9,N] stream -> double-buffered H2D
    chunks -> kernel -> D2H of final X, P.  Also measures, in the same run and with every rank copying AT THE SAME TIME,
    the plain pinned H2D copy of the same buffer: the ceiling the host link offers this rank while its neighbours load
    theirs."""
    torch = ctx.torch
    from poseestimationkf_b200 import batched as B
    N = streams.shape[2]
    want = args.e2e_timesteps or timesteps_total
    # pinned host memory: this rank's share of what is available, with head-room (a box that runs out of memory is a strike)
    budget = int(0.35 * host_memory_available() / max(ctx.world, 1))
    Te = max(1, min(want, streams.shape[0], budget // (36 * N))) if budget > 0 else min(want, streams.shape[0], 250)
    host = torch.empty((Te, 9, N), dtype=torch.float32, pin_memory=True)
    host.copy_(streams[:Te])
    ar_h, mr_h = acc_ref.cpu().pin_memory(), mag_ref.cpu().pin_memory()
    q_h, r_h = q.cpu().pin_memory(), r.cpu().pin_memory()
    # host-link ceiling, synchronised across ranks: barrier, then every rank copies its whole buffer (twice; second timed)
    scratch = torch.empty((min(Te, 64), 9, N), dtype=torch.float32, device=ctx.dev)
    csz = scratch.shape[0]

    def plain_copy():
        for t0 in range(0, Te, csz):
            n = min(csz, Te - t0)
            scratch[:n].copy_(host[t0:t0 + n], non_blocking=True)
        torch.cuda.synchronize()

    plain_copy()
    ctx.barrier()
    tl0 = time.perf_counter()
    plain_copy()
    link_s = time.perf_counter() - tl0
    ctx.barrier()
    link_gbs = host.numel() * 4 / link_s / 1e9
    del scratch
    ws = B.HostWorkspace(N, device=ctx.local)
    # result buffers pinned once (a fresh 58 MB pinned allocation per call costs ~10 ms of page pinning)
    x_h = torch.empty((4, N), dtype=torch.float32, pin_memory=True)
    p_h = torch.empty((10, N), dtype=torch.float32, pin_memory=True)
    kw = dict(dt=0.01, q=q_h, r=r_h, wahba=args.wahba, device=ctx.local, workspace=ws, precise_state=args.precise_state,
              out_x=x_h, out_p=p_h)
    B.replay_host(host, ar_h, mr_h, **kw)   # warm-up
    ctx.barrier()
    reps_e = 3 if Te * N * 36 < (16 << 30) else 2
    t0 = time.perf_counter()
    for _ in range(reps_e):
        B.replay_host(host, ar_h, mr_h, **kw)
    own_s = (time.perf_counter() - t0) / reps_e
    ctx.barrier()
    dt_e = ctx.max_over_ranks(own_s)
    h2d = host.numel() * 4 + (ar_h.numel() + mr_h.numel() + q_h.numel() + r_h.numel()) * 4
    d2h = (x_h.numel() + p_h.numel()) * 4
    per_rank = ctx.gather_objects({"rank": ctx.rank, "h2d_gbs": h2d / own_s / 1e9, "plain_copy_gbs_synchronised": link_gbs,
                                   "host_affinity": ctx.affinity})
    ceil_min = min(p["plain_copy_gbs_synchronised"] for p in per_rank)
    e2e = {"value": ctx.world * N * Te / dt_e, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
           "timesteps": Te, "timesteps_of_workload": timesteps_total, "filters_per_gpu": N, "seconds_per_pass": dt_e,
           "note": note_prefix + "posekf_replay_host_f32: pinned host [T,9,N] stream -> double-buffered H2D chunks -> kernel -> "
                   "D2H of final X,P; bound by the host link (36 B per filter-step)",
           "h2d_gbs": h2d / dt_e / 1e9,
           "host_link_plain_copy_gbs": ceil_min,
           "host_link_note": "plain pinned H2D copy of the same buffer, all ranks copying at the same time (barrier before); "
                             "min over ranks -- the ceiling for the slowest rank, which sets the max-over-ranks time",
           "frac_of_plain_copy_ceiling": (h2d / dt_e / 1e9) / ceil_min,
           "box_aggregate_plain_copy_gbs": sum(p["plain_copy_gbs_synchronised"] for p in per_rank),
           "per_rank": per_rank}
    if Te < want:
        e2e["timesteps_note"] = (f"{Te} of the {want} timesteps: pinned host memory is bounded to 35 % of MemAvailable / ranks "
                                 f"({budget / 2**30:.0f} GiB per rank here)")
    del host
    ws.close()
    return e2e


def build_roofline(ctx, args, steps_per_s_kernel, avg_kernel_ms, fp32_peak, clocks, n_steps_per_launch, packed):
    torch = ctx.torch
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    hbm_src = "MEASURED_PEAKS.json (driver-measured copy bandwidth)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    flops, lane_ops, arith_src = executed_arithmetic(args.wahba)
    flops += FLOPS_COMPENSATED_EXTRA if args.precise_state else 0
    ach_tf = steps_per_s_kernel * flops / 1e12
    ach_gbs = steps_per_s_kernel * BYTES_PER_STEP / 1e9
    # the binding roof is the slower of FP32 issue and HBM streaming (north_star); report both
    t_fp32 = flops / (fp32_peak * 1e12)
    t_hbm = BYTES_PER_STEP / (hbm_peak * 1e9)
    bound = "fp32" if t_fp32 >= t_hbm else "hbm"
    sms = torch.cuda.get_device_properties(ctx.dev).multi_processor_count
    sm_mhz = (clocks or {}).get("sm_mhz")
    roofline = {
        "bound": bound,
        "achieved": ach_tf if bound == "fp32" else ach_gbs,
        "peak": fp32_peak if bound == "fp32" else hbm_peak,
        "unit": "TFLOP/s" if bound == "fp32" else "GB/s",
        "frac": (ach_tf / fp32_peak) if bound == "fp32" else (ach_gbs / hbm_peak),
        "traffic": None,
        "kernel": ("replay_tma2_kernel (packed f32x2, two filters per thread)" if packed
                   else f"replay_{'tma' if args.staging != 'ldg' else 'ldg'}_kernel<{args.wahba}>"),
        "kernel_ms": avg_kernel_ms,
        "algorithmic_flops_per_filter_step": flops,
        "algorithmic_bytes_per_filter_step": BYTES_PER_STEP,
        "arithmetic_source": arith_src,
        "fp32": {"achieved_tflops": ach_tf, "peak_tflops": fp32_peak, "frac": ach_tf / fp32_peak,
                 "peak_source": "FFMA probe kernel measured in this run (posekf_fp32_peak_tflops)"},
        "hbm": {"achieved_gbs": ach_gbs, "peak_gbs": hbm_peak, "frac": ach_gbs / hbm_peak, "peak_source": hbm_src},
        "roofline_steps_per_s_per_gpu": 1.0 / max(t_fp32, t_hbm),
        # what actually binds the kernel (DESIGN.md section 5, profiles/microbench/r02_pipes.*): the register file delivers one
        # 64-bit operand per lane per cycle, so a packed instruction costs max(2, operands read) cycles whatever its pipe
        "fp32_pipe_lane_cycles_frac": (steps_per_s_kernel * lane_ops / (sms * 128 * sm_mhz * 1e6)
                                       if lane_ops and not args.precise_state and sm_mhz else None),
        "frac_of_roofline": steps_per_s_kernel * max(t_fp32, t_hbm),
    }
    # ncu traffic: dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture of this kernel, per filter-step,
    # scaled to this launch -- quoted only when the capture was taken from the SAME device sources (stamped hash)
    if packed and not args.precise_state:
        try:
            prof = json.load(open(NCU_FULL))
            per_step = prof["dram_bytes_per_launch"] / prof["workload"]["filter_steps"]
            if prof.get("kernel_source_sha") == kernel_source_sha():
                roofline["traffic"] = per_step * n_steps_per_launch
                roofline["traffic_source"] = (f"{os.path.relpath(NCU_FULL, ROOT)}: {per_step:.2f} B per filter-step measured vs "
                                              f"{BYTES_PER_STEP} algorithmic (same device sources: {prof['kernel_source_sha']})")
            else:
                roofline["traffic_source"] = (f"{os.path.relpath(NCU_FULL, ROOT)} was captured from other device sources "
                                              f"({prof.get('kernel_source_sha')} vs {kernel_source_sha()}): not quoted, re-profile")
        except Exception as exc:
            roofline["traffic_source"] = f"no ncu capture available ({type(exc).__name__})"
    return roofline


def run_c2(ctx, args):
    torch = ctx.torch
    from poseestimationkf_b200 import batched as B
    from poseestimationkf_b200 import workloads as WL
    _, N, T = resolve_workload(args, 1)
    K, W = args.steps, max(args.warmup, 3)
    w = WL.build_c2(N, T, ctx.dev, seed=1000 + ctx.rank)
    streams, acc_ref, mag_ref, q, r = w.streams, w.acc_ref, w.mag_ref, w.q, w.r
    torch.cuda.synchronize()

    def one_pass(state):      # ONE kernel launch: the state was created for this very r tensor, so nothing is rescaled
        B.replay(streams, acc_ref, mag_ref, dt=0.01, q=q, r=r, state=state, wahba=args.wahba, staging=args.staging,
                 precise_state=args.precise_state)

    fp32_peak, _ = B.fp32_peak_tflops(ctx.local)
    torch.cuda.profiler.start()        # ncu --profile-from-start off: list warm-up + timed launches only
    for _ in range(W):
        one_pass(B.ReplayState.initial(N, ctx.dev, r=r))
    ctx.barrier()

    # --- timed region: exactly K passes; per-launch CUDA events on the launching stream ---------
    sampler = ClockSampler(ctx.local)
    if ctx.rank == 0:
        sampler.start()
        time.sleep(0.2)
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    fresh = [B.ReplayState.initial(N, ctx.dev, r=r) for _ in range(K)]
    ctx.barrier()
    t_wall0 = time.perf_counter()
    e_all0, e_all1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e_all0.record()
    for k in range(K):
        evs[k][0].record()
        one_pass(fresh[k])
        evs[k][1].record()
    e_all1.record()
    ctx.barrier()
    t_wall1 = time.perf_counter()
    torch.cuda.profiler.stop()
    total_ms = ctx.max_over_ranks(e_all0.elapsed_time(e_all1))
    kernel_ms = [a.elapsed_time(b) for a, b in evs]
    clocks = sampler.stop(t_wall0, t_wall1) if ctx.rank == 0 else None
    if ctx.rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, state_arrays(fresh[-1]))
    del fresh

    ms_per_step = total_ms / K
    value = ctx.world * N * T / (ms_per_step * 1e-3)
    avg_kernel_ms = sum(kernel_ms) / len(kernel_ms)
    steps_per_s_kernel = N * T / (avg_kernel_ms * 1e-3)

    # --- context: the other kernels on the first 250 timesteps of the same resident workload (not the headline) ----
    variants = {}
    if ctx.rank == 0 and not args.no_variants:
        Tv = min(250, T)
        sub = streams[:Tv]
        traj_buf = torch.empty((Tv, N, 4), dtype=torch.float32, device=ctx.dev)

        def rate(**kw):
            best = 1e30
            for i in range(3):
                st = B.ReplayState.initial(N, ctx.dev, r=r)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                B.replay(sub, acc_ref, mag_ref, dt=0.01, q=q, r=r, state=st, **kw)
                e1.record()
                torch.cuda.synchronize()
                if i:
                    best = min(best, e0.elapsed_time(e1))
            return N * Tv / (best * 1e-3)

        variants = {
            "packed_tma (default)": rate(precise_state=False, staging="tma_packed"),
            "scalar_tma": rate(precise_state=False, staging="tma"),
            "scalar_ldg": rate(precise_state=False, staging="ldg"),
            "packed_tma + precise variant (sweeps)": rate(precise_state=True, staging="tma_packed"),
            "packed_tma + trajectory stored [T,N,4]": rate(precise_state=False, staging="tma_packed", out_traj=traj_buf),
            "scalar_tma, Jacobi SVD Wahba (north_star literal)": rate(precise_state=False, staging="tma", wahba="jacobi"),
        }
        del traj_buf
        variants = {k: round(v / 1e9, 2) for k, v in variants.items()}

    e2e = None if args.no_e2e else measure_e2e(ctx, args, streams, acc_ref, mag_ref, q, r, T)
    if ctx.rank != 0:
        return None
    packed = args.staging in ("auto", "tma_packed") and args.wahba == "qr2" and N % 4 == 0
    roofline = build_roofline(ctx, args, steps_per_s_kernel, avg_kernel_ms, fp32_peak, clocks, N * T, packed)
    # every pass's own device time: a drift across the K passes is the power / thermal state of the box, not the kernel
    roofline["kernel_ms_per_pass"] = [round(v, 3) for v in kernel_ms]
    roofline["best_pass_steps_per_s"] = N * T / (min(kernel_ms) * 1e-3)
    return {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": ctx.world, "steps": K, "warmup": W,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_text("c2", ctx.world, N, T),
                   "filters_per_gpu": N, "timesteps": T, "wahba": args.wahba, "staging": args.staging,
                   "store_trajectory": False, "state": "two-float compensated" if args.precise_state else "float32",
                   "parallelism": f"filter-sharded x{ctx.world}, no collective",
                   "l2_policy": f"input stream is {N * T * 36 / 1e9:.1f} GB per pass (>> 126 MB L2), streamed once"},
        "roofline": roofline,
        "e2e": e2e,
        "gpu_launches": K,            # one replay kernel per pass, nothing else inside the timed region
        "clocks": clocks,
        "variants_gsteps_per_s_1gpu_250_timesteps": variants,
    }


def run_c5(ctx, args):
    """BASELINE.json configs[4]: 16 Mi filters x 2000 steps sharded over the ranks (strong scaling in the filter axis),
    time chunks generated on the device (untimed) with the state carried in the kernel's frame; `value` counts the
    filter kernels only (CUDA events, summed per rank, MAX over ranks); the final gather is timed apart."""
    torch = ctx.torch
    from poseestimationkf_b200 import batched as B
    from poseestimationkf_b200 import workloads as WL
    _, N_total, T = resolve_workload(args, ctx.world)
    K, W = args.steps, max(args.warmup, 3)
    job = WL.ShardedLongReplay(ctx.dev, ctx.rank, ctx.world, n_filters=N_total, n_steps=T)
    fp32_peak, _ = B.fp32_peak_tflops(ctx.local)
    # warm-up: W short passes over the first chunk (same kernels, same shapes) + one untimed full pass
    view = job.fill_chunk(0, min(job.chunk_steps, T))
    for _ in range(W):
        B.replay(view, job.acc_ref, job.mag_ref, dt=job.dt, q=job.q, r=job.r, state=job.new_state(), precise_state=False)
    ctx.barrier()
    sampler = ClockSampler(ctx.local)
    if ctx.rank == 0:
        sampler.start()
        time.sleep(0.2)
    ctx.barrier()
    t_wall0 = time.perf_counter()
    per_pass = []
    state = None
    for _ in range(K):
        state = job.new_state()
        ctx.barrier()
        per_pass.append(ctx.max_over_ranks(job.run_pass(state)))
    ctx.barrier()
    t_wall1 = time.perf_counter()
    clocks = sampler.stop(t_wall0, t_wall1) if ctx.rank == 0 else None
    if ctx.rank == 0 and args.dump_outputs:         # rank 0's shard
        dump_outputs(args.dump_outputs, state_arrays(state))
    ms_per_step = sum(per_pass) / K
    value = N_total * T / (ms_per_step * 1e-3)
    own_rate = job.n_local * T / (ms_per_step * 1e-3)

    # --- epilogue, timed apart: gather of the final states [4, N] (and [10, N] covariances) over NCCL ---------------
    gather = {"gather_ms": None}
    if ctx.world > 1:
        SH = ctx.SH
        SH.gather_states(state.x, N_total)          # warm-up (NCCL channel set-up, allocator) for both shapes
        SH.gather_states(state.p, N_total)
        ctx.barrier()
        g0, g1, g2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        g0.record()
        full_x = SH.gather_states(state.x, N_total)
        g1.record()
        full_p = SH.gather_states(state.p, N_total)
        g2.record()
        ctx.barrier()
        gather = {"gather_ms": ctx.max_over_ranks(g0.elapsed_time(g1)),
                  "gather_bytes_per_rank": int(full_x.numel() * 4),
                  "gather_covariance_ms": ctx.max_over_ranks(g1.elapsed_time(g2)),
                  "gather_note": "all_gather of the final states [4, N] (every rank receives all of them), NCCL over NVLink; "
                                 "outside `value`"}
        ok = bool(torch.isfinite(full_x).all())
        del full_x, full_p
        gather["gathered_states_finite"] = ok
        # the sharded replay is the single-GPU replay, bit for bit (128 Ki filters x 40 steps, gathered the same way)
        gather["sharded_equals_single"] = WL.sharded_equals_single(ctx.dev, ctx.rank, ctx.world)
    # --- e2e on this rank's shard ---------------------------------------------------------------------------------------
    e2e = None
    if not args.no_e2e:
        Te = args.e2e_timesteps or max(1, min(T, (9 << 30) // (36 * job.n_local)))      # ~9 GiB of host stream per rank
        args_e = argparse.Namespace(**vars(args))
        args_e.e2e_timesteps = Te
        view = job.fill_chunk(0, min(job.chunk_steps, Te))
        e2e = measure_e2e(ctx, args_e, view[:Te] if Te <= view.shape[0] else view, job.acc_ref, job.mag_ref, job.q, job.r, T,
                          note_prefix=f"this rank's shard ({job.n_local} filters), first {min(Te, view.shape[0])} timesteps; ")
    if ctx.rank != 0:
        return None
    avg_kernel_ms = ms_per_step / job.launches_per_pass
    roofline = build_roofline(ctx, args, own_rate, avg_kernel_ms, fp32_peak, clocks, job.n_local * job.chunk_steps, True)
    roofline["kernel_ms_note"] = f"{job.launches_per_pass} launches of {job.chunk_steps} timesteps per pass; kernel_ms is their mean"
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": ctx.world, "steps": K, "warmup": W,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_text("c5", ctx.world, N_total, T), "filters_total": N_total,
                   "filters_per_gpu": job.n_local, "timesteps": T, "time_chunk_steps": job.chunk_steps,
                   "wahba": "qr2", "staging": "auto", "store_trajectory": False, "state": "float32",
                   "parallelism": f"filter-sharded x{ctx.world} (128-aligned contiguous shards), no collective on the path",
                   "timing": "sum of the filter kernels' CUDA-event times per rank, MAX over ranks; the per-chunk input "
                             "synthesis on the device is untimed (SURVEY.md section 8d); gather timed apart",
                   "l2_policy": f"each time chunk is {job.n_local * job.chunk_steps * 36 / 1e9:.1f} GB (>> 126 MB L2), streamed once"},
        "roofline": roofline,
        "e2e": e2e,
        "gpu_launches": K * job.launches_per_pass,
        "clocks": clocks,
    }
    line.update(gather)
    return line


def run_c3(ctx, args):
    torch = ctx.torch
    from poseestimationkf_b200 import batched as B
    from poseestimationkf_b200 import workloads as WL
    K, W = args.steps, max(args.warmup, 3)
    w = WL.build_c3(ctx.dev, rank=ctx.rank, world=ctx.world)
    fp32_peak, _ = B.fp32_peak_tflops(ctx.local)
    for _ in range(W):
        st = WL.run_c3(w)
    ctx.barrier()
    sampler = ClockSampler(ctx.local)
    if ctx.rank == 0:
        sampler.start()
        time.sleep(0.2)
    ctx.barrier()
    t0w = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        st = WL.run_c3(w)
    e1.record()
    ctx.barrier()
    t1w = time.perf_counter()
    clocks = sampler.stop(t0w, t1w) if ctx.rank == 0 else None
    if ctx.rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, state_arrays(st))
    ms_per_step = ctx.max_over_ranks(e0.elapsed_time(e1)) / K
    T, Ns = w.streams.shape[0], w.streams.shape[2]
    total_filters = 64 * 64 * Ns
    surf = WL.loss_surface(w, st)
    best = int(surf.argmin())
    if ctx.rank != 0:
        return None
    value = total_filters * T / (ms_per_step * 1e-3)
    flops, lane_ops, src = executed_arithmetic("qr2")
    return {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": ctx.world, "steps": K, "warmup": W, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_text("c3", ctx.world, total_filters, T), "filters": total_filters, "timesteps": T,
                       "distinct_streams": Ns, "precision": "automatic per cell (precise variant where r/q >= 100 or q/r >= 1e4)",
                       "measurements": "Wahba solution shared per (trajectory, step)",
                       "parallelism": f"grid rows sharded x{ctx.world}, trajectories replicated",
                       "l2_policy": "46 MB stream shared by all cells stays in the 126 MB L2: compute regime by construction",
                       "includes": "state initialisation, measurement stream, two replay launches, scatter of the cell groups"},
            "roofline": {"bound": "fp32", "achieved": value / ctx.world * flops / 1e12, "peak": fp32_peak, "unit": "TFLOP/s",
                         "frac": value / ctx.world * flops / 1e12 / fp32_peak, "traffic": None, "arithmetic_source": src,
                         "note": "flops of the plain variant per filter-step; the precise cells execute more"},
            "e2e": None, "gpu_launches": None, "clocks": clocks,
            "loss_surface_min_rank0": {"q": float(w.qs[best // 64]), "r": float(w.rs[best % 64]), "mean_sin2": float(surf.min())}}


def run_c4(ctx, args):
    torch = ctx.torch
    from poseestimationkf_b200 import workloads as WL
    K, W = args.steps, max(args.warmup, 3)
    w = WL.build_c4(ctx.dev)
    M = w.acc.shape[1]
    out = {}
    for weights in ("half", "reference"):
        for _ in range(W):
            WL.run_c4(w, args.wahba, weights)
        ctx.barrier()
        evs = []
        for _ in range(K):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); WL.run_c4(w, args.wahba, weights); e1.record()
            evs.append((e0, e1))
        ctx.barrier()
        ms = ctx.max_over_ranks(sum(a.elapsed_time(b) for a, b in evs) / K)
        out[weights] = ms
    if ctx.rank != 0:
        return None
    if args.dump_outputs:                           # the last timed step used the reference weights
        dump_outputs(args.dump_outputs, {"quat": w.out})
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    ms = out["half"]
    return {"metric": "wahba_solves_per_s", "value": ctx.world * M / (ms * 1e-3), "unit": "solves/s", "n_gpus": ctx.world, "steps": K,
            "warmup": W, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": workload_text("c4", ctx.world, M, 1), "pairs_per_gpu": M, "algo": args.wahba,
                       "weights": "(.5,.5) headline; reference weights (|a_z|, 1-|a_z|) beside it",
                       "l2_policy": "4 GB of inputs + outputs per pass (>> 126 MB L2), streamed once"},
            "roofline": {"bound": "hbm", "achieved": M * 40 / (ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                         "frac": M * 40 / (ms * 1e-3) / 1e9 / hbm_peak, "traffic": None,
                         "algorithmic_bytes_per_solve": 40},
            "reference_weights": {"ms_per_step": out["reference"], "solves_per_s": M / (out["reference"] * 1e-3)},
            "e2e": None, "gpu_launches": K, "clocks": None}


def run_ours(args):
    ctx = Ctx(args)
    name, _, _ = resolve_workload(args, ctx.world)
    line = {"c2": run_c2, "c3": run_c3, "c4": run_c4, "c5": run_c5}[name](ctx, args)
    if ctx.rank == 0:
        if not args.no_cpu_baseline and ctx.world >= 1 and name in ("c2", "c5", "c3"):
            os.sched_setaffinity(0, ctx.all_cpus)          # the CPU arm uses every host core again
            if ctx.world == 1:                             # rank 0 at N=1 only (contract)
                line["cpu_baseline"] = cpu_baseline(args.cpu_seconds)
                try:
                    line["cpu_baseline_compiled"] = cpu_baseline_compiled()
                except Exception as exc:      # the C checker is optional infrastructure
                    line["cpu_baseline_compiled"] = {"unavailable": str(exc)}
        print(json.dumps(line))
    ctx.finish()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
