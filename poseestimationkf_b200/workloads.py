"""Synthetic workloads of BASELINE.json configs 2-5: builders and runners shared by `bench.py` (timing) and the
`-m gpu` full-size tests (which add the parity check).  This module only builds inputs with `synth.make_imu`
(plumbing, never timed) and drives the batched API; it knows nothing about the test-side float64 checker.

  C2  1 Mi independent filters x 1000 steps on one GPU (the headline configuration)
  C3  Q/R tuning sweep: 64x64 log-spaced (Q,R) grid x 256 trajectories x 5000 steps, loss surface on the device
      (knobs of `Python Kalman Filter/main_file.py:21-22`)
  C4  Wahba-only: 100 M (acc, mag) pairs -> quaternion (`Python Kalman Filter/Wahba.py:49-50`; weights (.5,.5) of
      `main_file.py:40` and the filter's own (|a_z|, 1-|a_z|) of `ExtendedKalmanFilter.py:71`)
  C5  16 Mi filters x 2000 steps sharded over the ranks of one box, time-chunked with carried state; the inputs of each
      chunk are generated on the device (1.2 TB would not fit); final states gathered afterwards
"""
from __future__ import annotations

from dataclasses import dataclass

import torch

from . import batched as B
from . import sharding as SH
from .synth import make_imu

C5_FILTERS, C5_STEPS = 1 << 24, 2000
C3_GRID, C3_STREAMS, C3_STEPS = 64, 256, 5000
C4_PAIRS = 100_000_000


# ------------------------------------------------------------------------------------------------
# C2
# ------------------------------------------------------------------------------------------------
@dataclass
class ReplayWorkload:
    streams: torch.Tensor      # [T, 9, N]
    acc_ref: torch.Tensor      # [3, N]
    mag_ref: torch.Tensor
    q: torch.Tensor            # [N]
    r: torch.Tensor
    dt: float


def build_c2(n_filters: int, n_steps: int, device, seed: int = 1000, base_n: int = 1 << 14) -> ReplayWorkload:
    """[T,9,N] float32 resident in HBM (36 GB at 1 Mi x 1000): `base_n` distinct trajectories are generated (float64
    ground truth on the device), replicated along the filter axis, and every replica gets its own additive sensor
    noise, so that no two filters do the same arithmetic."""
    N, T = n_filters, n_steps
    base_n = min(N, base_n)
    imu = make_imu(base_n, T, seed=seed, sigma=0.0, device=device)
    reps = (N + base_n - 1) // base_n
    streams = torch.empty((T, 9, N), dtype=torch.float32, device=device)
    g = torch.Generator(device=device)
    g.manual_seed(7 + seed)
    for t0 in range(0, T, 50):
        blk = imu.streams[t0:t0 + 50].repeat(1, 1, reps)[:, :, :N]
        blk = blk + 0.01 * torch.randn(blk.shape, generator=g, device=device)
        for sl in (slice(3, 6), slice(6, 9)):
            blk[:, sl] = blk[:, sl] / torch.linalg.vector_norm(blk[:, sl], dim=1, keepdim=True)
        streams[t0:t0 + 50] = blk
        del blk
    acc_ref = imu.acc_ref.repeat(1, reps)[:, :N].contiguous()
    mag_ref = imu.mag_ref.repeat(1, reps)[:, :N].contiguous()
    q = torch.full((N,), 1.0, device=device)
    r = torch.full((N,), 0.1, device=device)
    return ReplayWorkload(streams, acc_ref, mag_ref, q, r, imu.dt)


# ------------------------------------------------------------------------------------------------
# C3
# ------------------------------------------------------------------------------------------------
@dataclass
class SweepWorkload:
    streams: torch.Tensor      # [T, 9, Ns]   shared by all cells (46 MB: L2 resident)
    acc_ref: torch.Tensor
    mag_ref: torch.Tensor
    truth: torch.Tensor | None  # [T, Ns, 4]   ground-truth attitude for the tuning objective (None: a recording)
    qs: torch.Tensor           # [G] grid values
    rs: torch.Tensor
    q: torch.Tensor            # [G*G*Ns] per-filter; cell g = iq*G + ir owns filters g*Ns .. (g+1)*Ns
    r: torch.Tensor
    dt: float | torch.Tensor   # seconds, [T] per-step (a recording) or [T, Ns] per stream (a batch of recordings)
    lengths: torch.Tensor | None = None     # [Ns] int32 steps of each stream (a batch of recordings), None: all T

    @property
    def n_filters(self) -> int:
        return self.q.numel()

    def cell(self, iq: int, ir: int) -> slice:
        g = iq * self.qs.numel() + ir
        ns = self.streams.shape[2]
        return slice(g * ns, (g + 1) * ns)


def build_c3(device, grid: int = C3_GRID, n_streams: int = C3_STREAMS, n_steps: int = C3_STEPS, seed: int = 3,
             lo: float = -3.0, step: float = 0.1, rank: int = 0, world: int = 1) -> SweepWorkload:
    """The (Q,R) grid is log-spaced from 1e-3 in steps of 0.1 decade on both axes (64 values: 1e-3 .. 2e3), so that it
    holds the reference's own tuning Q = 1 (index 30), R = 0.1 (index 20) (`main_file.py:21-22`); with `world` > 1 the
    ROWS of the grid (Q values) are dealt out to the ranks and the 46 MB of trajectories are replicated (SURVEY.md
    section 8e)."""
    hi = lo + step * (grid - 1)
    imu = make_imu(n_streams, n_steps, seed=seed, sigma=0.01, device=device, keep_truth=True)
    qs_all = torch.logspace(lo, hi, grid, device=device)
    rs = torch.logspace(lo, hi, grid, device=device)
    b, e = SH.shard_bounds(grid, rank, world, align=1)
    qs = qs_all[b:e].contiguous()
    q = qs.repeat_interleave(grid).repeat_interleave(n_streams).contiguous()
    r = rs.repeat(qs.numel()).repeat_interleave(n_streams).contiguous()
    truth = imu.q_true.permute(0, 2, 1).to(torch.float32).contiguous()
    w = SweepWorkload(imu.streams, imu.acc_ref, imu.mag_ref, truth, qs, rs, q, r, imu.dt)
    return w


def run_c3(w: SweepWorkload, *, precise_state=None, share_measurements=None, objective: str = "truth",
           staging: str = "auto", gate: float | None = None) -> B.ReplayState:
    """One sweep: every cell replays all trajectories; returns the state with its tuning objective: `.loss` [N] (sum
    over steps of sin^2 of the angle to the ground truth; objective "truth"), `.innov` [2,N] (innovation likelihood
    sums, see `innovation_surface`; objective "innovation" for the 4-D model, "innovation_tangent" for the tangent-space
    one) or neither ("none").  `gate`: replay with the innovation gate at that NIS3 threshold (`B.replay(gate=...)`;
    the per-filter counts of gated steps are in `.gate_count`)."""
    innov_model = {"innovation": "full", "innovation_tangent": "tangent"}.get(objective)
    if innov_model is None and objective not in ("truth", "none"):
        raise ValueError("objective is 'truth', 'innovation', 'innovation_tangent' or 'none'")
    N = w.n_filters
    st = B.ReplayState.initial(N, w.streams.device, r=w.r)
    B.replay(w.streams, w.acc_ref, w.mag_ref, dt=w.dt, q=w.q, r=w.r, n_filters=N, state=st,
             truth=w.truth if objective == "truth" else None, innovation=True if innov_model else None,
             innovation_model=innov_model or "full", precise_state=precise_state, share_measurements=share_measurements,
             staging=staging, lengths=w.lengths, gate=gate)
    return st


def loss_surface(w: SweepWorkload, st: B.ReplayState) -> torch.Tensor:
    """[Gq, Gr] mean sin^2 per cell."""
    T, _, Ns = w.streams.shape
    return st.loss.reshape(w.qs.numel(), w.rs.numel(), Ns).mean(2) / T


def innovation_surface(w: SweepWorkload, st: B.ReplayState):
    """([Gq, Gr] mean innovation NLL per step, [Gq, Gr] mean NIS) per cell, float64: the tuning objective that needs no
    ground truth (`B.innovation_nll`, in the model of the state's sums); the best (Q,R) is the argmin of the first."""
    T, _, Ns = w.streams.shape
    nll, nis = B.innovation_nll(st, T)
    shape = (w.qs.numel(), w.rs.numel(), Ns)
    return nll.reshape(shape).mean(2) / T, nis.reshape(shape).mean(2)


def build_recording_sweep(log, device, grid: int = C3_GRID, lo: float = -3.0, step: float = 0.1) -> SweepWorkload:
    """A (Q,R) grid over ONE recorded log (`logio.LogData`): the cell layout of `build_c3` (log-spaced from 1e-3 in
    steps of 0.1 decade on both axes) with Ns = 1 stream and the log's own per-step dt.  There is no ground truth:
    run it with `run_c3(w, objective="innovation_tangent")` (or "innovation") and read `innovation_surface`; pass
    `lo` = -7 or so to reach the R that the tangent objective picks on low-noise sensors."""
    streams, acc_ref, mag_ref, dt = log.to_streams(device)
    hi = lo + step * (grid - 1)
    qs = torch.logspace(lo, hi, grid, device=device)
    rs = torch.logspace(lo, hi, grid, device=device)
    q = qs.repeat_interleave(grid).contiguous()
    r = rs.repeat(grid).contiguous()
    return SweepWorkload(streams, acc_ref, mag_ref, None, qs, rs, q, r, dt)


def build_multi_recording_sweep(logs, device, grid: int = C3_GRID, lo: float = -7.0, step: float = 0.1) -> SweepWorkload:
    """A (Q,R) grid over a SET of recorded logs, all in one launch: the cell layout of `build_c3` with Ns = len(logs)
    streams (rounded up to a multiple of 4 with empty ones), each with its own dt and length (`logio.stack_logs`).  Run
    it with `run_c3(w, objective="innovation_tangent")` and read `pooled_innovation_surface`, whose argmin is the one
    (Q,R) that best explains every recording together."""
    from .logio import stack_logs
    return build_batch_sweep(stack_logs(logs, device), grid, lo, step)


def build_batch_sweep(b, grid: int = C3_GRID, lo: float = -7.0, step: float = 0.1) -> SweepWorkload:
    """`build_multi_recording_sweep` over a `logio.LogBatch` that is already on the device, such as the one
    `logio.align_recordings` makes from raw event recordings."""
    device = b.streams.device
    Ns = b.streams.shape[2]
    hi = lo + step * (grid - 1)
    qs = torch.logspace(lo, hi, grid, device=device)
    rs = torch.logspace(lo, hi, grid, device=device)
    q = qs.repeat_interleave(grid).repeat_interleave(Ns).contiguous()
    r = rs.repeat(grid).repeat_interleave(Ns).contiguous()
    return SweepWorkload(b.streams, b.acc_ref, b.mag_ref, None, qs, rs, q, r, b.dt, b.lengths)


def pooled_innovation_surface(w: SweepWorkload, st: B.ReplayState):
    """([Gq, Gr] pooled innovation NLL per step, [Gq, Gr] pooled mean NIS) per cell, float64: the joint likelihood of
    all recordings of the sweep under the cell's one (Q,R), sum_k NLL_k / sum_k L_k, and sum_k sum_t NIS / sum_k L_k
    (L_k: the length of recording k; streams of length 0 add nothing).  Its argmin is the pooled tuning."""
    T, _, Ns = w.streams.shape
    L = (w.lengths if w.lengths is not None else torch.full((Ns,), T, dtype=torch.int32, device=w.streams.device))
    L = L.to(torch.float64)
    n_steps = L.repeat(st.x.shape[1] // Ns)
    nll, _ = B.innovation_nll(st, n_steps)
    shape = (w.qs.numel(), w.rs.numel(), Ns)
    total = L.sum()
    return nll.reshape(shape).sum(2) / total, st.innov[0].to(torch.float64).reshape(shape).sum(2) / total


# ------------------------------------------------------------------------------------------------
# C4
# ------------------------------------------------------------------------------------------------
@dataclass
class WahbaWorkload:
    acc: torch.Tensor          # [3, M] unit vectors
    mag: torch.Tensor
    acc_ref: torch.Tensor      # [3] shared reference pair
    mag_ref: torch.Tensor
    out: torch.Tensor          # [4, M]


def build_c4(device, n_pairs: int = C4_PAIRS, seed: int = 1) -> WahbaWorkload:
    g = torch.Generator(device=device)
    g.manual_seed(seed)

    def unit(v):
        return v / torch.linalg.vector_norm(v, dim=0, keepdim=True)

    acc = unit(torch.randn((3, n_pairs), generator=g, device=device))
    mag = unit(torch.randn((3, n_pairs), generator=g, device=device))
    ra = torch.tensor([0.0, 0.0, 1.0], device=device)
    rm = unit(torch.tensor([[0.4], [0.0], [-0.9165]], device=device))[:, 0].contiguous()
    return WahbaWorkload(acc, mag, ra, rm, torch.empty((4, n_pairs), device=device))


def run_c4(w: WahbaWorkload, algo: str = "qr2", weights: str = "half") -> torch.Tensor:
    """`weights`: "half" = (.5,.5) (`main_file.py:40`), "reference" = (|a_z|, 1-|a_z|) (`ExtendedKalmanFilter.py:71`)."""
    from . import _lib
    M = w.acc.shape[1]
    ref = weights == "reference"
    with torch.cuda.device(w.acc.device):
        rc = _lib.load().posekf_wahba_f32(M, w.acc_ref.data_ptr(), w.mag_ref.data_ptr(), 1, w.acc.data_ptr(), w.mag.data_ptr(),
                                          None, None, 0.0 if ref else 0.5, 0.0 if ref else 0.5, int(ref), None,
                                          w.out.data_ptr(), _lib.WAHBA[algo], 0, torch.cuda.current_stream().cuda_stream)
    _lib.check(rc, "posekf_wahba_f32")
    return w.out


# ------------------------------------------------------------------------------------------------
# C5
# ------------------------------------------------------------------------------------------------
class ShardedLongReplay:
    """This rank's shard of `n_filters` filters x `n_steps` steps, replayed in time chunks with carried state.

    The synthetic box-wide batch is `base_n` distinct trajectories tiled along the filter axis (global filter n follows
    trajectory n % base_n), so every rank can generate exactly its own columns of any time window on its own device and
    a sharded replay can be compared with a single-GPU one.  `chunk_bytes` bounds the device buffer of one window."""

    def __init__(self, device, rank: int = 0, world: int = 1, n_filters: int = C5_FILTERS, n_steps: int = C5_STEPS,
                 base_n: int = 1 << 14, seed: int = 8, chunk_bytes: int = 32 << 30, sigma: float = 0.01):
        self.device, self.rank, self.world = device, rank, world
        self.N, self.T = n_filters, n_steps
        self.begin, self.end = SH.shard_bounds(n_filters, rank, world)
        self.n_local = self.end - self.begin
        self.base_n = min(base_n, n_filters)
        self.base = make_imu(self.base_n, n_steps, seed=seed, sigma=sigma, device=device)    # same seed on every rank
        self.dt = self.base.dt
        self.chunk_steps = max(1, min(250, SH.chunk_steps_for_budget(max(self.n_local, 1), chunk_bytes)))
        self.buf = torch.empty((self.chunk_steps, 9, self.n_local), dtype=torch.float32, device=device)
        self.acc_ref = self._tile(self.base.acc_ref)
        self.mag_ref = self._tile(self.base.mag_ref)
        self.q = torch.full((self.n_local,), 1.0, device=device)
        self.r = torch.full((self.n_local,), 0.1, device=device)

    def _tile(self, a: torch.Tensor) -> torch.Tensor:
        """Columns [begin, end) of `a` tiled along its last axis with period base_n."""
        off = self.begin % self.base_n
        reps = (off + self.n_local + self.base_n - 1) // self.base_n
        return a.repeat(*([1] * (a.dim() - 1)), reps)[..., off:off + self.n_local].contiguous()

    def fill_chunk(self, t0: int, t1: int) -> torch.Tensor:
        """Device-side input generation for the window [t0, t1) of this shard (untimed)."""
        off = self.begin % self.base_n
        reps = (off + self.n_local + self.base_n - 1) // self.base_n
        view = self.buf[: t1 - t0]
        if off == 0 and self.n_local % self.base_n == 0:      # whole periods: one broadcast copy
            view.view(t1 - t0, 9, reps, self.base_n).copy_(self.base.streams[t0:t1].unsqueeze(2).expand(-1, -1, reps, -1))
            return view
        for k in range(reps):       # copy period by period: no [tc, 9, reps*base_n] temporary
            lo = max(k * self.base_n, off) - off
            hi = min((k + 1) * self.base_n, off + self.n_local) - off
            if hi > lo:
                src0 = lo + off - k * self.base_n
                view[:, :, lo:hi] = self.base.streams[t0:t1, :, src0:src0 + (hi - lo)]
        return view

    def new_state(self) -> B.ReplayState:
        return B.ReplayState.initial(self.n_local, self.device, r=self.r)

    def run_pass(self, state: B.ReplayState) -> float:
        """All time chunks once; returns the summed device time of the filter kernels (ms, CUDA events on the
        launching stream).  The state stays in the kernel's working frame between chunks."""
        events = []
        for t0, t1 in SH.time_chunks(self.T, self.chunk_steps):
            view = self.fill_chunk(t0, t1)          # same stream: ordered after the kernel that read the buffer last
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            B.replay(view, self.acc_ref, self.mag_ref, dt=self.dt, q=self.q, r=self.r, state=state, precise_state=False,
                     keep_filter_frame=t1 < self.T)
            e1.record()
            events.append((e0, e1))
        torch.cuda.synchronize(self.device)
        return sum(a.elapsed_time(b) for a, b in events)

    @property
    def launches_per_pass(self) -> int:
        return (self.T + self.chunk_steps - 1) // self.chunk_steps


def sharded_equals_single(device, rank: int, world: int, n_filters: int = 128 * 1024, n_steps: int = 40) -> bool:
    """Every rank replays its shard of a small batch, the states are gathered (the same `gather_states` epilogue as
    the full run), and rank 0 compares them bit for bit with its own single-GPU replay of the whole batch.  Returns
    the verdict on rank 0 (True elsewhere)."""
    imu = make_imu(n_filters, n_steps, seed=123, sigma=0.01, device=device)
    b, e = SH.shard_bounds(n_filters, rank, world)
    st, _, _ = B.replay(imu.streams[:, :, b:e].contiguous(), imu.acc_ref[:, b:e].contiguous(), imu.mag_ref[:, b:e].contiguous(),
                        dt=imu.dt, q=1.0, r=0.1)
    full_x = SH.gather_states(st.x, n_filters)
    full_p = SH.gather_states(st.p, n_filters)
    if rank != 0:
        return True
    ref, _, _ = B.replay(imu.streams, imu.acc_ref, imu.mag_ref, dt=imu.dt, q=1.0, r=0.1)
    return bool(torch.equal(full_x, ref.x) and torch.equal(full_p, ref.p))
