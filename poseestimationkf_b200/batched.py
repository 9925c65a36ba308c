"""Batched (N independent filters) API over torch CUDA tensors.

This is the host-side mirror of the reference's interface for the replay path: the same
operations as `KalmanFilter.Prediction/Correction`, `Wahba.getRotation/getQuarternion`,
`RungeKutta4`, ... (`Python Kalman Filter/ExtendedKalmanFilter.py`, `Wahba.py`,
`UtilityFunctions.py`), for a batch, plus the fused `replay` that runs the loop of
`Python Kalman Filter/main_file.py:38-47` on the device.  torch is used for device memory and
streams only; all arithmetic happens in libposekf_b200.so (include/posekf.h).

Layout: batched arrays are component-major `[k, N]` float32 CUDA tensors (filter index fastest);
IMU streams are `[T, 9, N]` (gyro xyz, acc xyz, mag xyz); stored trajectories are `[T, N, 4]`.  Helpers convert from/to the reference's
per-filter `[N, k]` / `[N, 4, 4]` shapes.
"""
from __future__ import annotations

import math
import weakref
from dataclasses import dataclass

import torch

from . import _lib

_TRI = [(0, 0), (0, 1), (0, 2), (0, 3), (1, 1), (1, 2), (1, 3), (2, 2), (2, 3), (3, 3)]


# ------------------------------------------------------------------------------------------------
# helpers
# ------------------------------------------------------------------------------------------------
def _require_cuda(*tensors):
    for t in tensors:
        if t is None:
            continue
        if not isinstance(t, torch.Tensor) or not t.is_cuda:
            raise _lib.PosekfError("poseestimationkf_b200 runs on CUDA tensors only (no CPU fallback)")
        if t.dtype != torch.float32 and t.dtype != torch.uint8:
            raise TypeError(f"expected float32 tensors, got {t.dtype}")
        if not t.is_contiguous():
            raise ValueError("tensors passed to the batched API must be contiguous")


def _ptr(t):
    return None if t is None else t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def tri_from_full(P: torch.Tensor) -> torch.Tensor:
    """[N,4,4] covariance -> packed upper triangle [10,N] (order 00 01 02 03 11 12 13 22 23 33)."""
    return torch.stack([P[:, i, j] for i, j in _TRI]).contiguous()


def full_from_tri(p: torch.Tensor) -> torch.Tensor:
    """[10,N] -> symmetric [N,4,4]."""
    N = p.shape[1]
    P = torch.empty((N, 4, 4), dtype=p.dtype, device=p.device)
    for k, (i, j) in enumerate(_TRI):
        P[:, i, j] = p[k]
        P[:, j, i] = p[k]
    return P


def soa(a: torch.Tensor) -> torch.Tensor:
    """per-filter rows [N,k] (or [N,r,c]) -> component-major [k,N] (or [r*c,N])."""
    return a.reshape(a.shape[0], -1).t().contiguous()


def aos(a: torch.Tensor, *shape) -> torch.Tensor:
    """component-major [k,N] -> per-filter [N,k] (optionally reshaped to [N,*shape])."""
    out = a.t().contiguous()
    return out.reshape(out.shape[0], *shape) if shape else out


# ------------------------------------------------------------------------------------------------
# fused replay
# ------------------------------------------------------------------------------------------------
@dataclass
class ReplayState:
    """Filter state carried between `replay` calls (time-chunked replay, checkpoint/resume).
    x [4,N]; p [10,N] packed upper triangle of P/r (the covariance in units of each filter's r --
    the form the kernel works in, so that chunked and unchunked replays are bit-identical);
    r: the float or [N] tensor the scaling refers to -- 1.0 after a replay with general Q / R matrices, whose kernels
    carry P itself (`replay` converts p whenever the next call needs the other form); lpf [6,N] or None.
    frame: "reference" (x, p in the reference's own coordinates -- what every `replay` call returns by
    default) or "filter" (left in the kernel's working frame by `replay(..., keep_filter_frame=True)`
    between the chunks of a time-chunked replay; `to_reference_frame` converts).
    innov [2,N]: the innovation likelihood sums (sum_t NIS_t, sum_t ln det S_t) of `replay(..., innovation=...)`;
    innov_model: the model they belong to ("full" or "tangent", see `replay(..., innovation_model=...)`).
    gate_count [N] int32: the number of steps the innovation gate rejected (see `replay(..., gate=...)`)."""
    x: torch.Tensor
    p: torch.Tensor
    r: object = 0.1
    lpf: torch.Tensor | None = None
    loss: torch.Tensor | None = None     # [N] accumulated tuning objective (see replay(truth=...))
    x_lo: torch.Tensor | None = None     # [4,N] low-order part of the compensated (two-float) state
    frame: str = "reference"
    innov: torch.Tensor | None = None    # [2,N] innovation likelihood sums (see replay(innovation=...))
    innov_model: str | None = None       # "full" / "tangent": the model of `innov`
    gate_count: torch.Tensor | None = None   # [N] int32 gated steps (see replay(gate=...))

    @staticmethod
    def initial(n_filters: int, device, r=0.1, with_lpf: bool = False, P0: torch.Tensor | None = None) -> "ReplayState":
        """X=[1,0,0,0], P=I4 (Python Kalman Filter/main_file.py:23,26) unless P0 [N,4,4] is given;
        low-pass state 0 (Kalman Filter Server/PoseEstimator/KalmanFilter.cpp:16-18)."""
        x = torch.zeros((4, n_filters), dtype=torch.float32, device=device)
        x[0] = 1.0
        if P0 is None:
            p = torch.zeros((10, n_filters), dtype=torch.float32, device=device)
            p[[0, 4, 7, 9]] = 1.0
        else:
            p = tri_from_full(P0.to(device=device, dtype=torch.float32))
        p = p / (r if isinstance(r, torch.Tensor) else float(r))
        lpf = torch.zeros((6, n_filters), dtype=torch.float32, device=device) if with_lpf else None
        return ReplayState(x, p.contiguous(), r, lpf)

    def covariance(self) -> torch.Tensor:
        """P [N,4,4] (unscaled)."""
        return full_from_tri(self.p * (self.r if isinstance(self.r, torch.Tensor) else float(self.r)))

    def clone(self) -> "ReplayState":
        c = lambda t: None if t is None else t.clone()
        return ReplayState(self.x.clone(), self.p.clone(), self.r, c(self.lpf), c(self.loss), c(self.x_lo), self.frame,
                           c(self.innov), self.innov_model, c(self.gate_count))

    def to_reference_frame(self, acc_ref: torch.Tensor, mag_ref: torch.Tensor) -> "ReplayState":
        """Convert (in place) a state that `replay(..., keep_filter_frame=True)` left in the kernel's working
        frame back to the reference's coordinates.  acc_ref, mag_ref [3,Ns] as given to `replay`."""
        if self.frame == "filter":
            _convert_frame(self, acc_ref, mag_ref, FILTER_FRAME_IN)
            self.frame = "reference"
        return self


FILTER_FRAME_IN, FILTER_FRAME_OUT = 1, 2      # POSEKF_STATE_IN_FILTER_FRAME / POSEKF_STATE_OUT_FILTER_FRAME


def _convert_frame(state: "ReplayState", acc_ref, mag_ref, flags: int) -> None:
    """A zero-step launch that only moves the state between the reference and the filter frame."""
    _require_cuda(state.x, state.p, state.x_lo, acc_ref, mag_ref)
    N, Ns, dev = state.x.shape[1], acc_ref.shape[1], state.x.device
    ones = torch.ones((N,), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        rc = _lib.load().posekf_replay_f32(N, 0, None, Ns, None, 0, _ptr(acc_ref), _ptr(mag_ref), _ptr(ones), _ptr(ones),
                                           -1.0, -1.0, _ptr(state.x), _ptr(state.x_lo), _ptr(state.p), None, None, None, None,
                                           None, _lib.WAHBA["qr2"], _lib.STAGING["ldg"], int(flags), _stream())
    _lib.check(rc, "posekf_replay_f32 (frame conversion)")


_scalar_cache: dict = {}


def _scalar_tensor(value: float, device) -> torch.Tensor:
    """One-element float32 tensor holding `value` on `device`, cached so that repeated replay calls
    launch nothing but the filter kernel."""
    key = (float(value), str(device))
    t = _scalar_cache.get(key)
    if t is None:
        if len(_scalar_cache) > 64:
            _scalar_cache.clear()
        t = torch.full((1,), float(value), dtype=torch.float32, device=device)
        _scalar_cache[key] = t
    return t


def _same_scale(a, b) -> bool:
    if isinstance(a, torch.Tensor) or isinstance(b, torch.Tensor):
        if isinstance(a, torch.Tensor) and isinstance(b, torch.Tensor):
            return a is b or (a.shape == b.shape and bool(torch.equal(a, b)))
        return False
    return float(a) == float(b)


_checked_scales: dict = {}


def _scales_need_precise(q, r) -> bool:
    """One pass over the (Q,R) values: validates them (r > 0, q >= 0: R = rI must be positive definite because the
    kernels carry P/r) and answers whether any filter sits where the plain float32 step leaves the 1e-5 rad tolerance
    (r/q >= 100: gains below half an ulp of the state; q/r >= 1e4: the process noise swamps A K A^T).  For tensors the
    answer costs one reduction and one host read-back, cached per (q, r) tensor pair and version so that the chunks of
    a time-chunked replay (same tensor objects) pay for it once."""
    if not isinstance(q, torch.Tensor) and not isinstance(r, torch.Tensor):
        qf, rf = float(q), float(r)
        if not rf > 0.0 or not qf >= 0.0:
            raise ValueError("r must be > 0 and q >= 0 (the kernel carries the covariance in units of r)")
        return rf >= 100.0 * qf or qf >= 1.0e4 * rf
    # cache entry: weak references to the very tensor objects (an id alone can be recycled by a new tensor after the old
    # one is freed) and their version counters (bumped by any in-place write, also through views)
    key = tuple(id(t) if isinstance(t, torch.Tensor) else float(t) for t in (q, r))
    hit = _checked_scales.get(key)
    if hit is not None:
        refs, versions, flag = hit
        same = all((ref is None and not isinstance(t, torch.Tensor)) or (ref is not None and ref() is t and t._version == ver)
                   for t, ref, ver in zip((q, r), refs, versions))
        if same:
            return flag
    qt = q if isinstance(q, torch.Tensor) else torch.full((1,), float(q), dtype=torch.float32, device=r.device)
    rt = r if isinstance(r, torch.Tensor) else torch.full((1,), float(r), dtype=torch.float32, device=q.device)
    bad = ~(rt > 0) | ~(qt >= 0)
    need = (rt >= 100.0 * qt) | (qt >= 1.0e4 * rt)
    flags = torch.stack((bad.any(), need.any())).tolist()
    if flags[0]:
        raise ValueError("every r must be > 0 and every q >= 0 (the kernel carries the covariance in units of r)")
    if len(_checked_scales) > 64:
        _checked_scales.clear()
    refs = tuple(weakref.ref(t) if isinstance(t, torch.Tensor) else None for t in (q, r))
    versions = tuple(t._version if isinstance(t, torch.Tensor) else 0 for t in (q, r))
    _checked_scales[key] = (refs, versions, bool(flags[1]))
    return bool(flags[1])


_TRI3 = [(0, 0), (0, 1), (0, 2), (1, 1), (1, 2), (2, 2)]


def _is_matrix(v) -> bool:
    """A q / r argument that selects the general-matrix replay: a [k,k] or [N,k,k] tensor or array."""
    return hasattr(v, "shape") and len(v.shape) >= 2


def _as_matrices(v, k: int, n: int, device, name: str) -> torch.Tensor:
    """[1,k,k] or [n,k,k] float64 on `device` from a [k,k] / [n,k,k] matrix, or from a float / [n] tensor (v I_k)."""
    if isinstance(v, torch.Tensor) and not v.is_cuda and torch.device(device).type == "cuda":
        raise _lib.PosekfError("poseestimationkf_b200 runs on CUDA tensors only (no CPU fallback); matrices may be numpy "
                               "arrays or CUDA tensors of any float dtype")
    t = torch.as_tensor(v, dtype=torch.float64, device=device)
    eye = torch.eye(k, dtype=torch.float64, device=device)
    if t.dim() == 0:
        return (t * eye)[None]
    if t.dim() == 1 and t.shape == (n,):
        return t[:, None, None] * eye[None]
    if t.dim() == 2 and t.shape == (k, k):
        return t[None]
    if t.dim() == 3 and t.shape == (n, k, k):
        return t
    raise ValueError(f"{name} must be a float, an [N] tensor, a [{k},{k}] or an [N,{k},{k}] matrix (N = {n}), "
                     f"got shape {tuple(t.shape)}")


_general_cache: dict = {}


def general_qr_tri(q, r, n: int, device):
    """The matrices of a general-matrix replay (include/posekf.h, posekf_replay_general_f32) as the kernels read them:
    (q_tri [6,Nq], r_tri [10,Nr]) float32 upper triangles, Nq / Nr = 1 for one matrix shared by the launch, else n.
    q: [3,3] / [N,3,3] (Q), or a float / [N] tensor (q I3); r: [4,4] / [N,4,4] (R), or a float / [N] tensor (r I4).
    Checks, on the float32 values the kernels use: symmetry (to 1e-6 of the largest entry), R positive definite and Q
    positive semidefinite (torch.linalg.eigvalsh; an eigenvalue down to -1e-6 of the largest counts as 0).  One
    read-back, cached per tensor pair and version (pass the SAME tensor objects to every chunk of a chunked replay)."""
    key = tuple(id(t) if isinstance(t, torch.Tensor) else None for t in (q, r))
    hit = _general_cache.get(key) if all(k is not None for k in key) else None
    if hit is not None:
        refs, versions, dev, n0, out = hit
        if all(ref() is t and t._version == ver for t, ref, ver in zip((q, r), refs, versions)) and dev == str(device) and n0 == n:
            return out
    Q = _as_matrices(q, 3, n, device, "q").to(torch.float32).to(torch.float64)
    R = _as_matrices(r, 4, n, device, "r").to(torch.float32).to(torch.float64)
    bad = []
    for M, name in ((Q, "Q"), (R, "R")):
        asym = (M - M.transpose(1, 2)).abs().amax() > 1e-6 * M.abs().amax()
        lam = torch.linalg.eigvalsh(torch.triu(M) + torch.triu(M, 1).transpose(1, 2))
        low = lam.amin() <= 0 if name == "R" else lam.amin() < -1e-6 * lam.amax().clamp(min=0)
        bad += [asym, low | ~torch.isfinite(lam).all()]
    asym_q, neg_q, asym_r, neg_r = torch.stack(bad).tolist()
    if asym_q or asym_r:
        raise ValueError("Q and R must be symmetric")
    if neg_r:
        raise ValueError("R must be positive definite")
    if neg_q:
        raise ValueError("Q must be positive semidefinite")
    out = (torch.stack([Q[:, i, j] for i, j in _TRI3]).to(torch.float32).contiguous(),
           torch.stack([R[:, i, j] for i, j in _TRI]).to(torch.float32).contiguous())
    if all(k is not None for k in key):
        if len(_general_cache) > 64:
            _general_cache.clear()
        _general_cache[key] = (tuple(weakref.ref(t) for t in (q, r)), tuple(t._version for t in (q, r)), str(device), n, out)
    return out


def _per_filter(v, n, device):
    if isinstance(v, torch.Tensor):
        _require_cuda(v)
        if v.shape != (n,):
            raise ValueError(f"per-filter scalar must have shape ({n},), got {tuple(v.shape)}")
        return v
    return torch.full((n,), float(v), dtype=torch.float32, device=device)


def measurement_stream(streams, acc_ref, mag_ref, *, lpf_alpha_acc=None, lpf_alpha_mag=None, lpf_state=None,
                       algo: str = "qr2", out=None):
    """Solve the Wahba problem of every (stream, step) once: streams [T,9,Ns] -> a measurement stream of the
    same shape (rows 0-2 gyro, rows 3-6 the reference-signed Wahba quaternion, rows 7-8 zero) to be replayed
    with `wahba="precomputed"`.  The optional low-pass is applied here (state [6,Ns] carried across chunks).
    Returns (measurement stream, lpf_state)."""
    _require_cuda(streams, acc_ref, mag_ref, lpf_state, out)
    T, _, Ns = streams.shape
    use_lpf = lpf_alpha_acc is not None or lpf_alpha_mag is not None
    if use_lpf and lpf_state is None:
        lpf_state = torch.zeros((6, Ns), dtype=torch.float32, device=streams.device)
    if out is None:
        out = torch.empty_like(streams)
    with torch.cuda.device(streams.device):
        rc = _lib.load().posekf_measurement_stream_f32(
            Ns, T, _ptr(streams), _ptr(acc_ref), _ptr(mag_ref), -1.0 if lpf_alpha_acc is None else float(lpf_alpha_acc),
            -1.0 if lpf_alpha_mag is None else float(lpf_alpha_mag), _ptr(lpf_state), _ptr(out), _lib.WAHBA[algo], _stream())
    _lib.check(rc, "posekf_measurement_stream_f32")
    return out, lpf_state


def replay(streams: torch.Tensor, acc_ref: torch.Tensor, mag_ref: torch.Tensor, *, dt, q=1.0, r=0.1,
           state: ReplayState | None = None, n_filters: int | None = None, lpf_alpha_acc: float | None = None,
           lpf_alpha_mag: float | None = None, out_traj: torch.Tensor | None = None, store_trajectory: bool = False,
           store_flips: bool = False, truth: torch.Tensor | None = None, loss: torch.Tensor | None = None,
           precise_state: bool | None = None, share_measurements: bool | None = None, wahba: str = "qr2",
           staging: str = "auto", keep_filter_frame: bool = False, allow_imprecise: bool = False,
           innovation: bool | torch.Tensor | None = None, innovation_model: str = "full",
           lengths: torch.Tensor | None = None, gate: float | None = None, gate_count: torch.Tensor | None = None,
           out_gated: torch.Tensor | None = None, out_innovation: torch.Tensor | None = None):
    """Run T Prediction+Correction steps for N filters in one kernel launch.

    streams [T,9,Ns]; acc_ref, mag_ref [3,Ns]; dt: float seconds, [T] float32 CUDA tensor (one clock for every
    filter) or [T,Ns] (per stream: filter n steps with column n % Ns -- a batch of recordings, `logio.stack_logs`);
    q, r: floats or [N] tensors (Q=q*I3, R=r*I4), or general matrices: q [3,3] / [N,3,3] and r [4,4] / [N,4,4] (numpy
    arrays or CUDA tensors; either may stay a float or [N] tensor).  A matrix runs the general-matrix replay
    (include/posekf.h, posekf_replay_general_f32): the reference's KalmanFilter with its Q and R attributes assigned,
    symmetric Q positive semidefinite and R positive definite (checked, `general_qr_tri`).  It has no precise variant;
    its innovation sums, per-step innovation output and gate are `replay_general`'s.  Trajectories, flips, the loss,
    the low-pass, every Wahba mode, per-stream dt and lengths work as with scalars, and `state.p` then holds P itself
    (`state.r` = 1.0).  `n_filters` > Ns replays every trajectory
    N/Ns times (filter n reads column n % Ns) -- the Q/R sweep layout.  `state` is updated in place
    (created with the reference's initial values when None).  `truth` [T,Ns,4] enables the on-device
    tuning objective: `loss` [N] (created zeroed when None; pass it back in for chunked replays) is
    incremented by sum_t 1-(X_t.truth_t)^2 and is available as `state.loss`.
    `precise_state` selects the precise variant for extreme Q/R ratios (two-float state so that gains
    ~1e-7 are not lost when R >> Q; Sherman-Morrison gain when Q >> R; +25 % time); None = automatic:
    on when r/q >= 100 or q/r >= 1e4, off otherwise (the default Q=1, R=0.1 does not need it).  With per-filter
    q / r tensors the rule is applied per cell of a sweep (blocks of Ns filters that share one tuning; two
    launches over a permutation of the cells) when no per-step output is requested, and to the whole batch
    (precise when ANY filter needs it, decided from the values with one cached reduction) otherwise.
    `precise_state=False` with such a tuning raises unless `allow_imprecise=True` (the plain step is then 1.4e-5 to
    3e-5 rad off the float64 reference after 5000 steps, outside the 1e-5 rad tolerance).
    q, r: pass the SAME tensor objects to every chunk of a time-chunked replay (their validation and the precision
    rule are cached per tensor; `state.r is r` also skips the rescaling check).
    `share_measurements`: in the sweep layout (N > Ns) the Wahba solution of a sample is the same for every
    filter that shares its trajectory, so it is solved once per (trajectory, step) (`measurement_stream`) and
    the replay runs with `wahba="precomputed"`; None = automatic for N >= 4 Ns without a low-pass stage.
    `keep_filter_frame`: leave `state` in the kernel's working frame (the coordinates of the frame built from
    acc_ref / mag_ref, in which the Wahba stage is cheapest) instead of converting it back at the end of the
    launch.  Pass it on every chunk but the last of a time-chunked replay: the chunked replay is then
    bit-identical to the unchunked one.  `state.frame` records where the state is; a state left in the filter
    frame is accepted by the next `replay` call and converted by `state.to_reference_frame(acc_ref, mag_ref)`.
    `innovation`: accumulate the innovation likelihood of every filter on the device -- the (Q,R) tuning objective that
    needs no ground truth (include/posekf.h, posekf_replay_innovation_f32).  True creates a zeroed [2,N] accumulator
    (sum_t NIS_t, sum_t ln det S_t); a tensor is used as is (pass `state.innov` back in for chunked replays).  It is
    available as `state.innov`; `innovation_nll` turns it into per-filter NLL and mean NIS.  It does not perturb the
    filter.  None / False: the launch is exactly that of a replay without it.
    `innovation_model`: "full" (the 4-D model of the reference's S and e) or "tangent" (the same model in the 3-D
    tangent space of the prediction, posekf_replay_innovation_ex_f32, whose R axis has an interior minimum).  Recorded
    as `state.innov_model`; an accumulator that holds the sums of the other model is refused.
    `lengths`: [Ns] int32 CUDA tensor, the number of steps of THIS call that stream c has (0..T; checked with one
    read-back).  A filter whose stream has ended is held: its state, loss and innovation sums stay as they are, its
    trajectory rows repeat its final state and its flip bytes are 0; the samples and dt of those steps are never used
    (they may be NaN).  For a time-chunked replay pass each chunk its own lengths (`logio.LogBatch.window`).
    A [T,Ns] dt or `lengths` runs the batched kernels (include/posekf.h, posekf_replay_batch_f32).
    `gate`: innovation gating (include/posekf.h, posekf_replay_gated_f32) -- a step whose tangent-space normalised
    innovation squared NIS3 exceeds `gate` is not corrected: the filter keeps its prediction and its propagated
    covariance (an outlier measurement, e.g. a magnetic disturbance, is rejected).  NIS3 ~ chi^2_3 under a consistent
    model: `GATE_CHI2_3_999` = 16.27 rejects one step in a thousand of a consistent filter.  float('inf') gives the
    bits of the ungated replay.  The flip mask, the loss, the low-pass and the innovation sums still see every step.
    `gate_count`: [N] int32 CUDA tensor incremented by each filter's number of gated steps (created zeroed when None;
    pass `state.gate_count` back in for chunked replays); available as `state.gate_count`.  `out_gated`: a [T,N]
    uint8 CUDA tensor that receives 1 where a step was gated (0 elsewhere and on held steps).  Both need `gate`.
    `out_innovation`: a [2,T,N] float32 CUDA tensor that receives the innovation terms of every step
    (include/posekf.h, posekf_replay_innovation_steps_f32): [0] NIS_t, [1] ln det S_t of `innovation_model`, in the
    convention of the sums (`workloads.window_innovation_nll` scores windows of it).  Held steps get 0, gated steps
    their terms.  It needs neither `innovation` nor `gate` and changes no other output.  Its rows must be contiguous
    (stride N along t, 1 along n); the plane stride may be larger, so a time-chunked replay passes each chunk the view
    `out_innovation[:, t0:t1]` of one full-length buffer.  With general Q / R matrices see `replay_general`; the
    precision rule is the whole-batch one.
    Returns (state, traj [T,N,4] or None, flips [T,N] uint8 or None)."""
    return _replay(streams, acc_ref, mag_ref, dt=dt, q=q, r=r, state=state, n_filters=n_filters, lpf_alpha_acc=lpf_alpha_acc,
                   lpf_alpha_mag=lpf_alpha_mag, out_traj=out_traj, store_trajectory=store_trajectory, store_flips=store_flips,
                   truth=truth, loss=loss, precise_state=precise_state, share_measurements=share_measurements, wahba=wahba,
                   staging=staging, keep_filter_frame=keep_filter_frame, allow_imprecise=allow_imprecise,
                   innovation=innovation, innovation_model=innovation_model, lengths=lengths, gate=gate,
                   gate_count=gate_count, out_gated=out_gated, out_innovation=out_innovation, general_innovation=False)


def replay_general(streams: torch.Tensor, acc_ref: torch.Tensor, mag_ref: torch.Tensor, *, dt, q, r,
                   state: ReplayState | None = None, n_filters: int | None = None, lpf_alpha_acc: float | None = None,
                   lpf_alpha_mag: float | None = None, out_traj: torch.Tensor | None = None,
                   store_trajectory: bool = False, store_flips: bool = False, truth: torch.Tensor | None = None,
                   loss: torch.Tensor | None = None, precise_state: bool | None = None,
                   share_measurements: bool | None = None, wahba: str = "qr2", staging: str = "auto",
                   keep_filter_frame: bool = False, allow_imprecise: bool = False,
                   innovation: bool | torch.Tensor | None = None, innovation_model: str = "full",
                   lengths: torch.Tensor | None = None, gate: float | None = None, gate_count: torch.Tensor | None = None,
                   out_gated: torch.Tensor | None = None, out_innovation: torch.Tensor | None = None):
    """The general-matrix replay of `replay` (q [3,3] / [N,3,3] and/or r [4,4] / [N,4,4]; the other may stay a float or
    [N] tensor) with the innovation likelihood, its per-step terms and the innovation gate (include/posekf.h,
    posekf_replay_general_innovation_f32).  Every keyword means what it means in `replay`; `state.p` holds P itself.
    `innovation` / `innovation_model`: the sums of the 4-D ("full") or tangent-space model, NIS_t = e^T S^-1 e and
    ln det S_t with S = P^- + R in true units (`innovation_nll` and `state.innov` as for scalars).  `out_innovation`
    [2,T,N]: the per-step terms (`workloads.window_innovation_nll` reads them).  `gate`: a live step whose tangent-space
    NIS3 exceeds `gate` keeps its prediction and P^-; `gate_count`, `out_gated` and `state.gate_count` as in `replay`.
    Without any of these the launch is exactly `replay`'s with the same matrices, and with them every other output
    keeps those bits (ungated, or `gate=inf` without gate buffers).  There is no precise variant.  Scalar q and r are
    refused: that is `replay`.  Returns (state, traj [T,N,4] or None, flips [T,N] uint8 or None)."""
    if not (_is_matrix(q) or _is_matrix(r)):
        raise ValueError("replay_general takes a [3,3] / [N,3,3] q or a [4,4] / [N,4,4] r; for Q = qI3 and R = rI4 use "
                         "replay")
    return _replay(streams, acc_ref, mag_ref, dt=dt, q=q, r=r, state=state, n_filters=n_filters, lpf_alpha_acc=lpf_alpha_acc,
                   lpf_alpha_mag=lpf_alpha_mag, out_traj=out_traj, store_trajectory=store_trajectory, store_flips=store_flips,
                   truth=truth, loss=loss, precise_state=precise_state, share_measurements=share_measurements, wahba=wahba,
                   staging=staging, keep_filter_frame=keep_filter_frame, allow_imprecise=allow_imprecise,
                   innovation=innovation, innovation_model=innovation_model, lengths=lengths, gate=gate,
                   gate_count=gate_count, out_gated=out_gated, out_innovation=out_innovation, general_innovation=True)


def _replay(streams, acc_ref, mag_ref, *, dt, q, r, state, n_filters, lpf_alpha_acc, lpf_alpha_mag, out_traj,
            store_trajectory, store_flips, truth, loss, precise_state, share_measurements, wahba, staging,
            keep_filter_frame, allow_imprecise, innovation, innovation_model, lengths, gate, gate_count, out_gated,
            out_innovation, general_innovation: bool):
    """The body of `replay` and `replay_general`.  general_innovation: matrices may come with the innovation sums, the
    per-step terms and the gate (posekf_replay_general_innovation_f32)."""
    if innovation_model not in _lib.INNOV_MODEL:
        raise ValueError("innovation_model is 'full' or 'tangent'")
    if gate is None and (gate_count is not None or out_gated is not None):
        raise ValueError("gate_count / out_gated need gate=<threshold>")
    if gate is not None and math.isnan(float(gate)):
        raise ValueError("gate must be a number (NaN decides nothing)")
    _require_cuda(streams, acc_ref, mag_ref, out_traj)
    if streams.dim() != 3 or streams.shape[1] != 9:
        raise ValueError("streams must be [T, 9, Ns]")
    T, _, Ns = streams.shape
    N = Ns if n_filters is None else int(n_filters)
    if acc_ref.shape != (3, Ns) or mag_ref.shape != (3, Ns):
        raise ValueError("acc_ref / mag_ref must be [3, Ns]")
    dev = streams.device
    use_lpf = lpf_alpha_acc is not None or lpf_alpha_mag is not None
    dt_cols = None
    if isinstance(dt, torch.Tensor) and dt.dim() == 2:
        _require_cuda(dt)
        if dt.shape != (T, Ns):
            raise ValueError(f"a per-stream dt tensor must be [T, Ns] = [{T}, {Ns}]")
        dt_cols = dt
    if lengths is not None:
        _check_lengths(lengths, Ns, T)
    if share_measurements is None:
        share_measurements = N > Ns and N >= 4 * Ns and wahba == "qr2" and not use_lpf and T > 0
    if share_measurements:
        if wahba == "precomputed" or use_lpf or N == Ns:
            raise ValueError("share_measurements needs raw streams, N > Ns and no low-pass stage")
        streams, _ = measurement_stream(streams, acc_ref, mag_ref, algo=wahba)
        wahba = "precomputed"
    general = _is_matrix(q) or _is_matrix(r)
    if general:
        if not general_innovation and ((innovation is not None and innovation is not False) or gate is not None
                                       or out_innovation is not None):
            raise ValueError("general Q / R matrices: the innovation sums, the per-step innovation output and the gate "
                             "are replay_general's (same keywords)")
        if precise_state or (state is not None and state.x_lo is not None):
            raise ValueError("general Q / R matrices: the replay has no precise variant (precise_state, a two-float state)")
        q_tri, r_tri = general_qr_tri(q, r, N, dev)
        needs_precise, units = False, 1.0        # the general kernels carry P itself
    else:
        if isinstance(q, torch.Tensor):
            _require_cuda(q)
        if isinstance(r, torch.Tensor):
            _require_cuda(r)
        needs_precise = _scales_need_precise(q, r)      # also validates r > 0, q >= 0
        units = r
    if state is None:
        state = ReplayState.initial(N, dev, r=units, with_lpf=use_lpf)
    elif not _same_scale(state.r, units):
        # the covariance is stored in units of the r it was created with: re-express it in units of the new r
        old = state.r if isinstance(state.r, torch.Tensor) else float(state.r)
        new = units if isinstance(units, torch.Tensor) else float(units)
        state.p.mul_(old / new)
    state.r = units
    if precise_state is None:
        if not general and (isinstance(q, torch.Tensor) or isinstance(r, torch.Tensor)) and N > Ns and N % Ns == 0 \
                and out_traj is None and not store_trajectory and not store_flips and not use_lpf and T > 0 \
                and out_gated is None and out_innovation is None:
            # a (Q,R) sweep: only the cells with r/q >= 100 or q/r >= 1e4 need the precise variant (+25 % time)
            mixed = _replay_sweep_mixed(streams, acc_ref, mag_ref, dt=dt, q=q, r=r, state=state, N=N, Ns=Ns, truth=truth,
                                        loss=loss, wahba=wahba, staging=staging, keep_filter_frame=keep_filter_frame,
                                        innovation=innovation, innovation_model=innovation_model, lengths=lengths,
                                        gate=gate, gate_count=gate_count)
            if mixed is not None:
                return mixed
        precise_state = state.x_lo is not None or needs_precise
    elif not precise_state and needs_precise and not allow_imprecise:
        raise ValueError("precise_state=False with r/q >= 100 or q/r >= 1e4 leaves the 1e-5 rad tolerance of the float64 "
                         "reference (the plain float32 step absorbs gains ~1e-7); pass allow_imprecise=True to run it anyway")
    if precise_state and state.x_lo is None:
        state.x_lo = torch.zeros((4, N), dtype=torch.float32, device=dev)
    _require_cuda(state.x_lo)
    if use_lpf and state.lpf is None:
        state.lpf = torch.zeros((6, N), dtype=torch.float32, device=dev)
    _require_cuda(state.x, state.p, state.lpf)
    if state.x.shape != (4, N) or state.p.shape != (10, N):
        raise ValueError("state has the wrong shape for this batch")
    if dt_cols is not None:
        dt_t, per_step = None, 0
    elif isinstance(dt, torch.Tensor):
        _require_cuda(dt)
        if dt.shape != (T,):
            raise ValueError("dt tensor must be [T] or [T, Ns]")
        dt_t, per_step = dt, 1
    else:
        dt_t, per_step = _scalar_tensor(dt, dev), 0
    q_t, r_t = (None, None) if general else (_per_filter(q, N, dev), _per_filter(r, N, dev))
    if wahba == "precomputed":
        # no Wahba stage in the kernel: its working frame is the reference frame
        state.to_reference_frame(acc_ref, mag_ref)
        frame_flags = 0
    else:
        frame_flags = (FILTER_FRAME_IN if state.frame == "filter" else 0) | (FILTER_FRAME_OUT if keep_filter_frame else 0)
    if store_trajectory and out_traj is None:
        out_traj = torch.empty((T, N, 4), dtype=torch.float32, device=dev)
    if out_traj is not None and out_traj.shape != (T, N, 4):
        raise ValueError("out_traj must be [T, N, 4]")
    flips = torch.empty((T, N), dtype=torch.uint8, device=dev) if store_flips else None
    if truth is not None:
        _require_cuda(truth, loss)
        if truth.shape != (T, Ns, 4):
            raise ValueError("truth must be [T, Ns, 4]")
        if loss is None:
            loss = torch.zeros((N,), dtype=torch.float32, device=dev)
        state.loss = loss
    innov = _innovation_buffer(innovation, N, dev, state, innovation_model)
    if gate is not None:
        gate_count = _gate_buffers(gate_count, out_gated, N, T, dev)
    if out_innovation is not None:
        _check_innovation_steps(out_innovation, N, T)
    args = (N, T, _ptr(streams), Ns, _ptr(dt_t), per_step, _ptr(acc_ref), _ptr(mag_ref), _ptr(q_t), _ptr(r_t),
            -1.0 if lpf_alpha_acc is None else float(lpf_alpha_acc),
            -1.0 if lpf_alpha_mag is None else float(lpf_alpha_mag),
            _ptr(state.x), _ptr(state.x_lo if precise_state else None), _ptr(state.p), _ptr(state.lpf), _ptr(out_traj),
            _ptr(flips), _ptr(truth), _ptr(loss if truth is not None else None))
    tail = (_lib.WAHBA[wahba], _lib.STAGING[staging], frame_flags, _stream())
    batch = dt_cols is not None or lengths is not None
    with torch.cuda.device(dev):
        if general and general_innovation:
            rc = _lib.load().posekf_replay_general_innovation_f32(
                N, T, _ptr(streams), Ns, _ptr(dt_t), per_step, _ptr(acc_ref), _ptr(mag_ref), _ptr(q_tri), q_tri.shape[1],
                _ptr(r_tri), r_tri.shape[1], *args[10:], _ptr(innov), _lib.INNOV_MODEL[innovation_model], *tail,
                _ptr(dt_cols), _ptr(lengths), math.inf if gate is None else float(gate),
                _ptr(gate_count if gate is not None else None), _ptr(out_gated), _ptr(out_innovation),
                out_innovation.stride(0) if out_innovation is not None else 0)
        elif general:
            rc = _lib.load().posekf_replay_general_f32(
                N, T, _ptr(streams), Ns, _ptr(dt_t), per_step, _ptr(acc_ref), _ptr(mag_ref), _ptr(q_tri), q_tri.shape[1],
                _ptr(r_tri), r_tri.shape[1], *args[10:], None, _lib.INNOV_MODEL["full"], *tail, _ptr(dt_cols), _ptr(lengths))
        elif out_innovation is not None:
            rc = _lib.load().posekf_replay_innovation_steps_f32(
                *args, _ptr(innov), _lib.INNOV_MODEL[innovation_model], *tail, _ptr(dt_cols), _ptr(lengths),
                math.inf if gate is None else float(gate), _ptr(gate_count if gate is not None else None), _ptr(out_gated),
                _ptr(out_innovation), out_innovation.stride(0))
        elif gate is not None:
            rc = _lib.load().posekf_replay_gated_f32(*args, _ptr(innov), _lib.INNOV_MODEL[innovation_model], *tail, _ptr(dt_cols),
                                                     _ptr(lengths), float(gate), _ptr(gate_count), _ptr(out_gated))
        elif batch:
            rc = _lib.load().posekf_replay_batch_f32(*args, _ptr(innov), _lib.INNOV_MODEL[innovation_model], *tail, _ptr(dt_cols),
                                                     _ptr(lengths))
        elif innov is None:
            rc = _lib.load().posekf_replay_f32(*args, *tail)
        else:
            rc = _lib.load().posekf_replay_innovation_ex_f32(*args, _ptr(innov), _lib.INNOV_MODEL[innovation_model], *tail)
    _lib.check(rc, "posekf_replay_general_innovation_f32" if general and general_innovation else
               "posekf_replay_general_f32" if general else "posekf_replay_innovation_steps_f32" if out_innovation is not None
               else "posekf_replay_gated_f32" if gate is not None else
               "posekf_replay_batch_f32" if batch else
               ("posekf_replay_f32" if innov is None else "posekf_replay_innovation_ex_f32"))
    if innov is not None:
        state.innov, state.innov_model = innov, innovation_model
    if gate is not None:
        state.gate_count = gate_count
    if wahba != "precomputed":
        state.frame = "filter" if keep_filter_frame else "reference"
    return state, out_traj, flips


def _check_lengths(lengths, n_streams: int, n_steps: int) -> None:
    """replay(lengths=...): an [Ns] int32 CUDA tensor with every value in [0, T] (one reduction and one read-back)."""
    if not isinstance(lengths, torch.Tensor) or lengths.dtype != torch.int32 or not lengths.is_contiguous() \
            or lengths.shape != (n_streams,):
        raise ValueError(f"lengths must be a contiguous int32 tensor of shape ({n_streams},)")
    if n_streams:
        lo, hi = torch.stack((lengths.min(), lengths.max())).tolist()
        if lo < 0 or hi > n_steps:
            raise ValueError(f"lengths must lie in [0, {n_steps}] (the steps of this call), got [{lo}, {hi}]")
    if not lengths.is_cuda:
        raise _lib.PosekfError("poseestimationkf_b200 runs on CUDA tensors only (no CPU fallback)")


# the 0.999 quantile of chi^2 with 3 degrees of freedom: a gate threshold that rejects one step in a thousand of a
# consistent filter (replay(gate=...))
GATE_CHI2_3_999 = 16.266236196238129


def _gate_buffers(gate_count, out_gated, n: int, n_steps: int, device):
    """replay(gate=...): checks out_gated [T,N] uint8 and returns the [N] int32 gate_count (zeros when None)."""
    for t, shape, dtype, name in ((gate_count, (n,), torch.int32, "gate_count"), (out_gated, (n_steps, n), torch.uint8, "out_gated")):
        if t is None:
            continue
        if not isinstance(t, torch.Tensor) or t.dtype != dtype or tuple(t.shape) != shape or not t.is_contiguous():
            raise ValueError(f"{name} must be a contiguous {dtype} tensor of shape {shape}")
        if not t.is_cuda:
            raise _lib.PosekfError("poseestimationkf_b200 runs on CUDA tensors only (no CPU fallback)")
    if gate_count is None:
        gate_count = torch.zeros((n,), dtype=torch.int32, device=device)
    return gate_count


def _check_innovation_steps(out, n: int, n_steps: int) -> None:
    """replay(out_innovation=...): a [2,T,N] float32 CUDA tensor whose rows are contiguous (plane stride >= T N)."""
    if not isinstance(out, torch.Tensor) or out.dtype != torch.float32 or tuple(out.shape) != (2, n_steps, n):
        raise ValueError(f"out_innovation must be a float32 tensor of shape (2, {n_steps}, {n})")
    if n and n_steps and (out.stride(2) != 1 or (n_steps > 1 and out.stride(1) != n) or out.stride(0) < n_steps * n):
        raise ValueError("out_innovation must have contiguous [T, N] planes (strides (>= T N, N, 1)), e.g. a time slice "
                         "out[:, t0:t1] of a contiguous buffer")
    if not out.is_cuda:
        raise _lib.PosekfError("poseestimationkf_b200 runs on CUDA tensors only (no CPU fallback)")


def _innovation_buffer(innovation, n: int, device, state=None, model: str = "full"):
    """The [2,N] accumulator of replay(innovation=...): None when off, zeros for True, the caller's tensor otherwise.
    The state's own accumulator is refused when it holds the sums of another model."""
    if innovation is None or innovation is False:
        return None
    if innovation is True:
        return torch.zeros((2, n), dtype=torch.float32, device=device)
    if state is not None and innovation is state.innov and state.innov_model not in (None, model):
        raise ValueError(f"the accumulator holds sums of the {state.innov_model!r} innovation model, not {model!r}")
    _require_cuda(innovation)
    if innovation.shape != (2, n):
        raise ValueError(f"innovation accumulator must be [2, {n}]")
    return innovation


def innovation_nll(innov, n_steps, model: str | None = None):
    """Per-filter innovation likelihood from the [2,N] sums of `replay(..., innovation=...)` (or a ReplayState holding
    them) over `n_steps` steps (an int, or an [N] tensor of per-filter step counts -- a batch of recordings of different
    lengths; a filter with 0 steps has NLL 0 and mean NIS nan): (NLL [N], mean NIS [N]) in float64,
        NLL = 1/2 sum_t [NIS_t + ln det S_t] + (dof/2) T ln 2 pi,     mean NIS = sum_t NIS_t / T
    (natural log; P and R unscaled), dof = 4 for the "full" model and 3 for the "tangent" one.  A ReplayState supplies
    its own model (`model`, when given, must agree with it); for a bare tensor `model` defaults to "full".  A good (Q,R)
    minimises the NLL."""
    if model is not None and model not in _lib.INNOV_MODEL:
        raise ValueError("model is 'full' or 'tangent'")
    if isinstance(innov, ReplayState):
        own = innov.innov_model or "full"
        if model is not None and model != own:
            raise ValueError(f"the state holds sums of the {own!r} innovation model, not {model!r}")
        model, a = own, innov.innov
    else:
        a = innov
    if a is None:
        raise ValueError("no innovation sums: replay with innovation=True")
    dof = 3 if model == "tangent" else 4
    a = a.to(torch.float64)
    T = n_steps.to(device=a.device, dtype=torch.float64) if isinstance(n_steps, torch.Tensor) else float(n_steps)
    return 0.5 * (a[0] + a[1]) + 0.5 * dof * T * math.log(2.0 * math.pi), a[0] / T


def sweep_partition(q_t: torch.Tensor, r_t: torch.Tensor, n_streams: int):
    """Filter indices of a sweep split by the precision its cells need.  A cell is a block of `n_streams` consecutive
    filters (one per trajectory); it needs the precise variant when any of its filters has r/q >= 100 or q/r >= 1e4.
    Returns (plain, precise) index tensors; both keep whole cells in their original order, so filter k of either group
    still reads stream column k % n_streams."""
    n = q_t.numel()
    if n % n_streams:
        raise ValueError("a sweep has a whole number of cells")
    need = ((r_t >= 100.0 * q_t) | (q_t >= 1.0e4 * r_t)).view(n // n_streams, n_streams).any(dim=1)
    lane = torch.arange(n_streams, device=q_t.device)
    expand = lambda cells: (cells[:, None] * n_streams + lane[None, :]).flatten()
    return expand((~need).nonzero().flatten()), expand(need.nonzero().flatten())


def _replay_sweep_mixed(streams, acc_ref, mag_ref, *, dt, q, r, state, N, Ns, truth, loss, wahba, staging, keep_filter_frame,
                        innovation=None, innovation_model="full", lengths=None, gate=None, gate_count=None):
    """Sweep layout with automatic precision: the cells (blocks of Ns filters sharing one (q, r)) whose tuning is
    extreme run the precise variant, the others the plain one -- two launches over a cell permutation that keeps
    every filter on its own stream column (n % Ns).  Returns None when one launch serves all cells."""
    dev = streams.device
    q_t, r_t = _per_filter(q, N, dev), _per_filter(r, N, dev)
    idx_plain, idx_precise = sweep_partition(q_t, r_t, Ns)
    if idx_plain.numel() == 0 or idx_precise.numel() == 0:
        return None
    parts = []
    if truth is not None and loss is None:
        loss = torch.zeros((N,), dtype=torch.float32, device=dev)
    innov = _innovation_buffer(innovation, N, dev, state, innovation_model)
    if gate is not None:
        gate_count = _gate_buffers(gate_count, None, N, streams.shape[0], dev)
    for idx, precise in ((idx_plain, False), (idx_precise, True)):
        sub = ReplayState(state.x[:, idx].contiguous(), state.p[:, idx].contiguous(), r_t[idx].contiguous(), None, None,
                          state.x_lo[:, idx].contiguous() if (precise and state.x_lo is not None) else None, state.frame)
        sub_loss = loss[idx].contiguous() if truth is not None else None
        sub_innov = innov[:, idx].contiguous() if innov is not None else None
        sub_gc = gate_count[idx].contiguous() if gate is not None else None
        replay(streams, acc_ref, mag_ref, dt=dt, q=q_t[idx].contiguous(), r=sub.r, state=sub, n_filters=idx.numel(), truth=truth,
               loss=sub_loss, precise_state=precise, share_measurements=False, wahba=wahba, staging=staging,
               keep_filter_frame=keep_filter_frame, innovation=sub_innov, innovation_model=innovation_model,
               lengths=lengths, gate=gate, gate_count=sub_gc)   # (the plain group holds no extreme cell by construction)
        parts.append((idx, sub, sub_loss, sub_innov, precise, sub_gc))
    if state.x_lo is None:
        state.x_lo = torch.zeros((4, N), dtype=torch.float32, device=dev)
    for idx, sub, sub_loss, sub_innov, precise, sub_gc in parts:
        state.x[:, idx] = sub.x
        state.p[:, idx] = sub.p
        if precise:
            state.x_lo[:, idx] = sub.x_lo
        if truth is not None:
            loss[idx] = sub_loss
        if innov is not None:
            innov[:, idx] = sub_innov
        if gate is not None:
            gate_count[idx] = sub_gc
        state.frame = sub.frame
    if truth is not None:
        state.loss = loss
    if innov is not None:
        state.innov, state.innov_model = innov, innovation_model
    if gate is not None:
        state.gate_count = gate_count
    state.r = r
    return state, None, None


class HostWorkspace:
    """Reusable device staging buffers / streams of `replay_host` for batches of `n_filters`."""

    def __init__(self, n_filters: int, *, chunk_steps: int = 0, with_trajectory: bool = False, device: int = 0):
        import ctypes as C
        self.n_filters, self.with_trajectory, self.device = int(n_filters), bool(with_trajectory), int(device)
        h = C.c_void_p()
        _lib.check(_lib.load().posekf_host_workspace_create(self.device, self.n_filters, int(chunk_steps),
                                                            int(with_trajectory), C.byref(h)), "posekf_host_workspace_create")
        self.handle = h

    def close(self):
        if getattr(self, "handle", None):
            _lib.load().posekf_host_workspace_destroy(self.handle)
            self.handle = None

    __del__ = close


def replay_host(streams, acc_ref, mag_ref, *, dt: float, q, r, lpf_alpha_acc=None, lpf_alpha_mag=None,
                store_trajectory=False, chunk_steps: int = 0, wahba: str = "qr2", precise_state: bool = True,
                device: int = 0, workspace: "HostWorkspace | None" = None, out_x=None, out_p=None, out_traj=None):
    """End-to-end replay from HOST memory (CPU torch tensors, ideally pinned): the stream is pushed
    through the GPU in double-buffered time chunks and the final state (and optionally the
    trajectory) is copied back.  streams [T,9,N] float32 CPU; acc_ref/mag_ref [3,N]; q, r [N].
    `precise_state` (default on: per-filter q/r are given as arrays here, and the link, not the kernel,
    bounds this path) selects the precise variant for extreme Q/R ratios.
    `out_x` / `out_p` / `out_traj`: result buffers to fill (pinned CPU tensors of the shapes below); a caller
    that replays in a loop passes them to avoid pinning fresh pages on every call (a 58 MB pinned allocation
    costs ~10 ms, as much as 6 % of a 1 Mi x 250 replay).
    Returns (x [4,N], p [10,N], traj [T,N,4] or None) as CPU tensors."""
    for t in (streams, acc_ref, mag_ref, q, r):
        if t.is_cuda or t.dtype != torch.float32 or not t.is_contiguous():
            raise ValueError("replay_host takes contiguous float32 CPU tensors")
    T, _, N = streams.shape
    pin = streams.is_pinned()

    def _out(buf, shape):
        if buf is None:
            return torch.empty(shape, dtype=torch.float32, pin_memory=pin)
        if buf.is_cuda or buf.dtype != torch.float32 or not buf.is_contiguous() or tuple(buf.shape) != tuple(shape):
            raise ValueError(f"output buffer must be a contiguous float32 CPU tensor of shape {tuple(shape)}")
        return buf

    x = _out(out_x, (4, N))
    p = _out(out_p, (10, N))
    traj = _out(out_traj, (T, N, 4)) if (store_trajectory or out_traj is not None) else None
    rc = _lib.load().posekf_replay_host_f32(
        N, T, _ptr(streams), float(dt), _ptr(acc_ref), _ptr(mag_ref), _ptr(q), _ptr(r),
        -1.0 if lpf_alpha_acc is None else float(lpf_alpha_acc),
        -1.0 if lpf_alpha_mag is None else float(lpf_alpha_mag),
        None, None, _ptr(x), _ptr(p), _ptr(traj), int(chunk_steps), _lib.WAHBA[wahba], int(bool(precise_state)), int(device),
        None if workspace is None else workspace.handle)
    _lib.check(rc, "posekf_replay_host_f32")
    return x, p, traj


# ------------------------------------------------------------------------------------------------
# stand-alone operators (component-major in / out)
# ------------------------------------------------------------------------------------------------
def wahba(acc_ref, mag_ref, acc, mag, *, k_acc=None, k_mag=None, weights_from_acc=False, want_rotation=False,
          want_quaternion=True, algo: str = "qr2", jacobi_sweeps: int = 0):
    """Wahba.getRotation / getQuarternion for N pairs.  acc, mag [3,N]; acc_ref, mag_ref [3,N] or
    [3] (shared); k_acc/k_mag: floats, [N] tensors, or None with weights_from_acc=True for the
    reference's |acc_z| / 1-|acc_z|.  Returns (R [9,N] or None, q [4,N] or None)."""
    _require_cuda(acc_ref, mag_ref, acc, mag)
    N = acc.shape[1]
    shared = int(acc_ref.dim() == 1)
    dev = acc.device
    ka_t = km_t = None
    ka_s = km_s = 0.0
    if isinstance(k_acc, torch.Tensor):
        _require_cuda(k_acc, k_mag)
        ka_t, km_t = k_acc, k_mag
    elif not weights_from_acc:
        if k_acc is None or k_mag is None:
            raise ValueError("give k_acc/k_mag or weights_from_acc=True")
        ka_s, km_s = float(k_acc), float(k_mag)
    R = torch.empty((9, N), dtype=torch.float32, device=dev) if want_rotation else None
    qt = torch.empty((4, N), dtype=torch.float32, device=dev) if want_quaternion else None
    with torch.cuda.device(dev):
        rc = _lib.load().posekf_wahba_f32(N, _ptr(acc_ref), _ptr(mag_ref), shared, _ptr(acc), _ptr(mag), _ptr(ka_t),
                                          _ptr(km_t), ka_s, km_s, int(weights_from_acc), _ptr(R), _ptr(qt),
                                          _lib.WAHBA[algo], int(jacobi_sweeps), _stream())
    _lib.check(rc, "posekf_wahba_f32")
    return R, qt


def tracks(streams, acc_ref, mag_ref, *, dt, n_filters=None, k_acc=0.5, k_mag=0.5, weights_from_acc=False,
           gyro_state=None, want_gyro=True, want_wahba=True, algo: str = "qr2"):
    """Gyro-only and Wahba-only comparison tracks (the curves main_file.py plots beside the filter).
    Returns (gyro [T,N,4] or None, wahba [T,N,4] or None, gyro_state [4,N] -- None for a Wahba-only call without a state)."""
    _require_cuda(streams, acc_ref, mag_ref, gyro_state)
    T, _, Ns = streams.shape
    N = Ns if n_filters is None else int(n_filters)
    dev = streams.device
    if isinstance(dt, torch.Tensor):
        _require_cuda(dt)
        dt_t, per_step = dt, 1
    else:
        dt_t, per_step = _scalar_tensor(dt, dev), 0
    if gyro_state is None and want_gyro:      # (a Wahba-only call integrates nothing)
        gyro_state = torch.zeros((4, N), dtype=torch.float32, device=dev)
        gyro_state[0] = 1.0
    og = torch.empty((T, N, 4), dtype=torch.float32, device=dev) if want_gyro else None
    ow = torch.empty((T, N, 4), dtype=torch.float32, device=dev) if want_wahba else None
    with torch.cuda.device(dev):
        rc = _lib.load().posekf_tracks_f32(N, T, _ptr(streams), Ns, _ptr(dt_t), per_step, _ptr(acc_ref), _ptr(mag_ref),
                                           float(k_acc), float(k_mag), int(weights_from_acc), _ptr(gyro_state), _ptr(og),
                                           _ptr(ow), _lib.WAHBA[algo], _stream())
    _lib.check(rc, "posekf_tracks_f32")
    return og, ow, gyro_state


def preprocess(gyro, raw_prev, raw_next, tspan, *, lpf_alpha_acc=None, lpf_alpha_mag=None, lpf_state=None, out=None):
    """Raw-sensor pre-processing (interpolate accel/mag to the gyro timestamp, normalise, optional
    low-pass): gyro [T,3,N], raw_prev/raw_next [T,6,N], tspan [T,4,N] seconds -> streams [T,9,N]
    (and the low-pass state [6,N])."""
    _require_cuda(gyro, raw_prev, raw_next, tspan, lpf_state, out)
    T, _, N = gyro.shape
    if raw_prev.shape != (T, 6, N) or raw_next.shape != (T, 6, N) or tspan.shape != (T, 4, N):
        raise ValueError("raw_prev/raw_next must be [T,6,N] and tspan [T,4,N]")
    use_lpf = lpf_alpha_acc is not None or lpf_alpha_mag is not None
    if use_lpf and lpf_state is None:
        lpf_state = torch.zeros((6, N), dtype=torch.float32, device=gyro.device)
    if out is None:
        out = torch.empty((T, 9, N), dtype=torch.float32, device=gyro.device)
    with torch.cuda.device(gyro.device):
        rc = _lib.load().posekf_preprocess_f32(N, T, _ptr(gyro), _ptr(raw_prev), _ptr(raw_next), _ptr(tspan),
                                               -1.0 if lpf_alpha_acc is None else float(lpf_alpha_acc),
                                               -1.0 if lpf_alpha_mag is None else float(lpf_alpha_mag),
                                               _ptr(lpf_state), _ptr(out), _stream())
    _lib.check(rc, "posekf_preprocess_f32")
    return out, lpf_state


def initial_values(samples, *, normalize: bool = True, want_variance: bool = False):
    """acc_0 / mag_0 of the online pipeline: (normalised) mean of the first K samples, samples [K,3,N] ->
    (mean [3,N], var [3,N] or None)."""
    _require_cuda(samples)
    K, _, N = samples.shape
    mean = torch.empty((3, N), dtype=torch.float32, device=samples.device)
    var = torch.empty((3, N), dtype=torch.float32, device=samples.device) if want_variance else None
    with torch.cuda.device(samples.device):
        _lib.check(_lib.load().posekf_initial_values_f32(N, K, _ptr(samples), int(normalize), _ptr(mean), _ptr(var), _stream()),
                   "posekf_initial_values_f32")
    return mean, var


def align_events(gyro_t, gyro_v, gyro_off, acc_t, acc_v, acc_off, mag_t, mag_v, mag_off, *, k_init: int = 100):
    """Raw event recordings -> (streams [T,9,Ns], dt [T,Ns], lengths [Ns] int32, acc_ref [3,Ns], mag_ref [3,Ns]) on the
    device (`posekf_align_events_f32`, whose header comment has the rules).  Per sensor: t [M] int64 ns, v [3,M] float32,
    off [Ns+1] int64 CUDA tensors, recording c owning events off[c]..off[c+1]-1, timestamps strictly increasing within a
    recording (checked by `logio.align_recordings`).  T = max(lengths), found with a first lengths-only call."""
    ts, vs, offs = (gyro_t, acc_t, mag_t), (gyro_v, acc_v, mag_v), (gyro_off, acc_off, mag_off)
    _require_cuda(*vs)
    for t, v, off in zip(ts, vs, offs):
        if not (t.is_cuda and off.is_cuda and t.dtype == torch.int64 and off.dtype == torch.int64):
            raise TypeError("timestamps and offsets must be int64 CUDA tensors")
        if not (t.is_contiguous() and off.is_contiguous()) or t.dim() != 1 or v.shape != (3, t.shape[0]):
            raise ValueError("each sensor needs contiguous t [M] and v [3, M]")
        if off.shape != gyro_off.shape or off.dim() != 1:
            raise ValueError("the offsets of the three sensors must all be [Ns + 1]")
    Ns = gyro_off.shape[0] - 1
    dev = gyro_t.device
    lib = _lib.load()
    args = [Ns, int(k_init), _ptr(gyro_t), _ptr(gyro_v), _ptr(gyro_off), _ptr(acc_t), _ptr(acc_v), _ptr(acc_off), _ptr(mag_t),
            _ptr(mag_v), _ptr(mag_off)]
    lengths = torch.empty((max(Ns, 0),), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.posekf_align_events_f32(*args, 0, None, None, _ptr(lengths), None, None, _stream()),
                   "posekf_align_events_f32")
        T = int(lengths.max().item()) if Ns > 0 else 0
        # one row at least, whose pointer is passed: with T = 0 an empty tensor's NULL pointer would select the
        # lengths-only call again, and the reference vectors would not be written
        streams = torch.empty((max(T, 1), 9, Ns), dtype=torch.float32, device=dev)
        dt = torch.empty((max(T, 1), Ns), dtype=torch.float32, device=dev)
        acc_ref = torch.empty((3, Ns), dtype=torch.float32, device=dev)
        mag_ref = torch.empty((3, Ns), dtype=torch.float32, device=dev)
        _lib.check(lib.posekf_align_events_f32(*args, T, _ptr(streams), _ptr(dt), _ptr(lengths), _ptr(acc_ref), _ptr(mag_ref),
                                               _stream()), "posekf_align_events_f32")
    return streams[:T], dt[:T], lengths, acc_ref, mag_ref


def traj2rpy(traj):
    """Quart2RPY over a stored trajectory [..., 4] -> degrees [..., 3]."""
    _require_cuda(traj)
    out = torch.empty(traj.shape[:-1] + (3,), dtype=torch.float32, device=traj.device)
    with torch.cuda.device(traj.device):
        _lib.check(_lib.load().posekf_traj2rpy_f32(traj.numel() // 4, _ptr(traj), _ptr(out), _stream()),
                   "posekf_traj2rpy_f32")
    return out


def rot2quat(rot):
    """Wahba.RotationMatrix2Quart: rot [9,N] -> [4,N]."""
    _require_cuda(rot)
    out = torch.empty((4, rot.shape[1]), dtype=torch.float32, device=rot.device)
    with torch.cuda.device(rot.device):
        _lib.check(_lib.load().posekf_rot2quat_f32(rot.shape[1], _ptr(rot), _ptr(out), _stream()), "posekf_rot2quat_f32")
    return out


def predict(gyro, dt, x, p, q_mat, r_mat, q_scale=None, r_scale=None):
    """KalmanFilter.Prediction: gyro [3,N], dt float or [N] tensor (seconds), x [4,N], p [16,N],
    q_mat [9], r_mat [16] -> (z [4,N], P [16,N], K [16,N])."""
    _require_cuda(gyro, x, p, q_mat, r_mat, q_scale, r_scale)
    N = gyro.shape[1]
    dev = gyro.device
    if isinstance(dt, torch.Tensor):
        _require_cuda(dt)
        dt_t, shared = dt, 0
    else:
        dt_t, shared = torch.full((1,), float(dt), dtype=torch.float32, device=dev), 1
    z = torch.empty((4, N), dtype=torch.float32, device=dev)
    po = torch.empty((16, N), dtype=torch.float32, device=dev)
    ko = torch.empty((16, N), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        rc = _lib.load().posekf_predict_f32(N, _ptr(gyro), _ptr(dt_t), shared, _ptr(x), _ptr(p), _ptr(q_mat),
                                            _ptr(r_mat), _ptr(q_scale), _ptr(r_scale), _ptr(z), _ptr(po), _ptr(ko),
                                            _stream())
    _lib.check(rc, "posekf_predict_f32")
    return z, po, ko


def correct(mag, acc, acc_ref, mag_ref, z, p, k, *, want_flip=False, want_meas=False, algo: str = "qr2"):
    """KalmanFilter.Correction (NB reference order Mag, Acc): -> (X [4,N], P [16,N], flip [N] u8 or
    None, y [4,N] or None)."""
    _require_cuda(mag, acc, acc_ref, mag_ref, z, p, k)
    N = acc.shape[1]
    dev = acc.device
    shared = int(acc_ref.dim() == 1)
    x = torch.empty((4, N), dtype=torch.float32, device=dev)
    po = torch.empty((16, N), dtype=torch.float32, device=dev)
    flip = torch.empty((N,), dtype=torch.uint8, device=dev) if want_flip else None
    meas = torch.empty((4, N), dtype=torch.float32, device=dev) if want_meas else None
    with torch.cuda.device(dev):
        rc = _lib.load().posekf_correct_f32(N, _ptr(mag), _ptr(acc), _ptr(acc_ref), _ptr(mag_ref), shared, _ptr(z),
                                            _ptr(p), _ptr(k), _ptr(x), _ptr(po), _ptr(flip), _ptr(meas),
                                            _lib.WAHBA[algo], _stream())
    _lib.check(rc, "posekf_correct_f32")
    return x, po, flip, meas


def rk4(q, dt, w):
    """KalmanFilter.RungeKutta4 with dt in SECONDS: q [4,N], w [3,N] -> [4,N]."""
    _require_cuda(q, w)
    N = q.shape[1]
    dev = q.device
    if isinstance(dt, torch.Tensor):
        _require_cuda(dt)
        dt_t, shared = dt, 0
    else:
        dt_t, shared = torch.full((1,), float(dt), dtype=torch.float32, device=dev), 1
    out = torch.empty_like(q)
    with torch.cuda.device(dev):
        _lib.check(_lib.load().posekf_rk4_f32(N, _ptr(q), _ptr(dt_t), shared, _ptr(w), _ptr(out), _stream()),
                   "posekf_rk4_f32")
    return out


def jacobian_a(w):
    """GetJacobian_A: w [3,N] -> [16,N]."""
    _require_cuda(w)
    out = torch.empty((16, w.shape[1]), dtype=torch.float32, device=w.device)
    with torch.cuda.device(w.device):
        _lib.check(_lib.load().posekf_jacobians_f32(w.shape[1], _ptr(w), _ptr(out), None, None, _stream()),
                   "posekf_jacobians_f32")
    return out


def jacobian_b(q):
    """GetJacobian_B: q [4,N] -> [12,N] (4x3 row-major)."""
    _require_cuda(q)
    out = torch.empty((12, q.shape[1]), dtype=torch.float32, device=q.device)
    with torch.cuda.device(q.device):
        _lib.check(_lib.load().posekf_jacobians_f32(q.shape[1], None, None, _ptr(q), _ptr(out), _stream()),
                   "posekf_jacobians_f32")
    return out


def comparator(q1, q2):
    """KalmanFilter.Comparator: conj(q1) (x) q2, [4,N] each -> [4,N]."""
    _require_cuda(q1, q2)
    out = torch.empty_like(q1)
    with torch.cuda.device(q1.device):
        _lib.check(_lib.load().posekf_comparator_f32(q1.shape[1], _ptr(q1), _ptr(q2), _ptr(out), _stream()),
                   "posekf_comparator_f32")
    return out


def lowpass(x, alpha: float, state=None):
    """y <- alpha x + (1-alpha) y along time: x [T,3,N] -> (y [T,3,N], state [3,N])."""
    _require_cuda(x, state)
    T, _, N = x.shape
    if state is None:
        state = torch.zeros((3, N), dtype=torch.float32, device=x.device)
    out = torch.empty_like(x)
    with torch.cuda.device(x.device):
        _lib.check(_lib.load().posekf_lowpass_f32(N, T, _ptr(x), float(alpha), _ptr(state), _ptr(out), _stream()),
                   "posekf_lowpass_f32")
    return out, state


def quat2rpy(q):
    """UtilityFunctions.Quart2RPY: q [4,N] -> degrees [3,N]."""
    _require_cuda(q)
    out = torch.empty((3, q.shape[1]), dtype=torch.float32, device=q.device)
    with torch.cuda.device(q.device):
        _lib.check(_lib.load().posekf_quat2rpy_f32(q.shape[1], _ptr(q), _ptr(out), _stream()), "posekf_quat2rpy_f32")
    return out


def norm(v):
    """UtilityFunctions.norm: v [k,N] -> [N]."""
    _require_cuda(v)
    out = torch.empty((v.shape[1],), dtype=torch.float32, device=v.device)
    with torch.cuda.device(v.device):
        _lib.check(_lib.load().posekf_norm_f32(v.shape[1], v.shape[0], _ptr(v), _ptr(out), _stream()),
                   "posekf_norm_f32")
    return out


def fp32_peak_tflops(device: int = 0):
    """Measured FFMA rate of this GPU right now (TFLOP/s, ms of the probe kernel)."""
    import ctypes as C
    tf, ms = C.c_double(), C.c_double()
    _lib.check(_lib.load().posekf_fp32_peak_tflops(int(device), C.byref(tf), C.byref(ms)), "posekf_fp32_peak_tflops")
    return tf.value, ms.value
