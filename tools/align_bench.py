#!/usr/bin/env python
"""Speed of the raw-event alignment (posekf_align_events_f32, logio.align_recordings), one GPU, CUDA events, medians:

  * the alignment alone on 16 Ki recordings x 60 s at gyro 200 Hz and acc / mag 100 Hz (jittered clocks, random phase;
    the values are random: the cost does not depend on them), and the bytes it must move (every event read once, the
    streams and dt written) over its time, as a fraction of the device-to-device copy bandwidth measured in the same run;
  * the path a user has without it: the numpy bracket search per recording + B.preprocess + B.initial_values, on a
    subsample of recordings, scaled to the batch;
  * alignment + replay against the replay alone (q = 1, r = 0.1, the batch's own dt and lengths).

  python tools/align_bench.py [--reps 7] [--recordings 16384] [--seconds 60] [--out profiles/r08_align_events.json]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from batch_bench import alternate, card, median  # noqa: E402


def sensor(n_rec, seconds, hz, jitter, g, dev):
    """One sensor of every recording: t [M] int64 ns, v [3, M] float32, off [n_rec + 1] int64 (equal counts)."""
    import torch
    n = int(seconds * hz)
    k = torch.arange(n, device=dev, dtype=torch.float64)
    phase = torch.rand((n_rec, 1), generator=g, device=dev, dtype=torch.float64)
    u = torch.rand((n_rec, n), generator=g, device=dev, dtype=torch.float64) - 0.5
    t = torch.round((phase + k + jitter * u) / hz * 1e9).to(torch.int64) + 1_700_000_000_000_000_000
    v = torch.randn((3, n_rec * n), generator=g, device=dev)
    off = torch.arange(n_rec + 1, device=dev, dtype=torch.int64) * n
    return t.reshape(-1), v, off


def numpy_path(tg, vg, ta, va, tm, vm, k_init, dev):
    """Today's path for a few recordings (host numpy arrays per recording): brackets, spans and dt on the host, then
    B.initial_values and B.preprocess on the device."""
    import numpy as np
    import torch
    from poseestimationkf_b200 import batched as B
    n = len(tg)
    per = []
    for c in range(n):
        t_init = max(ta[c][k_init - 1], tm[c][k_init - 1])
        first = np.searchsorted(tg[c], t_init, side="right")
        stop = np.searchsorted(tg[c], min(ta[c][-1], tm[c][-1]), side="left")
        g = tg[c][first:stop]
        prev, nxt, span = [], [], []
        for t, v in ((ta[c], va[c]), (tm[c], vm[c])):
            j = np.searchsorted(t, g, side="right") - 1
            prev.append(v[j]); nxt.append(v[j + 1])
            span += [((t[j + 1] - t[j]) * 1e-9).astype(np.float32), ((g - t[j]) * 1e-9).astype(np.float32)]
        dt = (np.diff(np.concatenate([[t_init], g])) * 1e-9).astype(np.float32)
        per.append((vg[c][first:stop], np.concatenate(prev, 1), np.concatenate(nxt, 1), np.stack(span, 1), dt))
    T = max(p[0].shape[0] for p in per)
    arr = lambda i, w: np.stack([np.pad(p[i], ((0, T - p[i].shape[0]), (0, 0)), mode="edge") for p in per], axis=2)
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev)
    out, _ = B.preprocess(d(arr(0, 3)), d(arr(1, 6)), d(arr(2, 6)), d(arr(3, 4)))
    first_k = lambda vs: d(np.stack([v[:k_init] for v in vs], axis=2))
    B.initial_values(first_k(va))
    B.initial_values(first_k(vm))
    torch.cuda.synchronize()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--recordings", type=int, default=16384)
    ap.add_argument("--seconds", type=float, default=60.0)
    ap.add_argument("--rates", type=float, nargs=3, default=(200.0, 100.0, 100.0))
    ap.add_argument("--subsample", type=int, default=64, help="recordings timed on the numpy + B.preprocess path")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_align_events.json"))
    a = ap.parse_args()
    import torch
    from poseestimationkf_b200 import _lib
    from poseestimationkf_b200 import batched as B
    assert torch.cuda.is_available(), "needs a GPU"
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev)
    g.manual_seed(0)
    Ns, K = a.recordings, 100
    ev = [sensor(Ns, a.seconds, hz, 0.2, g, dev) for hz in a.rates]
    res = {"card": card(), "torch": torch.__version__, "recordings": Ns, "seconds": a.seconds, "rates_hz": list(a.rates),
           "k_init": K, "timing": "CUDA events around each call, one warm-up per variant, variants alternated, medians"}
    (tg, vg, og), (ta, va, oa), (tm, vm, om) = ev
    streams, dt, lengths, acc_ref, mag_ref = B.align_events(tg, vg, og, ta, va, oa, tm, vm, om, k_init=K)
    T = streams.shape[0]
    lib = _lib.load()
    args = [x.data_ptr() for x in (tg, vg, og, ta, va, oa, tm, vm, om)]

    def align():
        _lib.check(lib.posekf_align_events_f32(Ns, K, *args, T, streams.data_ptr(), dt.data_ptr(), lengths.data_ptr(),
                                               acc_ref.data_ptr(), mag_ref.data_ptr(), B._stream()), "align")

    def replay():
        B.replay(streams, acc_ref, mag_ref, dt=dt, q=1.0, r=0.1, lengths=lengths)

    def both():
        align()
        replay()

    # copy bandwidth of this device in this run: a 4 GiB device-to-device copy (read + write)
    src = torch.empty((1 << 30,), dtype=torch.float32, device=dev)
    dst = torch.empty_like(src)
    copy = alternate({"copy": lambda: dst.copy_(src)}, a.reps)["copy"]
    del src, dst
    copy_bw = 2 * (1 << 32) / (copy["ms_median"] * 1e-3)
    t = alternate({"align": align, "replay": replay, "align_then_replay": both}, a.reps)
    steps = int(lengths.sum())
    M = [int(o[-1]) for o in (og, oa, om)]
    nbytes = 20 * sum(M) + 40 * T * Ns          # 8 B timestamp + 12 B value per event read; 9 + 1 floats per step written
    ms = t["align"]["ms_median"]
    res.update(events={"gyro": M[0], "acc": M[1], "mag": M[2]}, T=T, steps=steps, min_bytes=nbytes,
               copy_ms=copy, copy_bandwidth_GBps=copy_bw / 1e9, **t,
               align_GBps=nbytes / (ms * 1e-3) / 1e9, align_fraction_of_copy=nbytes / (ms * 1e-3) / copy_bw,
               align_ns_per_step=ms * 1e6 / steps, replay_ms_per_G_filter_steps=t["replay"]["ms_median"] / (steps / 1e9))

    # the numpy + B.preprocess path on a subsample, scaled to the batch
    n = min(a.subsample, Ns)
    host = [[x.cpu().numpy() for x in s] for s in ev]
    split = lambda t_, v_, o_: ([t_[o_[c]:o_[c + 1]] for c in range(n)], [v_[:, o_[c]:o_[c + 1]].T.copy() for c in range(n)])
    (tgs, vgs), (tas, vas), (tms, vms) = (split(*h) for h in host)
    numpy_path(tgs, vgs, tas, vas, tms, vms, K, dev)            # warm-up
    wall = []
    for _ in range(a.reps):
        t0 = time.perf_counter()
        numpy_path(tgs, vgs, tas, vas, tms, vms, K, dev)
        wall.append((time.perf_counter() - t0) * 1e3)
    scaled = median(wall) * Ns / n
    res.update(numpy_path={"recordings_timed": n, "ms": wall, "ms_median": median(wall), "ms_scaled_to_batch": scaled},
               speedup_vs_numpy_path=scaled / ms)
    print(json.dumps(res))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
