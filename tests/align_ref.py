"""Float64 definition of the alignment of raw event recordings to the gyro clock (`posekf_align_events_f32`,
DESIGN section 5 f10), written with numpy: `np.searchsorted` for the brackets and the oracle's `interpolate_normalise` /
`initial_values` restatements, which tests/test_oracle.py pins bit for bit to the reference's own C++ text."""
import numpy as np

from oracle import ekf_oracle as O

PAD_ACC, PAD_MAG = np.array([0.0, 0.0, 1.0]), np.array([1.0, 0.0, 0.0])      # logio.stack_logs' padding references


def ns_to_f32_seconds(d):
    """An int64 ns difference as float32 seconds: float64 product with 1e-9, rounded to float32 once."""
    return (np.asarray(d, dtype=np.int64).astype(np.float64) * 1e-9).astype(np.float32)


def align_one(rec, k_init=100):
    """One `logio.RawRecording` -> dict with
    length, first (gyro index of step 0), t_init, acc_ref / mag_ref [3] float64, j_acc / j_mag [L] (index of the last
    event at or before each step's gyro timestamp; the next event is the other bracket), dt [L] float32,
    streams [L,9] float64 (gyro as recorded, acc / mag interpolated and normalised in float64 on the float32 events,
    the time spans in float64 ns)."""
    tg, ta, tm = (np.asarray(e.t_ns, dtype=np.int64) for e in (rec.gyro, rec.acc, rec.mag))
    vg, va, vm = (np.asarray(e.v, dtype=np.float32).astype(np.float64) for e in (rec.gyro, rec.acc, rec.mag))
    out = dict(length=0, first=0, t_init=0, acc_ref=PAD_ACC.copy(), mag_ref=PAD_MAG.copy(), j_acc=np.zeros(0, np.int64),
               j_mag=np.zeros(0, np.int64), dt=np.zeros(0, np.float32), streams=np.zeros((0, 9)))
    if ta.size < k_init or tm.size < k_init:
        return out
    t_init = max(int(ta[k_init - 1]), int(tm[k_init - 1]))
    t_end = min(int(ta[-1]), int(tm[-1]))
    first = int(np.searchsorted(tg, t_init, side="right"))         # first gyro event after t_init
    stop = int(np.searchsorted(tg, t_end, side="left"))            # first gyro event at or after the last acc / mag
    L = max(0, stop - first)
    out.update(t_init=t_init, first=first, length=L)
    out["acc_ref"] = O.normalize_values(O.initial_values(va[:k_init])[0])
    out["mag_ref"] = O.normalize_values(O.initial_values(vm[:k_init])[0])
    g = tg[first:first + L]
    streams = np.zeros((L, 9))
    streams[:, 0:3] = vg[first:first + L]
    for name, t, v, rows in (("j_acc", ta, va, slice(3, 6)), ("j_mag", tm, vm, slice(6, 9))):
        j = np.searchsorted(t, g, side="right") - 1                 # last event with t1 <= t_g
        out[name] = j
        # times relative to t1, differenced in int64: exact in float64 whatever the epoch of the timestamps
        streams[:, rows] = O.interpolate_normalise(v[j], v[j + 1], np.zeros(L), t[j + 1] - t[j], g - t[j]) if L else \
            np.zeros((0, 3))
    prev = np.concatenate([[t_init], g[:-1]]) if L else np.zeros(0, np.int64)
    out["dt"] = ns_to_f32_seconds(g - prev)
    out["streams"] = streams
    return out


def align_events(recs, k_init=100):
    """Every recording of a batch: a list of `align_one` dicts."""
    return [align_one(r, k_init) for r in recs]


def tspans(rec, a):
    """The float32 seconds the device forms for one recording's steps: [L,4] acc (t2-t1), acc (t3-t1), mag (t2-t1),
    mag (t3-t1), differenced in int64 ns (the `tspan` argument of `posekf_preprocess_f32`)."""
    tg = np.asarray(rec.gyro.t_ns, dtype=np.int64)[a["first"]:a["first"] + a["length"]]
    cols = []
    for e, j in ((rec.acc, a["j_acc"]), (rec.mag, a["j_mag"])):
        t = np.asarray(e.t_ns, dtype=np.int64)
        cols += [ns_to_f32_seconds(t[j + 1] - t[j]), ns_to_f32_seconds(tg - t[j])]
    return np.stack(cols, axis=1) if a["length"] else np.zeros((0, 4), np.float32)
