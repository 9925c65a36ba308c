"""Alignment of raw event recordings to the gyro clock without a GPU: the float64 definition (tests/align_ref.py) on
hand-built recordings with the lengths, brackets and dt worked out by hand, the host argument rules of
`logio.align_recordings`, and the POSEKF_EINVAL cases of `posekf_align_events_f32`."""
import numpy as np
import pytest

from oracle import ekf_oracle as O
from poseestimationkf_b200 import _lib, logio
from tests import align_ref as AR

MS = 1_000_000          # ns


def _ev(t, v=None, seed=0):
    t = np.asarray(t, dtype=np.int64)
    if v is None:
        v = np.random.default_rng(seed).normal(size=(t.size, 3)).astype(np.float32)
    return logio.SensorEvents(t, np.asarray(v, dtype=np.float32))


def _rec(tg, ta, tm, base=0):
    return logio.RawRecording(_ev(np.asarray(tg) + base, seed=1), _ev(np.asarray(ta) + base, seed=2),
                              _ev(np.asarray(tm) + base, seed=3))


# k_init = 2.  acc at 10, 20, 30, 40, 50 ms; mag at 12, 25, 38, 51 ms -> t_init = max(20, 25) = 25, and the last step
# must come before min(50, 51) = 50.  Gyro at 5, 18, 22, 25 (before or at t_init: dropped), 30, 33, 45 (the steps),
# 50, 52, 60 (at or after the last acc event: dropped).
TG = [5, 18, 22, 25, 30, 33, 45, 50, 52, 60]
TA = [10, 20, 30, 40, 50]
TM = [12, 25, 38, 51]


@pytest.mark.parametrize("base", [0, 2 ** 62 - 17 * MS], ids=["zero", "near_2^62"])
def test_hand_built_recording(base):
    rec = _rec(np.multiply(TG, MS), np.multiply(TA, MS), np.multiply(TM, MS), base)
    a = AR.align_one(rec, k_init=2)
    assert a["length"] == 3 and a["first"] == 4 and a["t_init"] == base + 25 * MS
    # gyro 30 ms equals an acc timestamp: that event is t1 (t1 <= t_g), the next one t2
    np.testing.assert_array_equal(a["j_acc"], [2, 2, 3])            # acc (30,40), (30,40), (40,50)
    # gyro 30 and 33 ms lie between the same pair of mag events (25, 38)
    np.testing.assert_array_equal(a["j_mag"], [1, 1, 2])            # mag (25,38), (25,38), (38,51)
    # dt: (30 - 25), (33 - 30), (45 - 33) ms, exact differences whatever the epoch
    np.testing.assert_array_equal(a["dt"], np.float32([5e-3, 3e-3, 12e-3]))
    np.testing.assert_array_equal(AR.tspans(rec, a),
                                  np.float32([[10e-3, 0.0, 13e-3, 5e-3], [10e-3, 3e-3, 13e-3, 8e-3],
                                              [10e-3, 5e-3, 13e-3, 7e-3]]))
    va, vm, vg = (e.v.astype(np.float64) for e in (rec.acc, rec.mag, rec.gyro))
    np.testing.assert_array_equal(a["streams"][:, 0:3], vg[4:7])
    want_acc = O.interpolate_normalise(va[[2, 2, 3]], va[[3, 3, 4]], 0.0, 10.0 * MS, np.array([0, 3, 5]) * MS)
    want_mag = O.interpolate_normalise(vm[[1, 1, 2]], vm[[2, 2, 3]], 0.0, 13.0 * MS, np.array([5, 8, 7]) * MS)
    np.testing.assert_array_equal(a["streams"][:, 3:6], want_acc)
    np.testing.assert_array_equal(a["streams"][:, 6:9], want_mag)
    np.testing.assert_array_equal(a["acc_ref"], O.normalize_values(O.initial_values(va[:2])[0]))
    np.testing.assert_array_equal(a["mag_ref"], O.normalize_values(O.initial_values(vm[:2])[0]))


def test_too_few_events_gives_length_zero_and_padding_references():
    rec = _rec(np.multiply(TG, MS), np.multiply(TA[:1], MS), np.multiply(TM, MS))
    a = AR.align_one(rec, k_init=2)
    assert a["length"] == 0 and a["dt"].size == 0
    np.testing.assert_array_equal(a["acc_ref"], [0, 0, 1])
    np.testing.assert_array_equal(a["mag_ref"], [1, 0, 0])
    # enough events, but no gyro event after t_init that both sensors bracket
    b = AR.align_one(_rec(np.multiply([5, 18, 60], MS), np.multiply(TA, MS), np.multiply(TM, MS)), k_init=2)
    assert b["length"] == 0 and b["t_init"] == 25 * MS


def test_align_recordings_argument_rules():
    good = _rec(np.multiply(TG, MS), np.multiply(TA, MS), np.multiply(TM, MS))
    with pytest.raises(ValueError, match="strictly increasing"):
        logio.align_recordings([good, _rec([1, 2, 2, 3], TA, TM)], device="cpu", k_init=2)
    with pytest.raises(ValueError, match="strictly increasing"):
        logio.align_recordings([_rec(TG, [10, 20, 15], TM)], device="cpu", k_init=2)
    bad = logio.RawRecording(good.gyro, logio.SensorEvents(good.acc.t_ns, good.acc.v[:-1]), good.mag)
    with pytest.raises(ValueError, match=r"v \[M,3\]"):
        logio.align_recordings([bad], device="cpu", k_init=2)
    with pytest.raises(TypeError, match="integer ns"):
        logio.align_recordings([logio.RawRecording(logio.SensorEvents(np.float64(TG), good.gyro.v), good.acc, good.mag)],
                               device="cpu", k_init=2)
    for k in (0, -1):
        with pytest.raises(ValueError, match="k_init"):
            logio.align_recordings([good], device="cpu", k_init=k)


def test_capi_argument_validation_without_gpu():
    lib = _lib.load()
    f = lib.posekf_align_events_f32
    p = 16                              # any non-null address: each call returns before it is used
    full = [p] * 9
    assert f(-1, 100, *full, 4, p, p, p, p, p, None) == _lib.EINVAL            # negative size
    assert f(4, 100, *full, -1, p, p, p, p, p, None) == _lib.EINVAL            # negative t_out
    assert f(4, 0, *full, 4, p, p, p, p, p, None) == _lib.EINVAL               # k_init < 1
    assert f(0, 100, *[None] * 9, 0, None, None, None, None, None, None) == 0  # empty batch is a no-op
    for i in (0, 2, 3, 5, 6, 8):        # timestamps and offsets are always required
        args = list(full)
        args[i] = None
        assert f(4, 100, *args, 4, None, None, p, None, None, None) == _lib.EINVAL, i
    assert f(4, 100, *full, 4, None, None, None, None, None, None) == _lib.EINVAL   # lengths
    for i in (1, 4, 7):                 # values, dt and references are required unless streams is NULL
        args = list(full)
        args[i] = None
        assert f(4, 100, *args, 4, p, p, p, p, p, None) == _lib.EINVAL, i
    for j in range(1, 5):
        outs = [p] * 5
        if j == 2:
            continue                    # (lengths, checked above)
        outs[j] = None
        assert f(4, 100, *full, 4, *outs, None) == _lib.EINVAL, j
