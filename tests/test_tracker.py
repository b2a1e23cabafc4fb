"""Native host side of the filter stage (csrc/tracker.cpp, SURVEY.md 8f item 1): the centroid tracker of
TrackFilter (watsor/filter/track.py:29-149) and the sieve write-back (watsor/filter/sieve.py:21-52).

Pinned by (a) the reference's known answers (watsor/test/test_filter.py:76-96), (b) the reference's TrackFilter
itself, its results recorded in tests/golden/reference/tracker.json (tests/reference_outputs.py), (c) the oracle restatement, (d) the CPython interpreter for
the set iteration orders the reference leaks into its results.  No GPU involved."""
import ctypes
import os
import random
import sys

import numpy as np
import pytest

from oracle.filters import Det, TrackOracle
from watsor_b200 import _lib
from watsor_b200.stream.share import MAX_DETECTIONS, BoundingBox, Detection

from tests.reference_outputs import REFERENCE as REF  # noqa: E402
from tests.reference_outputs import Recorded  # noqa: E402

recorded = Recorded('tracker')


class NativeTracker:
    def __init__(self, sensitivity=5, history=10):
        self.lib = _lib.load()
        self.h = ctypes.c_void_p()
        assert self.lib.wb_tracker_create(sensitivity, history, ctypes.byref(self.h)) == 0

    def __call__(self, dets, verdicts=None):
        n = len(dets)
        rows = (Detection * max(n, 1))()
        for i, d in enumerate(dets):
            ctypes.memmove(ctypes.addressof(rows[i]), ctypes.addressof(d), ctypes.sizeof(Detection))
        out = (Detection * max(n, 1))()
        n_out, sa = ctypes.c_int(), ctypes.c_int()
        v = (ctypes.c_uint32 * max(n, 1))(*verdicts) if verdicts is not None else None
        rc = self.lib.wb_tracker_update(self.h, rows, n, v, out, n, ctypes.byref(n_out), ctypes.byref(sa))
        assert rc == 0
        return [out[i] for i in range(n_out.value)], bool(sa.value)

    def __del__(self):
        self.lib.wb_tracker_destroy(self.h)


def key(d):
    bb = d.bounding_box if hasattr(d, 'bounding_box') else d
    return (d.label, tuple(d.zones), d.confidence, bb.x_min, bb.y_min, bb.x_max, bb.y_max)


def mk(label, conf, box, zones=()):
    d = Detection(label=label, confidence=conf, bounding_box=BoundingBox(*box))
    for i, z in enumerate(zones):
        d.zones[i] = z
    return d


def random_frames(rng, n_frames, max_per_label, n_labels, n_zone_ids, jitter=12):
    """A scene of moving objects with births, deaths and flicker; integer boxes inside 640x480."""
    objs = []
    frames = []
    for _ in range(n_frames):
        objs = [o for o in objs if rng.random() > 0.12]
        while len(objs) < rng.randint(0, max_per_label * n_labels):
            w, h = rng.randint(8, 120), rng.randint(8, 120)
            objs.append([rng.randint(1, n_labels), rng.randint(0, 639 - w), rng.randint(0, 479 - h), w, h])
        dets = []
        for o in objs:
            o[1] = min(max(o[1] + rng.randint(-jitter, jitter), 0), 639 - o[3])
            o[2] = min(max(o[2] + rng.randint(-jitter, jitter), 0), 479 - o[4])
            if rng.random() < 0.15:
                continue                                      # missed in this frame
            zones = sorted(rng.sample(range(1, n_zone_ids + 1), rng.randint(0, min(3, n_zone_ids))))
            dets.append((o[0], round(rng.uniform(0.3, 1.0), 3), (o[1], o[2], o[1] + o[3], o[2] + o[4]), zones))
        rng.shuffle(dets)
        if rng.random() < 0.1:
            dets = []
        frames.append(dets[:MAX_DETECTIONS])
    return frames


def test_reference_known_answers():
    # watsor/test/test_filter.py:76-96
    t = NativeTracker(sensitivity=1, history=2)
    out, sa = t([mk(1, 0.70, (50, 50, 60, 60)), mk(1, 0.70, (10, 10, 30, 30))])
    assert sa and [key(d)[3:] for d in out] == [(50, 50, 60, 60), (10, 10, 30, 30)]
    out, sa = t([mk(1, 0.70, (40, 40, 55, 55)), mk(1, 0.70, (80, 80, 90, 90))])
    assert sa and [key(d)[3:] for d in out] == [(40, 40, 60, 60), (80, 80, 90, 90)]
    out, sa = t([])
    assert not sa and out == []


def test_label_zero_and_verdicts_select_the_rows():
    t = NativeTracker(sensitivity=1, history=3)
    dets = [mk(0, 0.9, (1, 1, 5, 5)), mk(2, 0.9, (10, 10, 20, 20)), mk(3, 0.9, (30, 30, 40, 40))]
    out, sa = t(dets)
    assert sa and [d.label for d in out] == [2, 3]               # label > 0 (track.py:26)
    t = NativeTracker(sensitivity=1, history=3)
    out, sa = t(dets, verdicts=[_lib.WB_V_PASS | 1, 1, _lib.WB_V_PASS | 15])
    assert [d.label for d in out] == [0, 3]                        # the GPU verdict decides, not the label
    out, sa = t(dets, verdicts=[0, 0, 0])
    assert not sa and out == []


@pytest.mark.parametrize('seed', range(6))
def test_pyset_iteration_order_matches_interpreter(seed):
    lib = _lib.load()
    rng = random.Random(seed)
    for _ in range(400):
        hi = rng.choice([8, 12, 33, 64, 200])
        keys = [rng.randrange(0, hi) for _ in range(rng.randint(0, 45))]
        s = set()
        for k in keys:
            s.add(k)
        arr = (ctypes.c_int32 * max(len(keys), 1))(*keys)
        out = (ctypes.c_int32 * max(len(keys), 1))()
        n = ctypes.c_int()
        assert lib.wb_debug_pyset_order(arr, len(keys), out, ctypes.byref(n)) == 0
        assert list(out[:n.value]) == list(s), keys


@pytest.mark.parametrize('seed', range(4))
def test_unused_cols_order_matches_interpreter(seed):
    lib = _lib.load()
    rng = random.Random(100 + seed)
    for _ in range(600):
        n = rng.randint(0, 70)
        used = set(rng.sample(range(n), rng.randint(0, n))) if n else set()
        expect = list(set(range(n)).difference(used))             # track.py:90,98
        flags = (ctypes.c_uint8 * max(n, 1))(*[1 if i in used else 0 for i in range(n)])
        out = (ctypes.c_int32 * max(n, 1))()
        k = ctypes.c_int()
        assert lib.wb_debug_unused_order(n, flags, out, ctypes.byref(k)) == 0
        assert list(out[:k.value]) == expect, (n, sorted(used))


@pytest.mark.parametrize('seed,sens,hist,per_label,labels,zone_ids',
                         [(1, 1, 2, 3, 2, 3), (2, 3, 5, 5, 3, 6), (3, 5, 10, 12, 2, 12), (4, 2, 4, 14, 1, 9),
                          (5, 1, 1, 6, 4, 20), (6, 4, 3, 9, 3, 10)])
def test_native_tracker_equals_oracle(seed, sens, hist, per_label, labels, zone_ids):
    rng = random.Random(seed)
    frames = random_frames(rng, 120, per_label, labels, zone_ids)
    nat, orc = NativeTracker(sens, hist), TrackOracle(sensitivity=sens, history=hist)
    for f, dets in enumerate(frames):
        got, sa = nat([mk(*d) for d in dets])
        exp, sa_o = orc([Det(l, c, b, list(z) + [0] * (10 - len(z))) for l, c, b, z in dets])
        assert sa == sa_o, f
        assert [key(d) for d in got] == [d.key() for d in exp], f


def frame_digest(sa, dets):
    """A tracker's answer for one frame, (sa, the kept detections' keys), as a short digest."""
    import hashlib
    return hashlib.sha256(repr((sa, [key(d) for d in dets])).encode()).hexdigest()[:16]


def reference_trackfilter(frames, sens, hist):
    """frame_digest() of the reference's TrackFilter on every frame."""
    sys.path.insert(0, REF)
    try:
        from watsor.filter.track import TrackFilter as RefTrackFilter
        from watsor.stream.share import BoundingBox as RefBox
        from watsor.stream.share import Detection as RefDetection
    finally:
        sys.path.remove(REF)
    ref, out = RefTrackFilter(sensitivity=sens, history=hist), []
    for dets in frames:
        rdets = []
        for l, c, b, z in dets:
            d = RefDetection(label=l, confidence=c, bounding_box=RefBox(*b))
            for i, zz in enumerate(z):
                d.zones[i] = zz
            rdets.append(d)
        exp, sa = ref(rdets)
        assert isinstance(sa, bool)
        out.append(frame_digest(sa, exp))
    return out


@pytest.mark.parametrize('seed,sens,hist,per_label,labels,zone_ids',
                         [(11, 1, 2, 3, 2, 3), (12, 5, 10, 10, 3, 12), (13, 2, 4, 14, 1, 9), (14, 3, 6, 7, 5, 5)])
def test_native_tracker_equals_reference_trackfilter(seed, sens, hist, per_label, labels, zone_ids):
    """The reference's own TrackFilter (watsor/filter/track.py), frame by frame."""
    rng = random.Random(seed)
    frames = random_frames(rng, 150, per_label, labels, zone_ids)
    theirs = recorded('trackfilter %d' % seed, lambda: reference_trackfilter(frames, sens, hist))
    assert len(theirs) == len(frames)
    nat = NativeTracker(sens, hist)
    for f, dets in enumerate(frames):
        got, sa = nat([mk(*d) for d in dets])
        assert frame_digest(sa, got) == theirs[f], f


def test_sieve_rows_writes_back_and_zero_fills():
    # watsor/filter/sieve.py:21-52 with filters == [TrackFilter(sensitivity=1)]
    lib = _lib.load()
    h = ctypes.c_void_p()
    assert lib.wb_tracker_create(1, 2, ctypes.byref(h)) == 0
    rows = (Detection * MAX_DETECTIONS)()
    for i, (l, box) in enumerate([(0, (1, 1, 2, 2)), (2, (10, 10, 20, 20)), (0, (0, 0, 0, 0)), (1, (30, 30, 50, 50))]):
        rows[i].label, rows[i].confidence = l, 0.5 + 0.1 * i
        rows[i].bounding_box = BoundingBox(*box)
    sa = ctypes.c_int()
    assert lib.wb_sieve_rows(h, rows, MAX_DETECTIONS, None, ctypes.byref(sa)) == 0
    assert sa.value == 1
    assert [(rows[i].label, rows[i].bounding_box.x_min) for i in range(3)] == [(2, 10), (1, 30), (0, 0)]
    assert bytes(rows)[2 * ctypes.sizeof(Detection):] == bytes((MAX_DETECTIONS - 2) * ctypes.sizeof(Detection))
    assert lib.wb_sieve_rows(h, rows, MAX_DETECTIONS, None, ctypes.byref(sa)) == 0
    assert [rows[i].label for i in range(3)] == [2, 1, 0] and sa.value == 1
    lib.wb_tracker_destroy(h)


def test_python_trackfilter_and_sieve_use_the_native_tracker():
    """watsor_b200.filter.TrackFilter without predicates needs no GPU: stage 1 is `label > 0`."""
    from watsor_b200.filter.sieve import sieve_frame
    from watsor_b200.filter.track import TrackFilter
    t = TrackFilter(sensitivity=1, history=2)
    out, sa = t([mk(1, 0.70, (50, 50, 60, 60)), mk(1, 0.70, (10, 10, 30, 30)), mk(0, 0.9, (1, 1, 2, 2))])
    assert sa and [key(d)[3:] for d in out] == [(50, 50, 60, 60), (10, 10, 30, 30)]
    assert all(isinstance(d, Detection) for d in out)
    rows = (Detection * MAX_DETECTIONS)()
    rows[0].label, rows[0].confidence, rows[0].bounding_box = 1, 0.7, BoundingBox(40, 40, 55, 55)
    rows[5].label, rows[5].confidence, rows[5].bounding_box = 1, 0.8, BoundingBox(80, 80, 90, 90)
    assert t.can_sieve and sieve_frame(rows, [t]) is True
    assert [key(rows[i])[3:] for i in range(3)] == [(40, 40, 60, 60), (80, 80, 90, 90), (0, 0, 0, 0)]
    assert rows[0].confidence == 0.7 and rows[1].confidence == 0.8

    def foreign(d):
        return d.confidence > 0.75
    t2 = TrackFilter([foreign], sensitivity=1, history=2)
    assert not t2.can_sieve
    assert sieve_frame(rows, [t2]) is True                          # generic route, same contract
    assert [rows[i].label for i in range(2)] == [1, 0] and key(rows[0])[3:] == (80, 80, 90, 90)


@pytest.mark.parametrize('seed', range(12))
def test_sieve_rows_with_verdicts_equals_oracle_chain(seed):
    """The data flow of tests/test_gpu_filters.py::test_track_filter_fused_predicates_and_sieve_match_oracle with
    the predicate stage taken from the oracle instead of the GPU: 100 random rows per frame (5 labels, ~20 rows
    each, many equal minimum distances), verdict bits + zones in, sieve write-back out."""
    from oracle.filters import AreaOracle, ConfidenceOracle, MaskOracle, apply_predicates
    from tests.conftest import PORCH_CONFIG
    from tests.test_gpu_filters import random_rows
    lib = _lib.load()
    preds = [ConfidenceOracle(PORCH_CONFIG), AreaOracle(PORCH_CONFIG), MaskOracle(PORCH_CONFIG)]
    oracle = TrackOracle(preds, sensitivity=2, history=3)
    h = ctypes.c_void_p()
    assert lib.wb_tracker_create(2, 3, ctypes.byref(h)) == 0
    rng = np.random.default_rng(1000 + seed)
    anchors = [(int(rng.integers(0, 500)), int(rng.integers(0, 380)), int(rng.integers(1, 4))) for _ in range(6)]
    for frame in range(10):
        rows, dets = random_rows(rng, 640, 480, 100)
        for i, (x, y, lab) in enumerate(anchors):
            dx, dy = int(rng.integers(-3, 4)), int(rng.integers(-3, 4))
            rows[i].label, rows[i].confidence = lab, 0.9
            rows[i].bounding_box = BoundingBox(x + dx, y + dy, x + 120 + dx, y + 90 + dy)
            dets[i] = Det(lab, 0.9, (x + dx, y + dy, x + 120 + dx, y + 90 + dy))
        judged = [d.clone() for d in dets]
        _, bits = apply_predicates(judged, preds)                  # writes zones like the GPU stage does
        verdicts = (ctypes.c_uint32 * 100)()
        for r in range(100):
            verdicts[r] = bits[r] | (_lib.WB_V_PASS if bits[r] == 15 else 0)
            for z in range(10):
                rows[r].zones[z] = judged[r].zones[z]
        sa = ctypes.c_int()
        assert lib.wb_sieve_rows(h, rows, 100, verdicts, ctypes.byref(sa)) == 0
        want, want_sa = oracle(dets)
        assert bool(sa.value) == want_sa
        got = [key(rows[r]) for r in range(100)]
        assert got[:len(want)] == [d.key() for d in want], frame
        assert all(g == (0, (0,) * 10, 0.0, 0, 0, 0, 0) for g in got[len(want):])
    lib.wb_tracker_destroy(h)


def test_tracker_edge_cases():
    lib = _lib.load()
    # sensitivity above history: objects are tracked but never reported (track.py:108-110)
    t = NativeTracker(sensitivity=3, history=2)
    for _ in range(5):
        out, sa = t([mk(1, 0.9, (10, 10, 20, 20))])
        assert sa and out == []
    # a label that disappears loses its history and starts over (track.py:41-46)
    t = NativeTracker(sensitivity=2, history=5)
    assert t([mk(1, 0.9, (10, 10, 20, 20))])[0] == []
    assert len(t([mk(1, 0.8, (11, 11, 21, 21))])[0]) == 1
    assert t([mk(2, 0.9, (10, 10, 20, 20))])[0] == []                 # label 1 gone, label 2 new
    assert t([mk(1, 0.9, (10, 10, 20, 20)), mk(2, 0.7, (12, 12, 22, 22))])[0][0].label == 2
    # history window: the envelope forgets boxes older than `history` frames (deque maxlen)
    t = NativeTracker(sensitivity=1, history=2)
    t([mk(1, 0.9, (0, 0, 10, 10))])
    t([mk(1, 0.5, (2, 2, 12, 12))])
    out, _ = t([mk(1, 0.6, (4, 4, 14, 14))])
    assert key(out[0])[2:] == (0.6, 2, 2, 14, 14)                    # first frame dropped, max conf of the last two
    # empty input, bad arguments, out_cap too small
    h = ctypes.c_void_p()
    assert lib.wb_tracker_create(1, 0, ctypes.byref(h)) != 0          # deque(maxlen=0) cannot hold a detection
    assert lib.wb_tracker_create(1, 3, ctypes.byref(h)) == 0
    n_out, sa = ctypes.c_int(-1), ctypes.c_int(-1)
    assert lib.wb_tracker_update(h, None, 0, None, None, 0, ctypes.byref(n_out), ctypes.byref(sa)) == 0
    assert (n_out.value, sa.value) == (0, 0)
    rows = (Detection * 3)()
    for i in range(3):
        rows[i].label, rows[i].bounding_box = 1, BoundingBox(50 * i, 0, 50 * i + 10, 10)
    out = (Detection * 1)()
    assert lib.wb_tracker_update(h, rows, 3, None, out, 1, ctypes.byref(n_out), ctypes.byref(sa)) == 2
    assert n_out.value == 3 and out[0].bounding_box.x_min == 0
    assert lib.wb_tracker_update(h, rows, -1, None, out, 1, ctypes.byref(n_out), ctypes.byref(sa)) == 1
    lib.wb_tracker_destroy(h)


def test_negative_and_unordered_boxes_use_python_int_truncation():
    # track.py:120-123: int((a + b) / 2.0) truncates toward zero, also for negative sums
    t = NativeTracker(sensitivity=1, history=3)
    t([mk(1, 0.9, (-7, -7, 0, 0)), mk(1, 0.9, (-3, -3, 0, 0))])       # centroids (-3,-3) and (-1,-1)
    out, _ = t([mk(1, 0.8, (-4, -4, 0, 0))])                          # centroid (-2,-2): equidistant -> lower row first
    assert key(out[0])[3:] == (-7, -7, 0, 0) and len(out) == 1


_SCALAR_NUMPY_SCRIPT = r'''
import ctypes, json, random, sys
import numpy as np
sys.path.insert(0, %(root)r)
from watsor_b200 import _lib
lib = _lib.load()
rng = np.random.default_rng(3)
res = {'argsort_mismatch': 0, 'argsort_cases': 0, 'unstable_seen': 0}
for n in list(range(0, 110)) + [160, 100]:
    for vals in (2, 3, 7, 60, 10 ** 9):
        for _ in range(6):
            a = rng.integers(0, vals, n).astype(np.int64)
            want = np.argsort(a.astype(np.float64))
            res['unstable_seen'] += int(not np.array_equal(want, np.argsort(a, kind='stable')))
            out = (ctypes.c_int32 * max(n, 1))()
            assert lib.wb_debug_argsort(a.ctypes.data, n, out) == 0
            res['argsort_cases'] += 1
            res['argsort_mismatch'] += int(list(out[:n]) != list(want))
# organ-pipe / sawtooth patterns: deeper partition trees
for n in (64, 100):
    for a in (np.r_[np.arange(n // 2), np.arange(n // 2)[::-1]], np.arange(n) %% 5, np.zeros(n), np.arange(n)[::-1] // 3):
        a = a.astype(np.int64)
        out = (ctypes.c_int32 * n)()
        lib.wb_debug_argsort(a.ctypes.data, n, out)
        res['argsort_cases'] += 1
        res['argsort_mismatch'] += int(list(out) != list(np.argsort(a.astype(np.float64))))
# tie-heavy tracking: frame_digest() of every frame of 5 x 8 sequences, by the native tracker and -- where the original
# project is readable -- by its TrackFilter, both under this interpreter's scalar numpy
from tests.test_tracker import TIE_HEAVY, NativeTracker, frame_digest, mk
if %(with_ref)r:
    sys.path.insert(0, %(ref)r)
    from watsor.filter.track import TrackFilter
    from watsor.stream.share import BoundingBox, Detection
res['native'], res['reference'] = {}, {}
for max_n, grid in TIE_HEAVY:
    for seed in range(8):
        r = random.Random(seed)
        name = 'tie-heavy max_n=%%d grid=%%d seed=%%d' %% (max_n, grid, seed)
        nat = NativeTracker(2, 4)
        ref = TrackFilter(sensitivity=2, history=4) if %(with_ref)r else None
        res['native'][name], res['reference'][name] = [], []
        for f in range(40):
            dets = []
            for _ in range(r.randint(0, max_n)):
                x, y = r.randint(0, grid), r.randint(0, grid)
                dets.append((r.randint(1, 2), 0.5 + 0.01 * r.randint(0, 40), (x, y, x + r.choice([2, 4]), y + r.choice([2, 4])),
                             [r.randint(1, 12)] if r.random() < 0.5 else []))
            got, sa = nat([mk(*d) for d in dets])
            res['native'][name].append(frame_digest(sa, got))
            if ref is None:
                continue
            rd = []
            for l, c, b, z in dets:
                d = Detection(label=l, confidence=c, bounding_box=BoundingBox(*b))
                for i, zz in enumerate(z):
                    d.zones[i] = zz
                rd.append(d)
            exp, sa = ref(rd)
            assert isinstance(sa, bool)
            res['reference'][name].append(frame_digest(sa, exp))
print(json.dumps(res))
'''
TIE_HEAVY = ((12, 6), (24, 20), (40, 6), (40, 60), (100, 30))      # (max detections per frame, coordinate grid)


def test_argsort_and_tie_heavy_tracking_match_numpy_scalar_sort():
    """numpy_argsort() in tracker.cpp is numpy's index introsort; numpy >= 1.25 replaces it by SIMD sorting networks
    on AVX2 / AVX-512 machines, so the comparison runs in a child interpreter with those code paths disabled
    (NPY_DISABLE_CPU_FEATURES) -- the arithmetic of the reference's pinned numpy 1.23.  With it, the tie-heavy
    tracking sequences (tiny coordinate grids, up to 100 detections of a label per frame) equal the reference's
    TrackFilter on every frame (its answers recorded in tests/golden/reference/tracker.json)."""
    import json
    import subprocess
    from numpy._core._multiarray_umath import __cpu_features__ as feats
    simd = [k for k, v in feats.items() if v and (k.startswith('AVX512') or k in ('AVX2', 'FMA3'))
            and k in ('AVX2', 'FMA3', 'AVX512F', 'AVX512CD', 'AVX512_KNL', 'AVX512_KNM', 'AVX512_SKX', 'AVX512_CLX',
                      'AVX512_CNL', 'AVX512_ICL', 'AVX512_SPR')]
    env = dict(os.environ)
    if simd:
        env['NPY_DISABLE_CPU_FEATURES'] = ' '.join(simd)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    script = _SCALAR_NUMPY_SCRIPT % {'root': root, 'ref': REF, 'with_ref': bool(REF)}
    p = subprocess.run([sys.executable, '-c', script], env=env, capture_output=True, text=True, timeout=300)
    if p.returncode != 0 and 'NPY_DISABLE_CPU_FEATURES' in p.stderr:
        pytest.skip('numpy refused to disable its SIMD dispatch: ' + p.stderr.strip().splitlines()[-1])
    assert p.returncode == 0, p.stderr[-2000:]
    res = json.loads(p.stdout.strip().splitlines()[-1])
    assert res['unstable_seen'] > 0                              # the cases do exercise non-stable orders
    assert res['argsort_mismatch'] == 0, res
    assert len(res['native']) == 5 * 8
    for name, ours in res['native'].items():
        theirs = recorded(name, lambda: res['reference'][name])
        assert len(ours) == len(theirs) == 40, name
        diverging = [f for f, (a, b) in enumerate(zip(ours, theirs)) if a != b]
        assert not diverging, (name, 'first diverging frame', diverging[0])
