"""The write loop of the reference detector (watsor/detection/tensorflow_cpu.py:74-92) run here, as it is, against
the oracle's `to_detections` (SURVEY.md 8a row a2).  TensorFlow is not installed, so the class is imported with an
empty stand-in `tensorflow` module and instantiated without `__init__`; only `detect()` runs, with the arrays a
`sess.run` would return supplied by the test.  Two readings of `int(np.float32 * int)`:
  * legacy promotion (numpy 1.23, the reference's pin, docker/Dockerfile.base:33): the product is a float64, i.e.
    exact -- reproduced on any numpy by handing the loop float64 copies of the float32 boxes;
  * NEP 50 (numpy >= 2): the product is rounded to float32 first; it differs from the exact reading only where that
    rounding lands on an integer -- counted here, and every such case is checked to be exactly that.
CPU only; the rows the reference loop wrote are recorded in tests/golden/reference/detect_loop.json
(tests/reference_outputs.py)."""
import sys
import types

import numpy as np
import pytest

from oracle.ssd_graph import to_detections
from tests.reference_outputs import REFERENCE, Recorded, canon

recorded = Recorded('detect_loop')


@pytest.fixture(scope='module')
def ref():
    if not REFERENCE:
        yield None
        return
    saved = sys.modules.get('tensorflow')
    sys.modules['tensorflow'] = types.ModuleType('tensorflow')
    sys.path.insert(0, REFERENCE)
    try:
        from watsor.detection.tensorflow_cpu import TensorFlowObjectDetector
        from watsor.stream.share import Detection
        yield types.SimpleNamespace(Detector=TensorFlowObjectDetector, Detection=Detection)
    finally:
        sys.path.remove(REFERENCE)
        if saved is None:
            sys.modules.pop('tensorflow', None)
        else:
            sys.modules['tensorflow'] = saved


def run_reference_loop(ref, boxes, classes, scores, shape, n_rows=100):
    det = object.__new__(ref.Detector)
    setattr(det, '_TensorFlowObjectDetector__detect_fn', lambda image: (boxes, classes, scores))
    rows = (ref.Detection * n_rows)()
    ms = det.detect(shape, None, rows)
    assert ms >= 0.0
    return [(r.label, r.confidence, r.bounding_box.x_min, r.bounding_box.y_min, r.bounding_box.x_max,
             r.bounding_box.y_max) for r in rows]


def as_array(rows):
    """(label, confidence, x_min, y_min, x_max, y_max) rows as float64: every field exact, so equal arrays are equal
    rows."""
    return np.array(rows, np.float64).reshape(-1, 6)


def random_outputs(rng, n=100):
    boxes = rng.random((n, 4)).astype(np.float32)
    boxes[::7] = np.float32(1.0)                               # clipped to the window edge
    boxes[1::7] = np.float32(0.0)
    boxes[2::11, 2:] = np.nextafter(np.float32(1.0), np.float32(0.0))
    k = int(rng.integers(0, n))
    boxes[k:] = 0.0                                             # PadOrClipBoxList padding
    scores = np.sort(rng.random(n).astype(np.float32))[::-1].copy()
    scores[k:] = 0.0
    classes = rng.integers(1, 4, n).astype(np.float32)
    classes[k:] = 1.0                                           # padded rows: 0 + 1
    return boxes, classes, scores


@pytest.mark.parametrize('shape', [(480, 640, 3), (240, 320, 3), (1080, 1920, 3), (2, 2, 3), (1, 1, 3)])
def test_oracle_equals_reference_loop_under_legacy_promotion(ref, shape):
    rng = np.random.default_rng(shape[0])
    cases = [random_outputs(rng) for _ in range(40)]
    got = recorded('legacy %r' % (shape,), lambda: [
        as_array(run_reference_loop(ref, b.astype(np.float64), c, s, shape)) for b, c, s in cases])
    assert got == canon([as_array(to_detections(b, c, s, shape)) for b, c, s in cases])


def test_short_outputs_leave_the_remaining_rows_untouched(ref):
    rng = np.random.default_rng(1)
    boxes, classes, scores = random_outputs(rng, 7)
    got = recorded('short', lambda: as_array(run_reference_loop(ref, boxes.astype(np.float64), classes, scores,
                                                                (480, 640, 3))))
    # share.py:47-50 zeros stay
    want = np.concatenate([as_array(to_detections(boxes, classes, scores, (480, 640, 3))), np.zeros((93, 6))])
    assert got == canon(want)


def test_nep50_reading_differs_only_on_float32_rounding_to_an_integer(ref):
    if int(np.__version__.split('.')[0]) < 2:
        pytest.skip('NEP 50 promotion needs numpy >= 2')
    rng = np.random.default_rng(7)
    shape = (1080, 1920, 3)
    cases = [random_outputs(rng) for _ in range(200)]
    # the float32 boxes as they are, i.e. the NEP 50 reading: the rows, and where they differ from the exact reading
    # (float64 copies of the boxes), by (case, row, box column) -> the NEP 50 value
    theirs = recorded('nep50', lambda: nep50_reading(ref, cases, shape))
    diffs = {tuple(k): v for k, v in theirs['differing']}
    differing = total = 0
    for t, (boxes, classes, scores) in enumerate(cases):
        exact = to_detections(boxes, classes, scores, shape)
        assert canon(as_array(exact)) == theirs['legacy'][t]
        for d, b in enumerate(exact):
            for j, vb in enumerate(b[2:]):
                total += 1
                va = diffs.pop((t, d, j), vb)
                if va != vb:
                    differing += 1
                    col = (1, 0, 3, 2)[j]                       # x_min,y_min,x_max,y_max <- boxes[:, 1,0,3,2]
                    mx = (shape[1] - 1) if j % 2 == 0 else (shape[0] - 1)
                    p32 = np.float32(boxes[d][col]) * np.float32(mx)
                    assert va == vb + 1 and float(p32) == float(va), (d, j, boxes[d][col])
    assert not diffs and differing == len(theirs['differing'])
    assert differing < total * 1e-3


def nep50_reading(ref, cases, shape):
    legacy, differing = [], []
    for t, (boxes, classes, scores) in enumerate(cases):
        new = run_reference_loop(ref, boxes, classes, scores, shape)
        old = run_reference_loop(ref, boxes.astype(np.float64), classes, scores, shape)
        legacy.append(as_array(old))
        for d, (a, b) in enumerate(zip(new, old)):
            assert a[:2] == b[:2]
            differing += [[[t, d, j], va] for j, (va, vb) in enumerate(zip(a[2:], b[2:])) if va != vb]
    return {'legacy': legacy, 'differing': differing}
