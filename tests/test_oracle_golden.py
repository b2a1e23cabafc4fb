"""The oracle against the committed golden vectors, and the two oracle forms against each other."""
import hashlib
import os

import numpy as np
import pytest

from tests.artist import artist_frame
from tests.conftest import REF_PB, load_golden_frame


def test_artist_recipe_reproduces_committed_frames(golden):
    for case in golden['cases']:
        img = artist_frame(case['width'], case['height'], case['cam'], case['frame'])
        assert hashlib.md5(img.tobytes()).hexdigest() == case['frame_md5'], case['name']
        assert np.array_equal(img, load_golden_frame(case['name']))


def test_blob_oracle_reproduces_golden_vectors(golden, real_shapes_oracle):
    from oracle.ssd_graph import to_detections
    for case in golden['cases']:
        img = load_golden_frame(case['name'])
        pre = real_shapes_oracle.preprocess(img)
        assert hashlib.md5(pre.tobytes()).hexdigest() == case['pre_md5']      # pure numpy: bit exact
        b, s, cl, n = real_shapes_oracle.postprocess(*real_shapes_oracle.raw_heads(pre))
        assert n == case['num'] and [int(x) for x in cl[:n]] == case['classes']
        want_b = np.frombuffer(bytes.fromhex(case['boxes_f32']), '<f4').reshape(-1, 4)
        want_s = np.frombuffer(bytes.fromhex(case['scores_f32']), '<f4')
        assert np.allclose(b[:n], want_b, atol=2e-6) and np.allclose(s[:n], want_s, atol=2e-6)
        rows = to_detections(b, cl, s, img.shape)
        assert [list(r[:1]) + list(r[2:]) for r in rows[:n]] == [r[:1] + r[2:] for r in case['rows']]
        # rows past num are the graph's zero padding with class 0 + 1 (SURVEY.md A.6)
        assert rows[n] == (1, 0.0, 0, 0, 0, 0) and rows[99] == (1, 0.0, 0, 0, 0, 0)


def test_oracle_finds_the_drawn_shapes(real_shapes_oracle):
    """The reference's behavioural pin (test_detect.py:28-77): on 100x100 Artist frames the
    detector reports labelled shapes with confidence >= 0.5; here additionally the right
    class at the right place."""
    hits = total = 0
    for frame in range(6):
        img, truth = artist_frame(100, 100, 5, frame, with_truth=True)
        b, cl, s, n = real_shapes_oracle.run(img)
        from oracle.ssd_graph import to_detections
        rows = [r for r in to_detections(b, cl, s, img.shape)[:n] if r[1] >= 0.5]
        for shape, (x0, y0, x1, y1) in truth:
            total += 1
            for (label, conf, bx0, by0, bx1, by1) in rows:
                if label == shape and abs(bx0 - x0) <= 4 and abs(by0 - y0) <= 4 and abs(bx1 - x1) <= 4 \
                        and abs(by1 - y1) <= 4:
                    hits += 1
                    break
    assert hits >= 0.7 * total, (hits, total)


@pytest.mark.skipif(not os.path.isfile(REF_PB), reason='oracle/_ref/cpu.pb not built')
def test_graph_oracle_and_blob_oracle_agree_bit_for_bit(real_shapes_oracle):
    from oracle.ssd_graph import SsdGraphOracle
    og = SsdGraphOracle(REF_PB)
    img = np.random.default_rng(3).integers(0, 256, (240, 320, 3), dtype=np.uint8)
    pre = og.preprocess(img)
    assert np.array_equal(pre, real_shapes_oracle.preprocess(img))
    e1, l1 = og.raw_heads(pre)
    e2, l2 = real_shapes_oracle.raw_heads(pre)
    assert np.array_equal(e1, e2) and np.array_equal(l1, l2)
    for a, b in zip(og.postprocess(e1, l1), real_shapes_oracle.postprocess(e2, l2)):
        assert np.array_equal(a, b)


def test_golden_porch_verdicts(golden):
    from oracle.filters import AreaOracle, ConfidenceOracle, Det, MaskOracle, apply_predicates
    from tests.conftest import PORCH_CONFIG
    filters = [ConfidenceOracle(PORCH_CONFIG), AreaOracle(PORCH_CONFIG), MaskOracle(PORCH_CONFIG)]
    for case in golden['cases']:
        if 'porch_verdicts' not in case:
            continue
        dets = [Det(r[0], r[1], tuple(r[2:])) for r in case['rows']]
        _, verdicts = apply_predicates(dets, filters)
        assert verdicts == case['porch_verdicts'] and [d.zones for d in dets] == case['porch_zones']
