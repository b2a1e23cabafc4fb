"""The oracle's predicates against the reference's OWN filter classes, imported from the read-only tree and run here
(SURVEY.md 8c: "outputs of the reference itself run here").  ConfidenceFilter and AreaFilter are pure Python and run
as they are.  MaskFilter needs shapely, which is not installed: it is imported with a stand-in `shapely.geometry`
whose `Polygon.intersects` is the oracle's exact integer geometry, so this pins the reference's control flow --
alpha threshold, contour extraction and ordering, per-class zone lists, the order and cap of `zones[]` writes --
but not GEOS itself (that gap is stated in DESIGN.md section 5).  CPU only; the reference's verdicts are recorded in
tests/golden/reference/filters.json (tests/reference_outputs.py)."""
import os
import sys
import types
from tempfile import NamedTemporaryFile

import numpy as np
import pytest

from oracle.filters import AreaOracle, ConfidenceOracle, Det, MaskOracle, rect_intersects_polygon
from tests.conftest import PORCH_CONFIG
from tests.reference_outputs import REFERENCE, Recorded

recorded = Recorded('filters')


class _StandInPolygon:
    """shapely.geometry.Polygon as far as mask.py uses it (mask.py:26,45-54)."""

    def __init__(self, points):
        self.points = np.asarray(points, dtype=np.int64).reshape(-1, 2)
        if len(self.points) < 3:
            raise ValueError('A linearring requires at least 4 coordinates.')

    def intersects(self, other):
        # self is the detection's box (4 corners, mask.py:45-48), other a zone polygon
        xs, ys = self.points[:, 0], self.points[:, 1]
        return bool(rect_intersects_polygon(int(xs[0]), int(ys[0]), int(xs[2]), int(ys[2]), other.points))


@pytest.fixture(scope='module')
def ref():
    if not REFERENCE:
        yield None
        return
    saved = {k: sys.modules.get(k) for k in ('shapely', 'shapely.geometry')}
    shapely = types.ModuleType('shapely')
    geometry = types.ModuleType('shapely.geometry')
    geometry.Polygon = _StandInPolygon
    shapely.geometry = geometry
    sys.modules['shapely'], sys.modules['shapely.geometry'] = shapely, geometry
    sys.path.insert(0, REFERENCE)
    try:
        from watsor.filter.area import AreaFilter
        from watsor.filter.confidence import ConfidenceFilter
        from watsor.filter.mask import MaskFilter
        from watsor.stream.share import BoundingBox, Detection
        yield types.SimpleNamespace(AreaFilter=AreaFilter, ConfidenceFilter=ConfidenceFilter, MaskFilter=MaskFilter,
                                    BoundingBox=BoundingBox, Detection=Detection)
    finally:
        sys.path.remove(REFERENCE)
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


def random_dets(rng, w, h, n):
    out = []
    for r in range(n):
        x0, x1 = (int(v) for v in rng.integers(-5, w + 5, 2))
        y0, y1 = (int(v) for v in rng.integers(-5, h + 5, 2))
        if r % 3:
            x0, x1, y0, y1 = min(x0, x1), max(x0, x1), min(y0, y1), max(y0, y1)
        if r % 7 == 0:
            x1, y1 = x0, y0
        label = int(rng.integers(0, 6))
        conf = [0.5, 0.25, 0.75, float(np.float32(rng.random())), float(rng.random())][r % 5]
        out.append(Det(label, conf, (x0, y0, x1, y1)))
    return out


def verdicts(ref, filt, dets):
    """The reference filter `filt` on each Det: one character per verdict ('T' / 'F', both bools) and the zones it
    wrote, by index and without trailing zeros, where any are non-zero."""
    marks, zones = [], {}
    for i, d in enumerate(dets):
        rd = ref.Detection(label=d.label, confidence=d.confidence,
                           bounding_box=ref.BoundingBox(d.x_min, d.y_min, d.x_max, d.y_max))
        v = filt(rd)
        assert isinstance(v, bool)
        marks.append('T' if v else 'F')
        z = list(rd.zones)
        while z and z[-1] == 0:
            z.pop()
        if z:
            zones[str(i)] = ','.join(map(str, z))
    return {'verdicts': ''.join(marks), 'zones': zones}


def unpack(rec):
    """[(verdict, zones)] per Det from what `verdicts` recorded."""
    out = []
    for i, m in enumerate(rec['verdicts']):
        z = [int(v) for v in rec['zones'][str(i)].split(',')] if str(i) in rec['zones'] else []
        out.append((m == 'T', z + [0] * (10 - len(z))))
    return out


@pytest.mark.parametrize('seed', range(4))
def test_confidence_and_area_oracles_equal_the_reference_classes(ref, seed):
    rng = np.random.default_rng(seed)
    w, h = int(rng.integers(40, 2000)), int(rng.integers(40, 1200))
    cfg = {'width': w, 'height': h,
           'detect': [{'person': {'confidence': int(rng.integers(0, 101)), 'area': int(rng.integers(0, 101))}},
                      {'car': {'confidence': 50, 'area': 10}},
                      {'bicycle': {'confidence': 25, 'area': 0}},
                      {'motorcycle': {'confidence': 75, 'area': 100}}]}
    oc, oa = ConfidenceOracle(cfg), AreaOracle(cfg)
    # the last one is the full-frame box, exactly 100 % (area.py:18, :24-26)
    dets = random_dets(rng, w, h, 1500) + [Det(4, 0.75, (0, 0, w - 1, h - 1))]
    rc = unpack(recorded('confidence/%d' % seed, lambda: verdicts(ref, ref.ConfidenceFilter(cfg), dets)))
    ra = unpack(recorded('area/%d' % seed, lambda: verdicts(ref, ref.AreaFilter(cfg), dets)))
    assert len(rc) == len(ra) == len(dets)
    for od, (c, _), (a, _) in zip(dets, rc, ra):
        assert c == oc(od) and a == oa(od), od.key()
    assert ra[-1][0] is True and oa(dets[-1]) is True and rc[-1][0] is True and oc(dets[-1]) is True


def _random_alpha(rng, w, h):
    import cv2
    alpha = np.full((h, w), 216, np.uint8)
    for _ in range(int(rng.integers(1, 7))):
        x, y = int(rng.integers(0, w - 8)), int(rng.integers(0, h - 8))
        a, b = int(rng.integers(4, max(5, w // 3))), int(rng.integers(4, max(5, h // 3)))
        if rng.random() < 0.5:
            cv2.rectangle(alpha, (x, y), (min(w - 1, x + a), min(h - 1, y + b)), 255, -1)
        else:
            cv2.ellipse(alpha, (x + a // 2, y + b // 2), (a // 2 + 2, b // 2 + 2), 0, 0, 360, 255, -1)
    if rng.random() < 0.5:                                      # a hole: RETR_EXTERNAL ignores it
        cv2.circle(alpha, (w // 2, h // 2), min(w, h) // 10, 200, -1)
    return alpha


@pytest.mark.parametrize('seed', range(8))
def test_mask_oracle_equals_reference_control_flow(ref, seed):
    import cv2
    rng = np.random.default_rng(50 + seed)
    w, h = int(rng.integers(60, 260)), int(rng.integers(60, 200))
    rgba = np.zeros((h, w, 4), np.uint8)
    rgba[..., 3] = _random_alpha(rng, w, h)
    tmp = NamedTemporaryFile(suffix='.png', delete=False)
    try:
        cv2.imwrite(tmp.name, rgba)
        base = {'width': w, 'height': h, 'mask': tmp.name, 'detect': [{'person': {'zones': []}}]}
        try:
            n_zones = len(MaskOracle(base).polygons)
        except (AssertionError, ZeroDivisionError):
            # the reference rejects the same masks
            assert recorded('mask/%d/rejects' % seed, lambda: raised(ref.MaskFilter, base)) in \
                ('ValueError', 'ZeroDivisionError')
            return
        zones_b = sorted(int(z) for z in rng.choice(np.arange(1, n_zones + 1), size=int(rng.integers(1, n_zones + 1)),
                                                    replace=False))
        cfg = {'width': w, 'height': h, 'mask': tmp.name,
               'detect': [{'person': {'zones': []}}, {'bicycle': {'zones': zones_b}}, {'car': {'zones': [n_zones]}}]}
        om = MaskOracle(cfg)
        bad_zone = {**cfg, 'detect': [{'person': {'zones': [n_zones + 1]}}]}
        assert recorded('mask/%d/bad_zone' % seed, lambda: raised(ref.MaskFilter, bad_zone)) == 'AssertionError'
        with pytest.raises(AssertionError):
            MaskOracle(bad_zone)
        dets = random_dets(rng, w, h, 600)
        theirs = unpack(recorded('mask/%d' % seed, lambda: verdicts(ref, ref.MaskFilter(cfg), dets)))
        assert len(theirs) == len(dets)
    finally:
        tmp.close()
        os.unlink(tmp.name)
    for od, (verdict, zones) in zip(dets, theirs):
        assert verdict == om(od) and zones == od.zones, od.key()


def raised(fn, *args):
    """The name of the exception `fn(*args)` raises, None when it returns."""
    try:
        fn(*args)
    except Exception as e:
        return type(e).__name__
    return None


def test_porch_mask_reference_control_flow(ref):
    om = MaskOracle(PORCH_CONFIG)
    dets = random_dets(np.random.default_rng(3), 640, 480, 3000)
    theirs = unpack(recorded('porch', lambda: verdicts(ref, ref.MaskFilter(PORCH_CONFIG), dets)))
    assert len(theirs) == len(dets)
    hits = 0
    for od, (got, zones) in zip(dets, theirs):
        assert got == om(od) and zones == od.zones, od.key()
        hits += got
    assert 300 < hits < 2900
