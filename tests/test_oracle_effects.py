"""oracle/effects.py against the reference's OWN effect classes (watsor/output/{copy,blend,draw}.py), imported from the
read-only tree and run here on the same frames and Detection rows (SURVEY.md 8c: "outputs of the reference itself run
here").  draw.py imports watsor.filter.mask, which imports shapely (absent): a bare stand-in module satisfies the
import -- the effects never touch it.  CPU only; the reference's frames are recorded (as digests) in
tests/golden/reference/effects.json (tests/reference_outputs.py)."""
import os
import sys
import types
from tempfile import TemporaryDirectory

import cv2
import numpy as np
import pytest

from oracle import effects as oracle_fx
from tests.fx_cases import random_alpha, random_rows

from tests.reference_outputs import REFERENCE as REF  # noqa: E402
from tests.reference_outputs import Recorded, canon  # noqa: E402

recorded = Recorded('effects')


@pytest.fixture(scope='module')
def ref():
    if not REF:
        yield None
        return
    saved = {k: sys.modules.get(k) for k in ('shapely', 'shapely.geometry')}
    shapely, geometry = types.ModuleType('shapely'), types.ModuleType('shapely.geometry')
    geometry.Polygon = object
    shapely.geometry = geometry
    sys.modules['shapely'], sys.modules['shapely.geometry'] = shapely, geometry
    sys.path.insert(0, REF)
    try:
        from watsor.output.blend import BlendEffect
        from watsor.output.copy import CopyImageEffect
        from watsor.output.draw import DrawEffect, DrawEffectWithContours
        from watsor.stream.share import Detection
        yield types.SimpleNamespace(BlendEffect=BlendEffect, CopyImageEffect=CopyImageEffect, DrawEffect=DrawEffect,
                                    DrawEffectWithContours=DrawEffectWithContours, Detection=Detection)
    finally:
        sys.path.remove(REF)
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


def as_header(ref, rows):
    """The reference reads `header_out.detections`; its Detection struct has our layout (tests/test_abi.py)."""
    theirs = (ref.Detection * len(rows)).from_buffer_copy(bytes(rows))
    return types.SimpleNamespace(detections=theirs)


@pytest.mark.parametrize('size', [(320, 240), (640, 480), (97, 61)])
def test_copy_and_draw_chain(ref, size):
    w, h = size
    rng = np.random.default_rng(w + 1)
    for n_drawn in (0, 5, 30):
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        rows = random_rows(rng, w, h, n_drawn)
        theirs = recorded('copy+draw %dx%d %d' % (w, h, n_drawn), lambda: copy_and_draw(ref, img, rows))
        ours = oracle_fx.effect_chain(img, rows)
        assert canon(ours) == theirs, (size, n_drawn)


def copy_and_draw(ref, img, rows):
    header = as_header(ref, rows)
    theirs = np.zeros_like(img)
    ref.CopyImageEffect().apply(img, theirs, img.shape, header, header)
    ref.DrawEffect().apply(img, theirs, img.shape, header, header)
    return theirs


def blend_and_draw_with_contours(ref, config, img, rows):
    """[after BlendEffect, after DrawEffectWithContours as well]."""
    header = as_header(ref, rows)
    theirs = np.zeros_like(img)
    ref.BlendEffect(config).apply(img, theirs, img.shape, header, header)
    blended = theirs.copy()
    ref.DrawEffectWithContours(config).apply(img, theirs, img.shape, header, header)
    return [blended, theirs]


@pytest.mark.parametrize('size', [(320, 240), (200, 150)])
def test_blend_and_draw_with_contours_chain(ref, size):
    w, h = size
    rng = np.random.default_rng(h + 1)
    with TemporaryDirectory() as tmp:
        for nz in (1, 2, 4):
            alpha = random_alpha(rng, w, h, nz)
            rgba = np.dstack([rng.integers(0, 256, (h, w, 3), dtype=np.uint8), alpha])
            path = os.path.join(tmp, 'mask%d.png' % nz)
            assert cv2.imwrite(path, rgba)
            config = {'mask': path, 'width': w, 'height': h}
            img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
            rows = random_rows(rng, w, h, 12, n_zones=nz)
            blended, theirs = recorded('blend+contours %dx%d %d' % (w, h, nz),
                                       lambda: blend_and_draw_with_contours(ref, config, img, rows))
            assert canon(oracle_fx.effect_chain(img, rows, alpha, do_draw=False)) == blended, nz
            assert canon(oracle_fx.effect_chain(img, rows, alpha)) == theirs, nz


def test_reference_draw_test_case(ref):
    """watsor/test/test_output.py:33-50: a 2x2 frame; the oracle must survive (and equal) the degenerate geometry."""
    rows = random_rows(np.random.default_rng(0), 2, 2, 2)
    img = np.zeros((2, 2, 3), np.uint8)
    theirs = recorded('draw 2x2', lambda: draw_on_copy(ref, img, rows))
    assert canon(oracle_fx.effect_chain(img, rows)) == theirs


def draw_on_copy(ref, img, rows):
    header = as_header(ref, rows)
    theirs = img.copy()
    ref.DrawEffect().apply(img, theirs, img.shape, header, header)
    return theirs
