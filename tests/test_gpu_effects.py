"""GPU visual effects (wb_fx_*, watsor_b200/output/effects.py) against the oracle = the reference's numpy / OpenCV
arithmetic (oracle/effects.py, pinned to the reference's own classes in tests/test_oracle_effects.py).  Every output
byte must be equal."""
import os
from tempfile import TemporaryDirectory

import cv2
import numpy as np
import pytest

from oracle import effects as oracle_fx
from tests.fx_cases import random_alpha, random_rows

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def engine():
    from watsor_b200.output.effects import EffectsEngine
    with EffectsEngine(0) as e:
        yield e


def header_of(rows):
    import types
    return types.SimpleNamespace(detections=rows)


@pytest.mark.parametrize('size', [(640, 480), (320, 240), (97, 61), (1920, 1080)])
def test_copy_and_draw_equal_opencv(engine, size):
    from watsor_b200.output.effects import WB_FX_DRAW
    w, h = size
    rng = np.random.default_rng(w)
    cam = engine.add_camera(w, h)
    for n_drawn in (0, 4, 25, 100):
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        rows = random_rows(rng, w, h, n_drawn)
        out = np.zeros_like(img)
        engine.render([img], [out], [cam], [rows], WB_FX_DRAW)
        ref = oracle_fx.effect_chain(img, rows)
        assert np.array_equal(ref, out), (size, n_drawn, int((ref != out).sum()))


@pytest.mark.parametrize('size', [(640, 480), (200, 150)])
def test_blend_draw_and_zone_outlines_equal_opencv(engine, size):
    from watsor_b200.output.effects import WB_FX_BLEND, WB_FX_CONTOURS, WB_FX_DRAW, contour_bits
    w, h = size
    rng = np.random.default_rng(h)
    for nz in (1, 3, 5):
        alpha = random_alpha(rng, w, h, nz)
        cam = engine.add_camera(w, h, alpha, contour_bits(alpha))
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        rows = random_rows(rng, w, h, 15, n_zones=nz)
        out = np.zeros_like(img)
        engine.render([img], [out], [cam], [rows], WB_FX_BLEND)
        assert np.array_equal(oracle_fx.effect_chain(img, rows, alpha, do_draw=False), out), ('blend', size, nz)
        engine.render([img], [out], [cam], [rows], WB_FX_BLEND | WB_FX_DRAW | WB_FX_CONTOURS)
        ref = oracle_fx.effect_chain(img, rows, alpha)
        assert np.array_equal(ref, out), (size, nz, int((ref != out).sum()))


def test_reference_shaped_classes_and_the_fused_chain(engine):
    """The drop-in classes with the reference's constructors / apply() contract (main.py:302-312)."""
    from watsor_b200.output.effects import (BlendEffect, CopyImageEffect, DrawEffect, DrawEffectWithContours,
                                            FusedEffects)
    w, h = 320, 240
    rng = np.random.default_rng(5)
    with TemporaryDirectory() as tmp:
        alpha = random_alpha(rng, w, h, 3)
        path = os.path.join(tmp, 'mask.png')
        assert cv2.imwrite(path, np.dstack([np.zeros((h, w, 3), np.uint8), alpha]))
        masked = {'mask': path, 'width': w, 'height': h}
        plain = {'width': w, 'height': h}
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        rows = random_rows(rng, w, h, 10, n_zones=3)
        hdr = header_of(rows)
        # with a mask: BlendEffect, then DrawEffectWithContours on image_out
        out = np.zeros_like(img)
        BlendEffect(masked, engine).apply(img, out, img.shape, hdr, hdr)
        DrawEffectWithContours(masked, engine).apply(img, out, img.shape, hdr, hdr)
        ref = oracle_fx.effect_chain(img, rows, alpha)
        assert np.array_equal(ref, out)
        fused = np.zeros_like(img)
        FusedEffects(masked, engine).apply(img, fused, img.shape, hdr, hdr)
        assert np.array_equal(ref, fused)
        # without: CopyImageEffect, then DrawEffect
        out = np.zeros_like(img)
        CopyImageEffect().apply(img, out, img.shape, hdr, hdr)
        DrawEffect(engine).apply(img, out, img.shape, hdr, hdr)
        ref = oracle_fx.effect_chain(img, rows)
        assert np.array_equal(ref, out)
        fused = np.zeros_like(img)
        FusedEffects(plain, engine).apply(img, fused, img.shape, hdr, hdr)
        assert np.array_equal(ref, fused)


def test_batch_of_cameras_and_device_pointers(engine):
    import torch

    from watsor_b200.output.effects import WB_FX_BLEND, WB_FX_CONTOURS, WB_FX_DRAW, WB_FX_ON_DEVICE, contour_bits
    rng = np.random.default_rng(9)
    sizes = [(640, 480), (320, 240), (640, 480), (97, 61)]
    cams, alphas, imgs, rows = [], [], [], []
    for i, (w, h) in enumerate(sizes):
        alpha = random_alpha(rng, w, h, 2) if i % 2 == 0 else None
        cams.append(engine.add_camera(w, h, alpha, None if alpha is None else contour_bits(alpha)))
        alphas.append(alpha)
        imgs.append(rng.integers(0, 256, (h, w, 3), dtype=np.uint8))
        rows.append(random_rows(rng, w, h, 8, n_zones=2 if alpha is not None else 0))
    flags = WB_FX_BLEND | WB_FX_DRAW | WB_FX_CONTOURS
    outs = [np.zeros_like(i) for i in imgs]
    engine.render(imgs, outs, cams, rows, flags)
    refs = [oracle_fx.effect_chain(i, r, a) for i, r, a in zip(imgs, rows, alphas)]
    for k in range(len(sizes)):
        assert np.array_equal(refs[k], outs[k]), k
    # the same batch with frames resident on the device
    d_in = [torch.from_numpy(i).cuda() for i in imgs]
    d_out = [torch.zeros_like(t) for t in d_in]
    torch.cuda.synchronize()
    engine.render([t.data_ptr() for t in d_in], [t.data_ptr() for t in d_out], cams, rows, flags | WB_FX_ON_DEVICE)
    for k in range(len(sizes)):
        assert np.array_equal(refs[k], d_out[k].cpu().numpy()), k


def test_errors_are_loud(engine):
    from watsor_b200 import _lib
    from watsor_b200.output.effects import WB_FX_BLEND, WB_FX_DRAW
    img = np.zeros((20, 20, 3), np.uint8)
    rows = random_rows(np.random.default_rng(0), 20, 20, 1)
    with pytest.raises(_lib.WatsorB200Error, match='not been configured'):
        engine.render([img], [img.copy()], [12345], [rows], WB_FX_DRAW)
    cam = engine.add_camera(20, 20)
    with pytest.raises(_lib.WatsorB200Error, match='at least 43 rows'):
        engine.render([img], [img.copy()], [cam], [rows], WB_FX_DRAW)
    out = np.ones_like(img)
    engine.render([img], [out], [cam], [rows], WB_FX_BLEND)          # no alpha channel: a copy
    assert np.array_equal(out, img)


def test_equal_to_the_reference_classes_installed_under_baseline_ref(engine):
    """The UNMODIFIED reference package (oracle/_ref/site, copied by __graft_entry__.build() from a readable checkout)
    provides watsor.output.{blend,draw,copy}: run the reference's own effect chain on the CPU and the fused GPU effect
    on the same frame and rows.  watsor.filter.mask imports shapely (absent): an empty stand-in satisfies the import."""
    import sys
    import types

    from tests.conftest import ROOT
    from watsor_b200.output.effects import FusedEffects
    ref_root = os.path.join(ROOT, 'oracle', '_ref', 'site')
    if not os.path.isfile(os.path.join(ref_root, 'watsor', 'output', 'draw.py')):
        pytest.skip('oracle/_ref/site not installed')
    saved = {k: v for k, v in sys.modules.items() if k == 'shapely' or k.startswith('shapely.') or
             k == 'watsor' or k.startswith('watsor.')}
    for k in saved:
        del sys.modules[k]
    shapely, geometry = types.ModuleType('shapely'), types.ModuleType('shapely.geometry')
    geometry.Polygon = object
    shapely.geometry = geometry
    sys.modules['shapely'], sys.modules['shapely.geometry'] = shapely, geometry
    sys.path.insert(0, ref_root)
    try:
        from watsor.output.blend import BlendEffect as RefBlend
        from watsor.output.copy import CopyImageEffect as RefCopy
        from watsor.output.draw import DrawEffect as RefDraw
        from watsor.output.draw import DrawEffectWithContours as RefDrawContours
        from watsor.stream.share import Detection as RefDetection
        w, h = 640, 480
        rng = np.random.default_rng(21)
        with TemporaryDirectory() as tmp:
            alpha = random_alpha(rng, w, h, 4)
            path = os.path.join(tmp, 'mask.png')
            assert cv2.imwrite(path, np.dstack([np.zeros((h, w, 3), np.uint8), alpha]))
            for config in ({'mask': path, 'width': w, 'height': h}, {'width': w, 'height': h}):
                img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
                rows = random_rows(rng, w, h, 20, n_zones=4 if 'mask' in config else 0)
                theirs_hdr = types.SimpleNamespace(
                    detections=(RefDetection * len(rows)).from_buffer_copy(bytes(rows)))
                theirs = np.zeros_like(img)
                if 'mask' in config:
                    RefBlend(config).apply(img, theirs, img.shape, theirs_hdr, theirs_hdr)
                    RefDrawContours(config).apply(img, theirs, img.shape, theirs_hdr, theirs_hdr)
                else:
                    RefCopy().apply(img, theirs, img.shape, theirs_hdr, theirs_hdr)
                    RefDraw().apply(img, theirs, img.shape, theirs_hdr, theirs_hdr)
                ours = np.zeros_like(img)
                hdr = header_of(rows)
                FusedEffects(config, engine).apply(img, ours, img.shape, hdr, hdr)
                assert np.array_equal(theirs, ours), ('mask' in config, int((theirs != ours).sum()))
    finally:
        sys.path.remove(ref_root)
        for k in [k for k in sys.modules if k == 'shapely' or k.startswith('shapely.') or k == 'watsor' or
                  k.startswith('watsor.')]:
            del sys.modules[k]
        sys.modules.update(saved)
