"""Small tables and containers the filters and the frame ABI depend on, against the reference modules imported
from the read-only tree: the COCO label table (watsor/config/coco.py:14-131) and the Frame / FrameBuffer views
(watsor/stream/share.py:37-113).  CPU only; the reference's answers are recorded in tests/golden/reference/tables.json
(tests/reference_outputs.py)."""
import ctypes
import sys

import numpy as np
import pytest

from tests.reference_outputs import REFERENCE, Recorded

recorded = Recorded('tables')


@pytest.fixture(scope='module')
def ref_modules():
    if not REFERENCE:
        yield None, None
        return
    sys.path.insert(0, REFERENCE)
    try:
        import watsor.config.coco as coco
        import watsor.stream.share as share
        yield coco, share
    finally:
        sys.path.remove(REFERENCE)


def _coco_class(ref_coco, idx):
    try:
        return {'label': ref_coco.get_coco_class(idx).label}
    except Exception as e:
        return {'raises': type(e).__name__}


def test_coco_table_equals_reference(ref_modules):
    ref_coco, _ = ref_modules
    from watsor_b200.config import coco
    assert coco.COCO_CLASSES == recorded('COCO_CLASSES', lambda: list(ref_coco.COCO_CLASSES))
    for idx in list(range(-3, 95)) + [1000]:
        theirs = recorded('get_coco_class(%d)' % idx, lambda: _coco_class(ref_coco, idx))
        if 'raises' in theirs:                                  # whatever the reference does out of range ...
            with pytest.raises(Exception) as e:                  # ... we do the same
                coco.get_coco_class(idx)
            assert type(e.value).__name__ == theirs['raises'], idx
            continue
        # the reference record also carries drawing attributes (colours, font) of the out-of-scope output stage
        assert coco.get_coco_class(idx).label == theirs['label'], idx


def _frame_view(ref_share, w, h):
    theirs = ref_share.Frame(w, h, 3, 'B')
    st, it = theirs.get_numpy_image(np.uint8)
    return {'shape': list(st), 'array_shape': list(it.shape), 'dtype': str(it.dtype),
            'header_size': ctypes.sizeof(theirs.header.get_obj()),
            'header': [theirs.header.width, theirs.header.height, theirs.header.channels]}


def test_frame_views_equal_reference(ref_modules):
    _, ref_share = ref_modules
    from watsor_b200.stream import share
    for w, h in ((64, 48), (1, 1), (320, 240)):
        ours = share.Frame(w, h)
        theirs = recorded('Frame(%d, %d)' % (w, h), lambda: _frame_view(ref_share, w, h))
        so, io = ours.get_numpy_image(np.uint8)
        assert list(so) == theirs['shape'] == [h, w, 3]
        assert list(io.shape) == theirs['array_shape'] and str(io.dtype) == theirs['dtype']
        assert ctypes.sizeof(ours.header.get_obj()) == theirs['header_size'] == 7224
        assert [ours.header.width, ours.header.height, ours.header.channels] == theirs['header']
        io[...] = 7
        ours.header.detections[99].label = 5
        ours.clear()
        assert not io.any() and ours.header.detections[99].label == 0
    fb_o = share.FrameBuffer(3, 32, 16)
    assert len(fb_o.frames) == recorded('len(FrameBuffer(3, 32, 16).frames)',
                                        lambda: len(ref_share.FrameBuffer(3, 32, 16).frames)) == 3
