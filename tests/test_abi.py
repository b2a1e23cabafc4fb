"""Host-side contract: struct ABI, the C-ABI library loads and exports what the header declares,
and the product refuses to run without a GPU instead of falling back to the CPU."""
import ctypes
import os
import re

import pytest

from tests.conftest import ROOT, has_gpu
from tests.reference_outputs import REFERENCE, Recorded, canon
from watsor_b200 import _lib
from watsor_b200.stream.share import BoundingBox, Detection, Frame, FrameBuffer, Header


def test_struct_layout_matches_reference_share_py():
    # watsor/stream/share.py:11-32 (sizes verified against the reference's ctypes in SURVEY.md 8b)
    assert ctypes.sizeof(BoundingBox) == 16
    assert ctypes.sizeof(Detection) == 72
    assert ctypes.sizeof(Header) == 7224
    assert (Detection.label.offset, Detection.zones.offset, Detection.confidence.offset,
            Detection.bounding_box.offset) == (0, 4, 48, 56)
    assert (Header.width.offset, Header.height.offset, Header.channels.offset, Header.epoch.offset,
            Header.detections.offset) == (0, 4, 8, 16, 24)


def _layout(cls):
    return [ctypes.sizeof(cls), [(f[0], getattr(cls, f[0]).offset) for f in cls._fields_]]


def _reference_layouts():
    import importlib.util
    import sys
    sys.path.insert(0, REFERENCE)
    try:
        spec = importlib.util.spec_from_file_location('ref_share', os.path.join(REFERENCE, 'watsor', 'stream', 'share.py'))
        ref = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(ref)
    finally:
        sys.path.remove(REFERENCE)
    return {name: _layout(getattr(ref, name)) for name in ('BoundingBox', 'Detection', 'Header')}


def test_struct_layout_equals_reference_module():
    theirs = Recorded('abi')('share.py struct layouts', _reference_layouts)
    for name in ('BoundingBox', 'Detection', 'Header'):
        assert canon(_layout(globals()[name])) == theirs[name], name


def test_frame_buffer_shared_memory_view():
    fb = FrameBuffer(2, 64, 48)
    frame = fb.frames[1]
    shape, img = frame.get_numpy_image('uint8')
    assert shape == (48, 64, 3) and img.shape == shape
    img[3, 5, 1] = 77
    assert frame.image.get_obj()[(3 * 64 + 5) * 3 + 1] == 77
    frame.header.detections[4].label = 9
    frame.clear()
    assert frame.header.detections[4].label == 0 and img[3, 5, 1] == 0
    assert isinstance(Frame(4, 4).header.detections[0], Detection)


def test_library_exports_every_symbol_in_header():
    header = open(os.path.join(ROOT, 'include', 'watsor_b200.h')).read()
    declared = set(re.findall(r'^(?:int|const char\*)\s+(wb_\w+)\s*\(', header, re.M))
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    lib = _lib.load()
    for name in declared:
        assert getattr(lib, name) is not None
    assert lib.wb_abi_version() == 1


def test_header_structs_match_ctypes():
    header = open(os.path.join(ROOT, 'include', 'watsor_b200.h')).read()
    assert '#define WB_MAX_DETECTIONS 100' in header and '#define WB_MAX_ZONES 10' in header
    assert ctypes.sizeof(_lib.ClassFilter) == 32


def test_no_cpu_fallback_without_gpu():
    if has_gpu():
        pytest.skip('a GPU is present')
    from watsor_b200.engine import Engine
    from watsor_b200.filter._gpu import _null_model_blob
    with pytest.raises(_lib.WatsorB200Error):
        Engine(_null_model_blob(), device=0, max_batch=1)


def test_product_never_imports_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, 'watsor_b200')):
        for f in files:
            if f.endswith(('.py', '.cu', '.cuh', '.h')):
                src = open(os.path.join(dirpath, f)).read()
                assert 'import oracle' not in src and 'from oracle' not in src, f
