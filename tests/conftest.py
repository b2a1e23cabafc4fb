import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN_DIR = os.path.join(ROOT, 'tests', 'golden')
# built by __graft_entry__.build() where a checkout of the original watsor project is readable
# (oracle/reference_build.py); absent otherwise
REF_BUILD = os.path.join(ROOT, 'oracle', '_ref')
MODEL_BLOB = os.path.join(REF_BUILD, 'ssd_mobilenet_v1_shapes', 'b200.wb200')
REF_PB = os.path.join(REF_BUILD, 'cpu.pb')


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: needs a real B200 (run with `pytest -m gpu`)')


def has_gpu():
    from watsor_b200 import _lib
    try:
        return _lib.device_count() > 0
    except Exception:
        return False


@pytest.fixture(scope='session')
def golden():
    with open(os.path.join(GOLDEN_DIR, 'ssd_shapes_golden.json')) as f:
        return json.load(f)


@pytest.fixture(scope='session')
def real_shapes_model():
    """The original project's 3-class SSD-MobileNet-v1 test model (watsor/test/model/cpu.pb, real weights) as a
    compiled blob.  Its 22 MB of weights are not part of this repository: the tests that compare with vectors recorded
    on those weights run where oracle/_ref/ has been built."""
    from watsor_b200.model import Model
    if not os.path.isfile(MODEL_BLOB):
        pytest.skip('oracle/_ref/ blob missing (__graft_entry__.build() found no checkout of the original project)')
    return Model.load(MODEL_BLOB)


@pytest.fixture(scope='session')
def shapes_model():
    """The 3-class SSD-MobileNet-v1 for tests that compare two computations on the same model: the real weights where
    oracle/_ref/ has been built, else the same architecture with seeded synthetic weights (as smoke() runs)."""
    from watsor_b200.model import Model, synthetic_ssd_mobilenet_v1
    if os.path.isfile(MODEL_BLOB):
        return Model.load(MODEL_BLOB)
    return synthetic_ssd_mobilenet_v1(num_classes=3, seed=1, score_thr=0.3)


@pytest.fixture(scope='session')
def shapes_oracle(shapes_model):
    from oracle.ssd_model import SsdModelOracle
    return SsdModelOracle(shapes_model)


@pytest.fixture(scope='session')
def real_shapes_oracle(real_shapes_model):
    from oracle.ssd_model import SsdModelOracle
    return SsdModelOracle(real_shapes_model)


@pytest.fixture(scope='session')
def shapes_oracle64(shapes_model):
    from oracle.ssd_model import SsdModelOracle
    return SsdModelOracle(shapes_model, dtype=np.float64)


@pytest.fixture(scope='session')
def coco_model():
    """SSD-MobileNet-v1 with 90-class heads and seeded synthetic weights (no COCO weights exist
    offline); threshold 1e-8 as in the TF model-zoo graphs."""
    from watsor_b200.model import synthetic_ssd_mobilenet_v1
    return synthetic_ssd_mobilenet_v1(num_classes=90, seed=0, score_thr=1e-8)


def load_golden_frame(name):
    from PIL import Image
    return np.array(Image.open(os.path.join(GOLDEN_DIR, 'frames', name + '.png')).convert('RGB'))


PORCH_CONFIG = {
    'width': 640, 'height': 480, 'mask': os.path.join(GOLDEN_DIR, 'porch.png'),
    'detect': [{'person': {'confidence': 50, 'area': 1, 'zones': []}},
               {'bicycle': {'confidence': 50, 'area': 1, 'zones': [2]}},
               {'car': {'confidence': 50, 'area': 10, 'zones': []}}]}
