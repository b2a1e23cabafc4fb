"""The reference's own model test (ref: watsor/test/test_detect.py:28-77) with the reference's stream runtime
(`watsor.stream`: FrameBuffer, StateLatch, Work / Spin, ReadDetectPublish Artist, ShapeCounter) and this repository's
drop-in detector worker, sieve and filters on the real B200 back-end; the detector runs in a `Process` under
`spawn`.  The reference package and model come from oracle/_ref/ (built by __graft_entry__.build() from a readable
checkout of the original project, oracle/reference_build.py)."""
import json
import os
import subprocess
import sys

import pytest

from tests.conftest import MODEL_BLOB, ROOT

pytestmark = pytest.mark.gpu
REF_PKG = os.path.join(ROOT, 'oracle', '_ref', 'site')


@pytest.mark.skipif(not os.path.isfile(os.path.join(REF_PKG, 'watsor', 'stream', 'work.py')),
                    reason='oracle/_ref/site (copy of the reference package) is missing')
@pytest.mark.skipif(not os.path.isfile(MODEL_BLOB), reason='oracle/_ref/ blob missing')
def test_shape_detection_reference_runtime_real_backend_spawned_process():
    env = dict(os.environ, PYTHONPATH=REF_PKG + os.pathsep + ROOT)
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'tests', 'scenario_reference_worker.py')], env=env,
                         capture_output=True, text=True, timeout=300)
    print(out.stdout[-1500:], out.stderr[-1500:])
    assert out.returncode == 0, out.stderr[-3000:]
    r = json.loads(out.stdout.strip().splitlines()[-1])
    assert r['ok'], r                                   # >= 100 labelled detections with confidence >= 0.5
    assert 'B200' in r['device_name'] and r['detector_fps'] > 0 and r['inference_ms'] > 0
    assert not r['alive_after_join'] and not r['errors'], r
