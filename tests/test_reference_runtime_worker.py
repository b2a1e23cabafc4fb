"""The drop-in ObjectDetector hosted on the reference's own stream runtime (ref: watsor/stream/{spin,work,share,
sync}.py), in a fresh interpreter so that `watsor_b200.detection.detector` binds to `watsor.stream` at import."""
import json
import os
import subprocess
import sys

import pytest

from tests.conftest import ROOT


def reference_path():
    from oracle.reference_build import find_reference
    for p in (find_reference(), os.path.join(ROOT, 'oracle', '_ref', 'site')):
        if p and os.path.isfile(os.path.join(p, 'watsor', 'stream', 'work.py')):
            return p
    return None


@pytest.mark.skipif(reference_path() is None, reason='reference runtime not available')
def test_pipelined_worker_on_the_reference_runtime():
    env = dict(os.environ, PYTHONPATH=reference_path() + os.pathsep + ROOT)
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'tests', 'scenario_fake_backend.py')], env=env,
                         capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr[-2000:]
    r = json.loads(out.stdout.strip().splitlines()[-1])
    # every frame left DETECT exactly once: READY(0) -> DETECT(1) by the scenario, then one latch.next() -> PUBLISH
    assert r['states'] == [r['publish']] * 8
    # rows were written before the latch moved; frame 6's batch (collect raised) has no rows but its latch moved too
    bad = {5, 6, 7} if r['labels'][5] == 0 else {i for i in range(8) if r['labels'][i] == 0}
    assert 6 in bad and all(r['labels'][i] == i + 1 for i in range(8) if i not in bad)
    ev = [tuple(e) for e in r['events']]
    assert ('register', 8) in ev and ('configure', 0, 16, 8) in ev
    submits = [e for e in ev if e[0] == 'submit']
    assert sum(e[2] for e in submits) == 8 and max(e[2] for e in submits) <= 3
    # pipelining: the second submit happens before the first collect
    first_collect = next(i for i, e in enumerate(ev) if e[0] == 'collect')
    assert sum(1 for e in ev[:first_collect] if e[0] == 'submit') >= 2
    assert r['device_name'] == 'FAKE-PIPE:0' and r['inference_time'] == 0.75 and not r['alive']
