"""`b200_gpus()` against the reference's own `cuda_gpus()` (watsor/detection/devices.py:28-77), run here with
stand-in `pycuda.driver` / `watsor.detection.tensorrt_gpu` modules that only report a device count: same devices
in the same order, same TypeError, for every combination of CUDA_DEVICE, ~/.cuda_device and device count.
CPU only; the reference's answers are recorded in tests/golden/reference/devices.json (tests/reference_outputs.py)."""
import sys
import types

import pytest

from tests.reference_outputs import REFERENCE, Recorded, canon

recorded = Recorded('devices')


@pytest.fixture()
def both(monkeypatch):
    count = {'n': 0}
    driver = types.ModuleType('pycuda.driver')
    driver.init = lambda: None
    driver.Device = types.SimpleNamespace(count=lambda: count['n'])
    driver.RuntimeError = type('RuntimeError', (Exception,), {})
    pycuda = types.ModuleType('pycuda')
    pycuda.driver = driver
    trt = types.ModuleType('watsor.detection.tensorrt_gpu')
    trt.TensorRTObjectDetector = type('TensorRTObjectDetector', (), {})
    for name, mod in (('pycuda', pycuda), ('pycuda.driver', driver), ('watsor.detection.tensorrt_gpu', trt)):
        monkeypatch.setitem(sys.modules, name, mod)
    cuda_gpus = None
    if REFERENCE:
        monkeypatch.syspath_prepend(REFERENCE)
        from watsor.detection.devices import cuda_gpus
    from watsor_b200 import _lib
    from watsor_b200.detection.devices import b200_gpus
    monkeypatch.setattr(_lib, 'device_count', lambda: count['n'])

    def call(gen):
        try:
            return [d for d, _ in gen()]
        except TypeError as e:
            return 'TypeError: %s' % e

    def run(n, key):
        count['n'] = n
        return recorded(key, lambda: call(cuda_gpus)), canon(call(b200_gpus))
    yield run
    for name in [m for m in sys.modules if m == 'watsor' or m.startswith('watsor.')]:
        sys.modules.pop(name, None)


@pytest.mark.parametrize('n', [0, 1, 8])
@pytest.mark.parametrize('env', [None, '0', '3', ' 5 ', 'x', ''])
@pytest.mark.parametrize('dotfile', [None, '2', '7\n', 'gpu1', ''])
@pytest.mark.parametrize('home', [True, False])
def test_same_devices_as_the_reference_generator(both, monkeypatch, tmp_path, n, env, dotfile, home):
    if env is None:
        monkeypatch.delenv('CUDA_DEVICE', raising=False)
    else:
        monkeypatch.setenv('CUDA_DEVICE', env)
    if home:
        monkeypatch.setenv('HOME', str(tmp_path))
        if dotfile is not None:
            (tmp_path / '.cuda_device').write_text(dotfile)
    else:
        monkeypatch.delenv('HOME', raising=False)
    theirs, ours = both(n, repr((n, env, dotfile, home)))
    assert ours == theirs, (n, env, dotfile, home)
    if n == 0:
        assert ours == []
