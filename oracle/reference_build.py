"""Builds oracle/_ref/ (git-ignored) from a checkout of the original watsor project, for the tests that need more of
it than the vectors stored under tests/golden/:

    oracle/_ref/cpu.pb                                    its test model, watsor/test/model/cpu.pb (22 MB of weights)
    oracle/_ref/ssd_mobilenet_v1_shapes/b200.wb200        that graph compiled for libwatsor_b200.so
    oracle/_ref/site/watsor/                              a copy of the unmodified package, which hosts the drop-in
                                                          detector worker in the integration tests

The checkout is WATSOR_REFERENCE, else the project's usual checkout location (DEFAULT_CHECKOUT).  Nothing of it is
read by the product."""
import os
import shutil

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), '_ref')
PB = os.path.join(OUT, 'cpu.pb')
MODEL_BLOB = os.path.join(OUT, 'ssd_mobilenet_v1_shapes', 'b200.wb200')
SITE = os.path.join(OUT, 'site')
DEFAULT_CHECKOUT = '/root/reference'


def find_reference():
    """The root of a readable checkout of the original project (the directory holding watsor/), or None."""
    for root in (os.environ.get('WATSOR_REFERENCE'), DEFAULT_CHECKOUT):
        if root and os.access(os.path.join(root, 'watsor', 'test', 'model', 'cpu.pb'), os.R_OK):
            return root
    return None


def _write_if_changed(path, data):
    if os.path.isfile(path) and open(path, 'rb').read() == data:
        return
    os.makedirs(os.path.dirname(path), exist_ok=True)
    with open(path, 'wb') as f:
        f.write(data)


def build(reference):
    """`reference`: the root of the original project's checkout (the directory holding watsor/)."""
    from watsor_b200.model import compile_frozen_graph
    _write_if_changed(PB, open(os.path.join(reference, 'watsor', 'test', 'model', 'cpu.pb'), 'rb').read())
    model = compile_frozen_graph(PB, name='ssd_mobilenet_v1_shapes (watsor/test/model/cpu.pb)')
    _write_if_changed(MODEL_BLOB, model.to_blob())
    if not os.path.isfile(os.path.join(SITE, 'watsor', 'stream', 'work.py')):
        # a pure-Python package: the copy is what an install would put on the path (the model stays in cpu.pb above)
        shutil.rmtree(SITE, ignore_errors=True)
        shutil.copytree(os.path.join(reference, 'watsor'), os.path.join(SITE, 'watsor'),
                        ignore=shutil.ignore_patterns('__pycache__', '*.pyc', '*.pb'))
