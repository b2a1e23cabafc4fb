"""The oracle's conv arithmetic pinned by an independent executor of the reference's own frozen graph:
OpenCV's dnn module (its own TensorFlow importer and CPU kernels) run on the backbone + heads sub-graph of
watsor/test/model/cpu.pb.  Vectors: tests/golden/cvdnn_heads.npz, made by tools/make_golden_cvdnn.py --
"OpenCV-dnn, not TensorFlow".  Resize, anchors, decode and NMS are NOT covered by this pin (they stay restated
from the graph, oracle/ssd_graph.py)."""
import os
import sys

import numpy as np
import pytest

from tests.artist import artist_frame
from tests.conftest import GOLDEN_DIR, REF_PB, ROOT

NPZ = os.path.join(GOLDEN_DIR, 'cvdnn_heads.npz')
FRAMES = [(100, 100, 1, 0), (320, 240, 2, 1), (640, 480, 3, 2)]
TOL = 1e-4          # absolute, on tensors whose range is ~7 (encodings) and ~21 (logits)


def key(w, h, cam, frame):
    return 'artist_%dx%d_c%d_f%d' % (w, h, cam, frame)


def test_vectors_are_labelled_and_complete():
    z = np.load(NPZ)
    assert str(z['source']) == 'OpenCV-dnn, not TensorFlow'
    for f in FRAMES:
        assert z[key(*f) + '_enc'].shape == (1917, 4) and z[key(*f) + '_logits'].shape == (1917, 4)


def test_blob_oracle_equals_opencv_dnn(real_shapes_oracle):
    """oracle.raw_heads(pre) == OpenCV-dnn forward() of the reference's graph, <= 1e-4 (measured: 4e-5)."""
    z = np.load(NPZ)
    for f in FRAMES:
        pre = real_shapes_oracle.preprocess(artist_frame(*f))
        enc, lg = real_shapes_oracle.raw_heads(pre)
        assert np.abs(enc - z[key(*f) + '_enc']).max() <= TOL
        assert np.abs(lg - z[key(*f) + '_logits']).max() <= TOL


@pytest.mark.skipif(not os.path.isfile(REF_PB), reason='oracle/_ref/cpu.pb not built')
def test_live_opencv_run_reproduces_the_committed_vectors_and_the_graph_oracle():
    sys.path.insert(0, os.path.join(ROOT, 'tools'))
    from make_golden_cvdnn import cut_graph, run_cvdnn
    from oracle.ssd_graph import SsdGraphOracle
    graph_bytes, boxes, classes, ncp1 = cut_graph(REF_PB)
    oracle = SsdGraphOracle(REF_PB)
    z = np.load(NPZ)
    f = FRAMES[0]
    pre = oracle.preprocess(artist_frame(*f))
    enc, lg = run_cvdnn(graph_bytes, boxes, classes, ncp1, pre)
    # thread scheduling may change OpenCV's summation order between runs: not bit-equal, but far inside TOL
    assert np.abs(enc - z[key(*f) + '_enc']).max() <= 2e-5 and np.abs(lg - z[key(*f) + '_logits']).max() <= 2e-5
    oenc, olg = oracle.raw_heads(pre)
    assert np.abs(enc - oenc).max() <= TOL and np.abs(lg - olg).max() <= TOL
    # the unfused OpenCV execution (every BatchNorm / ReLU6 as its own layer) agrees too
    enc2, lg2 = run_cvdnn(graph_bytes, boxes, classes, ncp1, pre, fusion=False)
    assert np.abs(enc2 - oenc).max() <= TOL and np.abs(lg2 - olg).max() <= TOL


@pytest.mark.gpu
@pytest.mark.parametrize('precision', [0, 2], ids=['fp32-cuda-cores', 'fp32-3xtf32-tcgen05'])
def test_gpu_heads_equal_opencv_dnn(real_shapes_model, real_shapes_oracle, precision):
    """The CUDA path against the independent executor directly (no oracle in between except the bit-exact resize)."""
    from watsor_b200.engine import Engine
    z = np.load(NPZ)
    with Engine(real_shapes_model.to_blob(), device=0, max_batch=2, precision=precision) as e:
        for f in FRAMES:
            pre = e.preprocess([artist_frame(*f)])
            assert np.array_equal(pre[0], real_shapes_oracle.preprocess(artist_frame(*f)))
            enc, lg, _ = e.backbone(pre)
            assert np.abs(enc[0] - z[key(*f) + '_enc']).max() <= 2e-4
            assert np.abs(lg[0] - z[key(*f) + '_logits']).max() <= 2e-4
