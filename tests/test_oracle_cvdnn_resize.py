"""The legacy `ResizeBilinear` of the frozen graph (align_corners = false, half_pixel_centers = false: src = dst *
in/out, no half-pixel shift) executed by an independent implementation: OpenCV's dnn module imports the reference's
OWN node -- `Preprocessor/map/while/ResizeImage/resize/ResizeBilinear`, attributes untouched, rewired to a Placeholder
and a constant size -- and runs it with its own kernel.  oracle.preprocess (the restatement every GPU parity test of
the resize stage leans on, bit-exactly) must agree to float rounding at every size, up- and down-scaling.  Together
with tests/test_oracle_cvdnn.py (convolutions) and tests/test_oracle_cvdnn_post.py (decode / NMS / top-100) this
leaves no arithmetic stage of the graph pinned by the restatement's author alone.  CPU only; where oracle/_ref/cpu.pb
is absent the node is rebuilt with the same two attributes."""
import os

import cv2
import numpy as np
import pytest

from tests.conftest import REF_PB

SIZES = [(640, 480), (1920, 1080), (1280, 720), (100, 80), (300, 300), (641, 479), (37, 1000), (1, 1)]


def resize_graph(h, w, out_h, out_w):
    from tensorboard.compat.proto import graph_pb2, types_pb2
    g = graph_pb2.GraphDef()
    ph = g.node.add()
    ph.name, ph.op = 'image', 'Placeholder'
    ph.attr['dtype'].type = types_pb2.DT_FLOAT
    for d in (1, h, w, 3):
        ph.attr['shape'].shape.dim.add().size = d
    size = g.node.add()
    size.name, size.op = 'size', 'Const'
    size.attr['dtype'].type = types_pb2.DT_INT32
    t = size.attr['value'].tensor
    t.dtype = types_pb2.DT_INT32
    t.tensor_shape.dim.add().size = 2
    t.int_val.extend([out_h, out_w])
    node = g.node.add()
    if os.path.isfile(REF_PB):
        from oracle.tf_graph import FrozenGraph
        ref = FrozenGraph(REF_PB)
        name = [n for n in ref.order if ref.node(n).op == 'ResizeBilinear']
        assert len(name) == 1
        node.CopyFrom(ref.node(name[0]))
        del node.input[:]
    else:
        node.name, node.op = 'ResizeBilinear', 'ResizeBilinear'
        node.attr['T'].type = types_pb2.DT_FLOAT
        node.attr['align_corners'].b = False
        node.attr['half_pixel_centers'].b = False
    assert not node.attr['align_corners'].b and not node.attr['half_pixel_centers'].b
    node.input.extend(['image', 'size'])
    return g.SerializeToString()


@pytest.mark.parametrize('size', SIZES)
def test_legacy_resize_equals_opencv_dnn_running_the_reference_node(size, shapes_oracle):
    w, h = size
    o = shapes_oracle
    img = np.random.default_rng(w * 7 + h).integers(0, 256, (h, w, 3), dtype=np.uint8)
    net = cv2.dnn.readNetFromTensorflow(np.frombuffer(resize_graph(h, w, o.in_h, o.in_w), np.uint8))
    net.setInput(np.ascontiguousarray(img.astype(np.float32).transpose(2, 0, 1)[None]))
    resized = net.forward()[0].transpose(1, 2, 0)                       # NCHW -> HWC, values 0..255
    theirs = resized * np.float32(o.pre_mul) - np.float32(o.pre_sub)     # Preprocessor/mul, Preprocessor/sub
    ours = o.preprocess(img)
    assert ours.shape == theirs.shape == (o.in_h, o.in_w, 3)
    assert float(np.abs(ours - theirs).max()) <= 5e-7, size             # 2 ulp of values in [-1, 1]
