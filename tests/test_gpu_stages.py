"""Stage-by-stage parity of the CUDA kernels against the oracle, through the C-ABI."""
import numpy as np
import pytest

from tests.conftest import load_golden_frame
from tests.gpu_util import rows_to_tuples
from watsor_b200.engine import Engine
from watsor_b200.model import OP_ADD, OP_HEAD

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module', params=[0, 2], ids=['fp32-cuda-cores', 'fp32-3xtf32-tcgen05'])
def engine(shapes_model, request):
    with Engine(shapes_model.to_blob(), device=0, max_batch=8, precision=request.param) as e:
        yield e


# ------------------------------------------------------------------------------------ K1
@pytest.mark.parametrize('shape', [(100, 100), (240, 320), (480, 640), (1080, 1920), (53, 37), (300, 300),
                                   (1, 1), (299, 301), (600, 600)])
def test_preprocess_bit_exact(engine, shapes_oracle, shape):
    rng = np.random.default_rng(shape[0] * 7 + shape[1])
    img = rng.integers(0, 256, shape + (3,), dtype=np.uint8)
    got = engine.preprocess([img])[0]
    want = shapes_oracle.preprocess(img)
    assert got.dtype == np.float32 and np.array_equal(got, want)


def test_preprocess_batch_of_mixed_sizes(engine, shapes_oracle):
    rng = np.random.default_rng(1)
    imgs = [rng.integers(0, 256, s + (3,), dtype=np.uint8) for s in [(100, 100), (480, 640), (240, 320), (7, 900)]]
    got = engine.preprocess(imgs)
    for g, img in zip(got, imgs):
        assert np.array_equal(g, shapes_oracle.preprocess(img))


# ------------------------------------------------------------------------------- K2..K6
def test_anchors_equal_graph_constant(engine, shapes_oracle):
    assert np.array_equal(engine.anchors(), shapes_oracle.anchors)


def test_backbone_layer_by_layer(engine, shapes_model, shapes_oracle):
    """Every layer's activation vs torch-CPU fp32 on the same pre-processed input.  fp32 with a
    different summation order: agreement to ~1e-5 relative of the layer's range is the bar."""
    img = load_golden_frame('artist_640x480_c0_f0')
    pre = shapes_oracle.preprocess(img)
    enc, lg, memo = shapes_oracle.raw_heads(pre, return_memo=True)
    worst = 0.0
    for li, layer in enumerate(shapes_model.layers):
        if layer.op == OP_HEAD:
            continue
        want = shapes_oracle.feature(memo, li)
        _, _, got = engine.backbone(pre[None], stop_layer=li, layer_shape=want.shape)
        err = np.abs(got[0] - want).max()
        scale = max(1.0, float(np.abs(want).max()))
        worst = max(worst, err / scale)
        assert err <= 6e-5 * scale, (li, layer.name, err, scale)
    genc, glg, _ = engine.backbone(pre[None])
    assert np.abs(genc[0] - enc).max() <= 1e-4 and np.abs(glg[0] - lg).max() <= 3e-4
    print('worst relative layer error %.2e' % worst)


def test_backbone_batch_invariance(engine, shapes_oracle):
    rng = np.random.default_rng(5)
    pres = np.stack([shapes_oracle.preprocess(rng.integers(0, 256, (120, 160, 3), dtype=np.uint8)) for _ in range(5)])
    e_all, l_all, _ = engine.backbone(pres)
    e_rev, l_rev, _ = engine.backbone(pres[::-1].copy())            # same batch size, other order: bit-identical
    assert np.array_equal(e_rev[::-1], e_all) and np.array_equal(l_rev[::-1], l_all)
    for i in (0, 3, 4):                                             # other batch size: fp32 rounding only
        e1, l1, _ = engine.backbone(pres[i:i + 1])
        assert np.abs(e1[0] - e_all[i]).max() < 2e-5 and np.abs(l1[0] - l_all[i]).max() < 1e-4


# ------------------------------------------------------------------------------- K7..K9
def check_post(engine, oracle, enc, logits, cam=0, hw=(480, 640)):
    from oracle.ssd_graph import to_detections
    rows, verd, boxes, scores, classes, num = engine.postprocess(enc[None], logits[None], [cam])
    b, s, cl, n = oracle.postprocess(enc, logits)
    assert num[0] == n
    assert np.array_equal(classes[0], cl)
    # CUDA expf vs host exp may differ in the last ulp: boxes/scores to 2 ulp, never more
    assert np.allclose(boxes[0], b, rtol=0, atol=3e-7) and np.allclose(scores[0], s, rtol=0, atol=2e-7)
    want = to_detections(b, cl, s, hw + (3,))
    got = rows_to_tuples(rows[0])
    mism = [(g, w) for g, w in zip(got, want) if g[0] != w[0] or g[2:] != w[2:] or abs(g[1] - w[1]) > 2e-7]
    return n, mism


def test_post_on_oracle_heads_golden_frames(engine, shapes_oracle, golden, real_shapes_model):
    """The golden vectors were recorded on the real weights, which `engine` runs whenever they are built."""
    engine.set_camera(0, 640, 480)
    engine.set_camera(1, 100, 100)
    engine.set_camera(2, 320, 240)
    cams = {(640, 480): 0, (100, 100): 1, (320, 240): 2}
    for case in golden['cases']:
        img = load_golden_frame(case['name'])
        enc, lg = shapes_oracle.raw_heads(shapes_oracle.preprocess(img))
        n, mism = check_post(engine, shapes_oracle, enc, lg, cams[(case['width'], case['height'])],
                             (case['height'], case['width']))
        assert n == case['num'] and not mism, mism[:3]


@pytest.mark.parametrize('seed', range(4))
def test_post_random_heads_stress_nms(engine, shapes_oracle, seed):
    """Random head outputs: hundreds of candidates per class, overlapping boxes, exact score ties
    (quantised logits) -> exercises sort order, tie-breaks, strict thresholds, top-100 cut."""
    engine.set_camera(0, 640, 480)
    rng = np.random.default_rng(seed)
    n = shapes_oracle.num_anchors
    enc = (rng.standard_normal((n, 4)) * [1.5, 1.5, 1.0, 1.0]).astype(np.float32)
    lg = (rng.standard_normal((n, 4)) * 2.0 - (1.0 if seed % 2 else -0.5)).astype(np.float32)
    if seed >= 2:
        lg = np.round(lg * 4) / 4           # many exact ties
        lg = lg.astype(np.float32)
    cnt, mism = check_post(engine, shapes_oracle, enc, lg)
    assert cnt == 100 and not mism, mism[:3]


def test_post_edge_cases(engine, shapes_oracle):
    engine.set_camera(0, 640, 480)
    n = shapes_oracle.num_anchors
    # nothing above threshold: 100 padded rows (label 1, confidence 0, zero box)
    enc = np.zeros((n, 4), np.float32)
    lg = np.full((n, 4), -10.0, np.float32)
    rows, verd, boxes, scores, classes, num = engine.postprocess(enc[None], lg[None], [0])
    assert num[0] == 0 and set(rows_to_tuples(rows[0])) == {(1, 0.0, 0, 0, 0, 0)}
    # everything identical and above threshold: one survivor per class (IoU 1 > 0.6), lowest index wins
    lg = np.full((n, 4), 3.0, np.float32)
    cnt, mism = check_post(engine, shapes_oracle, enc, lg)
    assert not mism
    # boxes pushed far outside the window get a zero clipped area and must vanish
    enc = np.zeros((n, 4), np.float32)
    enc[:, 0] = 400.0
    cnt, mism = check_post(engine, shapes_oracle, enc, lg)
    assert not mism


@pytest.mark.parametrize('precision', [0, 2], ids=['fp32-cuda-cores', 'fp32-3xtf32-tcgen05'])
def test_post_coco_heads_90_classes(coco_model, precision):
    """90-class heads, threshold 1e-8 (every anchor is a candidate in every class); the post stage is the same
    code in every precision mode, run here in both the reported one and the CUDA-core one."""
    from oracle.ssd_model import SsdModelOracle
    oracle = SsdModelOracle(coco_model)
    rng = np.random.default_rng(11)
    n = oracle.num_anchors
    enc = (rng.standard_normal((n, 4)) * 0.8).astype(np.float32)
    lg = (rng.standard_normal((n, 91)) * 1.5 - 3.0).astype(np.float32)
    with Engine(coco_model.to_blob(), device=0, max_batch=2, precision=precision) as e:
        e.set_camera(0, 640, 480)
        cnt, mism = check_post(e, oracle, enc, lg)
        assert cnt == 100 and not mism, mism[:3]
