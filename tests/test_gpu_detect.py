"""End-to-end parity through the reference-facing detector (Detector protocol + batched API)."""
import ctypes

import numpy as np
import pytest

from tests.artist import artist_frame
from tests.conftest import PORCH_CONFIG, load_golden_frame
from tests.gpu_util import compare_rows, new_rows, rows_bytes, rows_to_tuples, zones_of
from watsor_b200 import _lib
from watsor_b200.detection.b200 import B200ObjectDetector
from watsor_b200.stream.share import Detection, FrameBuffer

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module', params=[0, 2], ids=['fp32-cuda-cores', 'fp32-3xtf32-tcgen05'])
def detector(shapes_model, request):
    with B200ObjectDetector(None, device=0, max_batch=64, precision=request.param,
                            model_blob=shapes_model.to_blob()) as d:
        yield d


def test_device_name(detector):
    assert 'B200' in detector.device_name and len(detector.device_name.encode()) < 255


def test_golden_cases_single_frame_protocol(detector, golden, real_shapes_model):
    """tensorflow_cpu.py:74-92 contract: detect(image_shape, image_np, detections) -> ms; all 100
    rows written; label/box ints exact (rounding ties tolerated and counted), confidence 1e-3."""
    flips = 0
    for case in golden['cases']:
        img = load_golden_frame(case['name'])
        rows = (Detection * 100)()
        ms = detector.detect(img.shape, img, rows)
        assert 0.0 < ms < 1000.0
        got = rows_to_tuples(rows)
        want = [tuple(r) for r in case['rows']] + [(1, 0.0, 0, 0, 0, 0)] * (100 - case['num'])
        flips += compare_rows(got, want, np.array(case['boxes_f64']), img.shape)
        assert zones_of(rows) == [[0] * 10] * 100          # detect() alone never writes zones
    print('tolerated rounding-tie flips:', flips)
    assert flips <= 2


def test_matches_oracle_on_fresh_artist_frames(detector, shapes_oracle, shapes_oracle64):
    from oracle.ssd_graph import to_detections
    flips = total = 0
    for (w, h, cam) in [(100, 100, 7), (320, 240, 8), (640, 480, 9), (1920, 1080, 10)]:
        for frame in range(3):
            img = artist_frame(w, h, cam, frame)
            rows = (Detection * 100)()
            detector.detect(img.shape, img, rows)
            b, cl, s, n = shapes_oracle.run(img)
            b64 = shapes_oracle64.run(img)[0]
            flips += compare_rows(rows_to_tuples(rows), to_detections(b, cl, s, img.shape), b64, img.shape)
            total += n
    assert total >= 20 and flips <= 2


def test_batch_with_fused_porch_filters(detector, golden, real_shapes_model):
    detector.configure_camera(0, 640, 480, PORCH_CONFIG)
    detector.configure_camera(1, 100, 100, None)
    detector.configure_camera(2, 320, 240, {'detect': [{'person': {'confidence': 50, 'area': 1}},
                                                       {'bicycle': {'confidence': 50, 'area': 1}},
                                                       {'car': {'confidence': 50, 'area': 1}}]})
    cam_of = {(640, 480): 0, (100, 100): 1, (320, 240): 2}
    cases = golden['cases']
    frames = [load_golden_frame(c['name']) for c in cases]
    cams = [cam_of[(c['width'], c['height'])] for c in cases]
    rows = new_rows(len(cases))
    verd = np.zeros((len(cases), 100), np.uint32)
    ms = detector.detect_batch(frames, cams, rows, [verd[i] for i in range(len(cases))], fuse_filters=True)
    assert ms > 0
    for i, c in enumerate(cases):
        want = [tuple(r) for r in c['rows']] + [(1, 0.0, 0, 0, 0, 0)] * (100 - c['num'])
        compare_rows(rows_to_tuples(rows[i]), want, np.array(c['boxes_f64']), frames[i].shape)
        n = c['num']
        if 'porch_verdicts' in c:
            assert [int(v) & 15 for v in verd[i][:n]] == c['porch_verdicts']
            assert zones_of(rows[i], n) == c['porch_zones']
        # padded rows: label 1 passes `label > 0` only; confidence 0 fails every threshold
        assert all(int(v) in (_lib.WB_V_LABEL,) for v in verd[i][n:])
        if cams[i] == 1:                                   # camera without filters: LABEL only
            assert all(int(v) == _lib.WB_V_LABEL for v in verd[i])


def test_async_slots_equal_sync(detector):
    """submit/collect on different slots give byte-identical rows to the synchronous call on the same
    batches (results are bit-reproducible for a given batch size; the split-K plan of the latency-bound
    layers depends on the batch size, so different batch sizes agree to fp32 rounding only)."""
    detector.configure_camera(5, 320, 240, None)
    frames = [artist_frame(320, 240, 20, f) for f in range(6)]
    sync_a, sync_b = new_rows(3), new_rows(3)
    detector.detect_batch(frames[:3], [5] * 3, sync_a, fuse_filters=False)
    detector.detect_batch(frames[3:], [5] * 3, sync_b, fuse_filters=False)
    a, b = new_rows(3), new_rows(3)
    detector.submit(1, frames[:3], [5] * 3, fuse_filters=False)
    detector.submit(2, frames[3:], [5] * 3, fuse_filters=False)
    detector.collect(1, a)
    detector.collect(2, b)
    for i in range(3):
        assert rows_bytes(a[i]) == rows_bytes(sync_a[i]) and rows_bytes(b[i]) == rows_bytes(sync_b[i])
    whole = new_rows(6)
    detector.detect_batch(frames, [5] * 6, whole, fuse_filters=False)
    for i in range(6):                       # other batch size: same detections, confidences to 1e-5
        ta, tb = rows_to_tuples(whole[i]), rows_to_tuples((sync_a + sync_b)[i])
        assert [t[0] for t in ta] == [t[0] for t in tb]
        assert max(abs(x[1] - y[1]) for x, y in zip(ta, tb)) < 1e-5
    with pytest.raises(_lib.WatsorB200Error, match='no batch in flight'):
        detector.collect(0, a)


def test_device_resident_frames_and_registered_shared_memory(detector):
    torch = pytest.importorskip('torch')
    detector.configure_camera(6, 640, 480, None)
    fb = FrameBuffer(4, 640, 480)
    detector.register_frame_buffer(fb)
    imgs = [artist_frame(640, 480, 30, f) for f in range(4)]
    for frame, img in zip(fb.frames, imgs):
        np.copyto(frame.get_numpy_image(np.uint8)[1], img)
    host_rows = [f.header.detections for f in fb.frames]      # written in place in shared memory
    detector.detect_batch([f.get_numpy_image(np.uint8)[1] for f in fb.frames], [6] * 4, host_rows,
                          fuse_filters=False)
    dev = [torch.from_numpy(img).cuda() for img in imgs]
    torch.cuda.synchronize()
    dev_rows = new_rows(4)
    detector.detect_batch([t.data_ptr() for t in dev], [6] * 4, dev_rows, fuse_filters=False, frames_on_device=True)
    for i in range(4):
        assert rows_to_tuples(fb.frames[i].header.detections) == rows_to_tuples(dev_rows[i])
        assert fb.frames[i].header.detections[0].label >= 1
    for frame in fb.frames:
        detector.engine.unregister_host(ctypes.addressof(frame.image.get_obj()))


def test_full_size_batch_properties(detector):
    """BASELINE configs at full size (64 frames of 640x480): size-independent properties --
    run-to-run determinism, independence from the frame's position and neighbours in the batch,
    every row written, rows sorted by score."""
    detector.configure_camera(7, 640, 480, None)
    rng = np.random.default_rng(0)
    frames = [artist_frame(640, 480, 40 + i, i) if i % 2 else
              rng.integers(0, 256, (480, 640, 3), dtype=np.uint8) for i in range(64)]
    r1, r2 = new_rows(64), new_rows(64)
    detector.detect_batch(frames, [7] * 64, r1, fuse_filters=False)
    detector.detect_batch(frames, [7] * 64, r2, fuse_filters=False)
    assert all(rows_bytes(a) == rows_bytes(b) for a, b in zip(r1, r2))
    perm = [int(i) for i in rng.permutation(64)]
    r3 = new_rows(64)
    detector.detect_batch([frames[i] for i in perm], [7] * 64, r3, fuse_filters=False)
    for k, i in enumerate(perm):                                  # independent of position / neighbours
        assert rows_bytes(r3[k]) == rows_bytes(r1[i])
    for rows in r1:
        t = rows_to_tuples(rows)
        assert all(row[0] >= 1 for row in t)                       # classes + 1 even on padding
        assert all(0 <= row[2] <= row[4] <= 639 and 0 <= row[3] <= row[5] <= 479 for row in t)
        confs = [row[1] for row in t]
        assert confs == sorted(confs, reverse=True)               # sorted by score (sortedness)


def test_errors_are_python_exceptions(detector):
    with pytest.raises(_lib.WatsorB200Error, match='has not been configured'):
        detector.engine.detect([np.zeros((10, 10, 3), np.uint8)], [200], new_rows(1))
    with pytest.raises(_lib.WatsorB200Error, match='batch size'):
        detector.engine.detect([np.zeros((480, 640, 3), np.uint8)] * 65, [7] * 65, new_rows(65))
    with pytest.raises(FileNotFoundError):
        B200ObjectDetector('/nonexistent/model/dir')
