#!/usr/bin/env python
"""The reference's only model test, restated with the reference's OWN stream runtime and the real B200 back-end
(ref: watsor/test/test_detect.py:28-77): an Artist thread draws shapes into a shared `FrameBuffer`, the detector
runs in a separate *process* under `spawn`, the DetectionSieve filters confidence >= 50 %, a ShapeCounter counts
labelled detections and the test passes when 100 have been seen.

Run as a script in a fresh interpreter (tests/test_gpu_worker.py does) with the reference package on PYTHONPATH
(oracle/_ref/site, copied there by __graft_entry__.build() from a readable checkout): the detector module must
bind to `watsor.stream.*` at import time, here and in the spawned child.

Everything from `watsor.*` below is the reference's code; `create_object_detectors`, `ObjectDetector`,
`DetectionSieve`, `TrackFilter`, `ConfidenceFilter` are this repository's drop-ins.  The one deviation: the
reference Artist hands float bounds to `random.randrange`, which Python 3.12 rejects, so its drawing routine is
replaced by tests/artist.py's integral restatement.
"""
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def main(width=100, height=100, wanted=100, wait_s=90.0):
    from logging import getLogger
    from logging.handlers import QueueHandler
    from multiprocessing import Event, Process, Queue, set_start_method
    from threading import Thread

    set_start_method('spawn')

    import watsor.stream.work as ref_work
    from watsor.stream.share import FrameBuffer
    from watsor.stream.sync import CountDownLatch
    from watsor.test.detect_stream import Artist, ShapeCounter

    from tests import artist as integral_artist
    from watsor_b200.config.coco import get_coco_class
    from watsor_b200.detection import detector as det_mod
    from watsor_b200.filter.confidence import ConfidenceFilter
    from watsor_b200.filter.sieve import DetectionSieve
    from watsor_b200.filter.track import TrackFilter

    assert det_mod.Work is ref_work.Work, 'the detector did not bind to the reference runtime'

    class IntegralArtist(Artist):
        @classmethod
        def draw_random_shapes(cls, image, draw):
            integral_artist.draw_random_shapes(image, draw)

    class RateLimiter:                      # ref: watsor/stream/ffmpeg.py RateLimiter as the sieve uses it
        def unlimited(self):
            return False

    frame_buffer = FrameBuffer(10, width, height)
    frame_queue, subscriber_queue, sieve_queue, log_queue = Queue(1), Queue(1), Queue(1), Queue()
    getLogger().addHandler(QueueHandler(log_queue))
    stop = Event()
    latch = CountDownLatch(wanted)
    artist = IntegralArtist('artist', stop, log_queue, frame_queue, frame_buffer)
    filters = [TrackFilter([ConfidenceFilter({'detect': [{get_coco_class(1).label: {'confidence': 50}},
                                                         {get_coco_class(2).label: {'confidence': 50}},
                                                         {get_coco_class(3).label: {'confidence': 50}}]})])]
    sieve = DetectionSieve('sieve', stop, log_queue, sieve_queue, frame_buffer, filters, RateLimiter())
    counter = ShapeCounter(Thread, 'counter', stop, log_queue, subscriber_queue, frame_buffer, latch)
    model_path = os.path.join(ROOT, 'oracle', '_ref', 'ssd_mobilenet_v1_shapes')
    detectors = det_mod.create_object_detectors(Process, stop, log_queue, frame_queue, {artist.name: frame_buffer},
                                                model_path)
    processes = [artist, sieve, counter] + detectors[:1]
    artist.subscribe(sieve_queue)
    sieve.subscribe(subscriber_queue)
    t0 = time.time()
    for p in processes:
        p.start()
    ok = False
    try:
        ok = latch.wait(wait_s)
    finally:
        elapsed = time.time() - t0
        stop.set()
        for p in processes:
            p.join(30)
    logs = []
    while not log_queue.empty():
        rec = log_queue.get_nowait()
        logs.append('%s %s' % (rec.levelname, rec.getMessage()))
    d = detectors[0]
    print(json.dumps({'ok': bool(ok), 'elapsed_s': elapsed, 'device_name': d.device_name.decode(errors='replace'),
                      'detector_fps': d.fps(), 'inference_ms': d.inference_time(),
                      'alive_after_join': [p.name for p in processes if p.is_alive()],
                      'errors': [l for l in logs if l.startswith(('ERROR', 'CRITICAL'))][:5]}))
    return 0 if ok else 1


if __name__ == '__main__':
    sys.exit(main())
