#!/usr/bin/env python
"""Statistical parity report: many Artist frames through the B200 detector (every precision mode)
vs the fp32 oracle, with the float64 oracle used to classify integer-coordinate mismatches as genuine
rounding ties or not.  Writes profiles/<round>_parity_report.md.  Run under gpurun."""
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from oracle.reference_build import MODEL_BLOB  # noqa: E402
from oracle.ssd_graph import to_detections  # noqa: E402
from oracle.ssd_model import SsdModelOracle  # noqa: E402
from tests.artist import artist_frame  # noqa: E402
from tests.gpu_util import rows_to_tuples  # noqa: E402
from watsor_b200.detection.b200 import B200ObjectDetector  # noqa: E402
from watsor_b200.model import Model  # noqa: E402
from watsor_b200.stream.share import Detection  # noqa: E402

n_frames = int(sys.argv[1]) if len(sys.argv) > 1 else 120
rnd = sys.argv[2] if len(sys.argv) > 2 else 'r01'
torch.set_num_threads(16)
model = Model.load(MODEL_BLOB)
o32, o64 = SsdModelOracle(model), SsdModelOracle(model, dtype=np.float64)
sizes = [(100, 100), (320, 240), (640, 480), (1920, 1080)]
frames = [artist_frame(*sizes[i % 4], cam=100 + i % 7, frame=i) for i in range(n_frames)]
t0 = time.time()
want = []
for img in frames:
    b, cl, s, n = o32.run(img)
    b64 = o64.run(img)[0]
    want.append((to_detections(b, cl, s, img.shape), n, b64))
t_oracle = time.time() - t0
report = {'frames': n_frames, 'oracle_seconds': t_oracle, 'modes': {}}
for prec, name in [(0, 'fp32 (CUDA cores)'), (2, 'tf32x3 (tcgen05, fp32-faithful)'), (1, 'bf16 (tcgen05)')]:
    st = dict(frames=0, frames_all_rows_equal=0, detections=0, label_mismatch=0, count_mismatch=0, coords=0,
              coord_mismatch=0, coord_mismatch_tie=0, coord_mismatch_gt1=0, max_conf_err=0.0, conf_gt_1e3=0)
    with B200ObjectDetector(None, device=0, max_batch=8, precision=prec, model_blob=model.to_blob()) as det:
        for img, (rows_w, n, b64) in zip(frames, want):
            rows = (Detection * 100)()
            det.detect(img.shape, img, rows)
            got = rows_to_tuples(rows)
            st['frames'] += 1
            n_got = sum(1 for g in got if g[1] > 0)
            if n_got != n:
                st['count_mismatch'] += 1
            ok = True
            for r in range(min(n, n_got)):
                g, w = got[r], rows_w[r]
                st['detections'] += 1
                if g[0] != w[0]:
                    st['label_mismatch'] += 1
                    ok = False
                    continue
                e = abs(g[1] - w[1])
                st['max_conf_err'] = max(st['max_conf_err'], e)
                if e > 1e-3:
                    st['conf_gt_1e3'] += 1
                    ok = False
                for k in range(4):
                    st['coords'] += 1
                    if g[2 + k] != w[2 + k]:
                        ok = False
                        st['coord_mismatch'] += 1
                        if abs(g[2 + k] - w[2 + k]) > 1:
                            st['coord_mismatch_gt1'] += 1
                        coord = b64[r][[1, 0, 3, 2][k]]
                        scale = (img.shape[1] - 1) if k in (0, 2) else (img.shape[0] - 1)
                        v = min(max(coord, 0.0), 1.0) * scale
                        if abs(v - round(v)) <= 2e-3:
                            st['coord_mismatch_tie'] += 1
            if ok and n_got == n:
                st['frames_all_rows_equal'] += 1
    report['modes'][name] = st
    print(name, st, flush=True)
os.makedirs(os.path.join(ROOT, 'profiles'), exist_ok=True)
with open(os.path.join(ROOT, 'gpurun_out', '%s_parity_report.json' % rnd), 'w') as f:
    json.dump(report, f, indent=1)
