"""Per-layer error of the tensor-core precisions against the oracle (run under gpurun)."""
import sys, os, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from watsor_b200.engine import Engine
from watsor_b200.model import Model, OP_HEAD, OP_NAMES
from oracle.reference_build import MODEL_BLOB
from oracle.ssd_model import SsdModelOracle
from tests.artist import artist_frame

prec = [int(x) for x in sys.argv[1].split(',')] if len(sys.argv) > 1 else [3, 2, 1]
m = Model.load(MODEL_BLOB)
o = SsdModelOracle(m)
imgs = [artist_frame(640, 480, 0, f) for f in range(3)]
pres = np.stack([o.preprocess(i) for i in imgs])
refs = [o.raw_heads(p, return_memo=True) for p in pres]
for p in prec:
    print('=== precision', p, flush=True)
    with Engine(m.to_blob(), device=0, max_batch=4, precision=p) as e:
        print(e.device_name, flush=True)
        for li, l in enumerate(m.layers):
            if l.op == OP_HEAD:
                continue
            want = np.stack([o.feature(r[2], li) for r in refs])
            _, _, got = e.backbone(pres, stop_layer=li, layer_shape=want.shape[1:])
            err = np.abs(got - want).max(); sc = max(1.0, np.abs(want).max())
            print('%2d %-5s %4dx%-4d->%4d  maxerr %.3e  rel %.2e' % (li, OP_NAMES[l.op], l.in_h, l.in_c, l.out_c, err, err / sc), flush=True)
        enc, lg, _ = e.backbone(pres)
        print('enc err %.3e logits err %.3e' % (np.abs(enc - np.stack([r[0] for r in refs])).max(), np.abs(lg - np.stack([r[1] for r in refs])).max()))
