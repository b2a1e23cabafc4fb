"""Pipeline timeline of CTA 0 of the tensor-core kernels (diagnostic build only).

    make -C watsor_b200/csrc -B EXTRA=-DWB_TRACE && gpurun -- python tools/trace_pipeline.py

Runs the backbone up to a chosen layer, then reads the clock64() stamps the last launch of the
kernel left (see WB_STAMP in tc_common.cuh) and prints them relative to the kernel start, in cycles.
"""
import ctypes
import sys

import numpy as np

sys.path.insert(0, '.')
from oracle.reference_build import MODEL_BLOB  # noqa: E402
from watsor_b200.engine import Engine  # noqa: E402

SLOTS, ITERS = 12, 64
GEMM = {0: 'tma_issue', 1: 'conv_full', 2: 'conv_done', 3: 'mma_ready', 4: 'mma_issued', 5: 'epi_start', 6: 'epi_done'}
FUSED = {0: 'halo_issue', 1: 'b_issue', 2: 'prod_halo', 3: 'prod_empty', 4: 'prod_done', 5: 'mma_ready',
         6: 'mma_issued', 7: 'epi_start', 8: 'epi_done'}


def dump(e, fn, names, start_kind, n_it):
    buf = (ctypes.c_longlong * (SLOTS * ITERS))()
    rc = getattr(e.lib, fn)(buf)
    assert rc == 0, rc
    t = np.array(buf, dtype=np.int64).reshape(SLOTS, ITERS)
    t0 = t[start_kind, 0]
    print('%-4s' % 'it' + ''.join('%11s' % names[k] for k in sorted(names)))
    for it in range(n_it):
        print('%-4d' % it + ''.join('%11d' % (t[k, it] - t0 if t[k, it] else -1) for k in sorted(names)))


def main():
    blob = open(MODEL_BLOB, 'rb').read()
    e = Engine(blob, max_batch=8, precision=2)
    pre = np.random.default_rng(0).uniform(-1, 1, (8, 300, 300, 3)).astype(np.float32)
    for rep in range(3):
        e.backbone(pre, stop_layer=2)
    print('== fused dw1+pw1 (layer 2)')
    dump(e, 'wb_trace_read_fused', FUSED, 9, 16)
    for rep in range(3):
        e.backbone(pre, stop_layer=6)
    print('== fused dw3+pw3 (layer 6)')
    dump(e, 'wb_trace_read_fused', FUSED, 9, 18)
    for rep in range(3):
        e.backbone(pre, stop_layer=14)
    print('== GEMM 512->512 at 19x19 (layer 14)')
    dump(e, 'wb_trace_read_gemm', GEMM, 7, 17)


main()
