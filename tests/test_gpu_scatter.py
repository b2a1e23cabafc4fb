"""The one collective on the path: the engine's frame scatter (BASELINE.json north star: "NCCL over NVLink only for
the engine's frame scatter").  Two ranks over NCCL on two GPUs: rank 0 owns every camera's frame of a tick and
scatters each rank's [C,H,W,3] u8 slab; every rank runs the detector on the receive buffer IN PLACE (device
pointers) and must get byte-identical Detection rows to running on its own local copy of the same frames.
Skipped on boxes with a single GPU (run it with `gpurun --gpus 2`)."""
import os
import socket
import sys

import numpy as np
import pytest

from tests.conftest import MODEL_BLOB, ROOT

pytestmark = pytest.mark.gpu


def free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def worker(rank, world, port, out):
    sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist

    from tests.artist import artist_frame
    from tests.gpu_util import new_rows, rows_bytes
    from watsor_b200.detection.b200 import B200ObjectDetector
    from watsor_b200.model import Model
    from watsor_b200.parallel import camera_shard, engine_scatter_frames, init_engine_comm, scatter_frames
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group('nccl', rank=rank, world_size=world, device_id=torch.device('cuda', rank))
    C, H, W = 4, 240, 320
    cams = camera_shard(rank, world, C)
    mine = np.stack([artist_frame(W, H, g, 0) for g in cams])
    per_rank = None
    if rank == 0:
        per_rank = [torch.from_numpy(np.stack([artist_frame(W, H, g, 0) for g in camera_shard(r, world, C)])).cuda()
                    for r in range(world)]
    recv = torch.empty((C, H, W, 3), dtype=torch.uint8, device='cuda')
    scatter_frames(recv, per_rank, src=0)
    torch.cuda.synchronize()
    same_bytes = bool((recv.cpu().numpy() == mine).all())
    with B200ObjectDetector(None, device=rank, max_batch=C, precision=2, model_blob=Model.load(MODEL_BLOB).to_blob()) as det:
        for c in range(C):
            det.configure_camera(c, W, H, None)
        a, b = new_rows(C), new_rows(C)
        det.detect_batch([recv[c].data_ptr() for c in range(C)], list(range(C)), a, fuse_filters=False,
                         frames_on_device=True)
        det.detect_batch([mine[c] for c in range(C)], list(range(C)), b, fuse_filters=False)
        same_rows = all(rows_bytes(x) == rows_bytes(y) for x, y in zip(a, b))
        found = sum(1 for rows in a for r in range(100) if rows[r].confidence > 0.5)
        # the same scatter through the C-ABI's own communicator (wb_comm_init / wb_scatter_frames): a second tick's
        # frames land in a fresh buffer and the batch submitted right after it is ordered behind the transfer
        init_engine_comm(det.engine, rank, world)
        mine2 = np.stack([artist_frame(W, H, g, 1) for g in cams])
        per_rank2 = None
        if rank == 0:
            per_rank2 = [torch.from_numpy(np.stack([artist_frame(W, H, g, 1) for g in camera_shard(r, world, C)])).cuda()
                         for r in range(world)]
        recv2 = torch.zeros((C, H, W, 3), dtype=torch.uint8, device='cuda')
        torch.cuda.synchronize()
        c_rows, d_rows = new_rows(C), new_rows(C)
        for _ in range(3):      # repeated ticks re-use the communicator and the receive buffer
            engine_scatter_frames(det.engine, recv2, per_rank2, root=0)
            det.detect_batch([recv2[c].data_ptr() for c in range(C)], list(range(C)), c_rows, fuse_filters=False,
                             frames_on_device=True)
        det.detect_batch([mine2[c] for c in range(C)], list(range(C)), d_rows, fuse_filters=False)
        torch.cuda.synchronize()
        same_bytes = same_bytes and bool((recv2.cpu().numpy() == mine2).all())
        same_rows = same_rows and all(rows_bytes(x) == rows_bytes(y) for x, y in zip(c_rows, d_rows))
        det.engine.comm_destroy()
    dist.barrier()
    out.put((rank, same_bytes, same_rows, found))
    dist.destroy_process_group()


@pytest.mark.skipif(not os.path.isfile(MODEL_BLOB), reason='oracle/_ref/ blob missing')
def test_two_rank_nccl_scatter_feeds_the_detector_in_place():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs (gpurun --gpus 2)')
    import torch.multiprocessing as mp
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = free_port()
    procs = [ctx.Process(target=worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=600) for _ in range(2))
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    assert all(r[1] and r[2] for r in res), res          # the slab arrived intact; in-place detection == local detection
    assert all(r[3] >= 4 for r in res), res              # and it detected the drawn shapes
