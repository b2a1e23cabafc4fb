#!/usr/bin/env python
"""bench.py -- aggregate detection FPS on synthetic 640x480 streams (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            our arm (B200, libwatsor_b200.so)
    python bench.py --impl reference --gpus N --steps K ...  CPU arm: the reference path's CPU
                                                             restatement (oracle/), all host threads

Default workload = BASELINE configs[2] to the letter (tests/workload.py): 8 cameras of 640x480 synthetic RGB
per GPU, batched, SSD-MobileNet-v2 300x300 with 90 COCO classes at the model-zoo score threshold 1e-8 (all
1917 anchors are NMS candidates in every class), a mask on every camera (camera 0 = the reference's porch.png,
cameras 1..7 synthetic RGBA masks), per-class filter defaults confidence 50 / area 10.  x8 GPUs = configs[3].

A step = one tick of the hot path over one batch: one frame from each of the C cameras a GPU serves, i.e.
resize+normalise -> SSD convs + heads -> decode -> per-class NMS -> top-100 -> integer conversion ->
confidence/area/mask-zone predicates -> Detection[100] per frame.

  value  device-timed throughput with frames already resident in HBM (ring of distinct frames per
         camera, larger than L2, so every step reads its input from HBM), exactly K steps
  e2e    same metric through the public detector API with HOST frames in pinned memory:
         H2D of every frame and D2H of every Detection block inside the timed region
  config.real_weights   the same two numbers on the only model with real weights (the reference's vendored
         3-class SSD-MobileNet-v1, watsor/test/model/cpu.pb), porch mask on camera 0
  e2e_worker   the same metric through the drop-in worker process (watsor_b200.detection.detector.ObjectDetector
         under `spawn`, frames in multiprocessing shared memory, payloads through a Queue)
  effects      auxiliary (not the headline): the output stage's effect chain -- BlendEffect +
         DrawEffectWithContours -- for the same cameras as one wb_fx_render per tick (SURVEY.md 8 (f)4)
Multi-GPU: one process per GPU (torchrun), cameras sharded, no data-path collective (weak scaling); the
N>1 line adds a `scatter` record: the same steps with the NCCL frame scatter from rank 0 that BASELINE.json's
north star names, through the library's own collective (wb_comm_init / wb_scatter_frames; --scatter-impl torch
runs torch.distributed.scatter instead).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = 'aggregate detection FPS on synthetic 640x480 streams'
UNIT = 'frames/s'
W, H = 640, 480
L2_BYTES = 126 * 1024 * 1024
# watsor_b200.stream.share.Detection (72 bytes, include/watsor_b200.h: wb_detection)
DETECTION_DTYPE = np.dtype({'names': ['label', 'zones', 'confidence', 'box'],
                            'formats': ['<i4', ('<i4', (10,)), '<f8', ('<i4', (4,))],
                            'offsets': [0, 4, 48, 56], 'itemsize': 72})


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument('--gpus', type=int, default=1)
    p.add_argument('--steps', type=int, default=1000)
    p.add_argument('--warmup', type=int, default=20)
    p.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    p.add_argument('--cameras', type=int, default=8, help='cameras (= batch) per GPU')
    p.add_argument('--model', default='v2', choices=['v2', 'coco', 'shapes', 'inception'],
                   help='v2: SSD-MobileNet-v2, 90 classes (BASELINE configs[2], default); coco: SSD-MobileNet-v1 '
                        'backbone, 90-class heads; shapes: vendored 3-class SSD-MobileNet-v1 (real weights); '
                        'inception: SSD-Inception-v2, 90 classes, 1920x1080 frames (BASELINE configs[4]; use --cameras 2)')
    p.add_argument('--precision', default='tf32x3', choices=['fp32', 'tf32x3', 'bf16'],
                   help='fp32: CUDA-core FFMA convs; tf32x3: fp32-faithful tcgen05 (3xTF32 split); bf16: tcgen05 bf16')
    p.add_argument('--frames', default='artist', choices=['artist', 'random'])
    p.add_argument('--ingest', default='local', choices=['local', 'scatter'])
    p.add_argument('--inflight', type=int, default=6, help='batches kept in flight (library slots, max 6)')
    p.add_argument('--no-cpu-baseline', action='store_true')
    p.add_argument('--no-roofline', action='store_true')
    p.add_argument('--no-real-weights', action='store_true', help='skip the second (real-weights v1) record')
    p.add_argument('--no-scatter', action='store_true', help='skip the NCCL scatter record at N>1')
    p.add_argument('--scatter-impl', default='cabi', choices=['cabi', 'torch'],
                   help="cabi: the library's own communicator (wb_comm_init / wb_scatter_frames); torch: "
                        'torch.distributed.scatter')
    p.add_argument('--no-worker', action='store_true', help='skip the e2e_worker record')
    p.add_argument('--no-effects', action='store_true', help='skip the visual-effects record')
    p.add_argument('--min-seconds', type=float, default=1.0,
                   help='the *_long / e2e measurements run at least this long')
    p.add_argument('--dump-outputs', metavar='DIR',
                   help='write what the last of the K timed steps returned (Detection rows and filter verdicts of '
                        'every camera) to DIR/<name>.npy, as float64, to compare two builds output for output')
    args = p.parse_args()
    if args.dump_outputs and args.impl == 'reference':
        # the CPU arm times a few frames of the batch per step, so it has no per-step batch output to compare
        p.error('--dump-outputs writes the outputs of the b200 arm; it cannot be combined with --impl reference')
    return args


# ------------------------------------------------------------------------------------------ inputs
def load_model(kind):
    from watsor_b200.model import Model, synthetic_ssd_mobilenet_v1
    from tests.workload import v2_coco_model
    blob = os.path.join(ROOT, 'oracle', '_ref', 'ssd_mobilenet_v1_shapes', 'b200.wb200')
    if kind == 'shapes' and os.path.isfile(blob):
        return Model.load(blob), 'ssd_mobilenet_v1 300x300, 3 classes, real weights (watsor/test/model/cpu.pb)'
    if kind == 'shapes':
        return (synthetic_ssd_mobilenet_v1(num_classes=3, seed=1, score_thr=0.3),
                'ssd_mobilenet_v1 300x300, 3 classes, seeded synthetic weights (vendored blob missing)')
    if kind == 'inception':
        from watsor_b200.model import synthetic_ssd_inception_v2
        return (synthetic_ssd_inception_v2(num_classes=90, seed=0, score_thr=1e-8),
                'ssd_inception_v2 300x300, 90 classes, score threshold 1e-8, seeded synthetic weights')
    if kind == 'v2':
        return (v2_coco_model(),
                'ssd_mobilenet_v2 300x300, 90 classes, score threshold 1e-8, seeded synthetic weights '
                '(no v2 weights exist offline)')
    return (synthetic_ssd_mobilenet_v1(num_classes=90, seed=0, score_thr=1e-8),
            'ssd_mobilenet_v1 300x300, 90-class heads, seeded synthetic weights')


def set_frame_size(args):
    """configs[4] (SSD-Inception-v2) is quoted on 1920x1080 streams; everything else on 640x480."""
    global W, H
    if args.model == 'inception':
        W, H = 1920, 1080


def make_frames(kind, cam, count):
    from tests.artist import artist_frame
    if kind == 'artist':
        return [artist_frame(W, H, cam, f) for f in range(count)]
    rng = np.random.default_rng(cam)
    return [rng.integers(0, 256, (H, W, 3), dtype=np.uint8) for _ in range(count)]


def camera_config(cam, model_kind):
    """configs[2]: a mask on every camera, schema-default thresholds for every COCO label.  The 3-class
    real-weights model keeps round 1's configuration (its labels 1..3 are person/bicycle/car ids)."""
    from tests import workload
    if model_kind == 'inception':
        return workload.camera_config(cam % 8, W, H)
    if model_kind == 'shapes':
        detect = [{'person': {'confidence': 50, 'area': 1, 'zones': []}},
                  {'bicycle': {'confidence': 50, 'area': 1, 'zones': []}},
                  {'car': {'confidence': 50, 'area': 10, 'zones': []}}]
        cfg = {'width': W, 'height': H, 'detect': detect}
        if cam == 0 and os.path.isfile(workload.PORCH):
            cfg['mask'] = workload.PORCH
        return cfg
    return workload.camera_config(cam % 8)


def workload_name(args):
    if args.model == 'inception':
        return ('BASELINE configs[4] per GPU: %d cameras x 1920x1080 synthetic RGB, batched, SSD-Inception-v2 300x300, '
                '90-class NMS at score threshold 1e-8, a synthetic RGBA mask on every camera, per-class defaults '
                'confidence 50 / area 10 (16 cameras on 8 GPUs = 2 per GPU)' % args.cameras)
    if args.model == 'shapes':
        return ('%d cameras x 640x480 synthetic RGB per GPU, batched, SSD-MobileNet-v1 300x300 (3 classes, real '
                'weights), per-camera confidence/area filters + porch.png mask zones on camera 0' % args.cameras)
    return ('BASELINE configs[2]: %d cameras x 640x480 synthetic RGB per GPU, batched, %s 300x300, 90-class NMS at '
            'score threshold 1e-8, a mask on every camera (cam 0 porch.png, others synthetic RGBA), per-class '
            'defaults confidence 50 / area 10 (x8 GPUs = configs[3])'
            % (args.cameras, 'SSD-MobileNet-v2' if args.model == 'v2' else 'SSD-MobileNet-v1'))


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
         'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(',')]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'], f[5:9]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(smax) if smax else None,
                'power_w_max': max(power) if power else None, 'samples': len(sm), 'reasons': sorted(reasons)}


# --------------------------------------------------------------------------------- reference arm
def oracle_step_fn(model, args):
    """The CPU restatement of the reference path for one frame: graph arithmetic
    (oracle/ssd_model.py) + tensorflow_cpu.py:79-90 conversion + the predicate chain."""
    import torch

    from oracle.filters import AreaOracle, ConfidenceOracle, Det, MaskOracle, apply_predicates
    from oracle.ssd_graph import to_detections
    from oracle.ssd_model import SsdModelOracle
    oracle = SsdModelOracle(model)
    # "all the host threads it can use": torch's intra-op pool thrashes on MobileNet-sized convs when
    # given every hardware thread of a big host (128 threads: 17 s/frame), so the thread count is
    # calibrated on one frame and the fastest setting is used and reported
    probe = make_frames('artist', 0, 1)[0]
    host = os.cpu_count() or 1
    best = None
    for nt in sorted({min(host, c) for c in (8, 16, 32, 64)}):
        torch.set_num_threads(nt)
        oracle.run(probe)
        t0 = time.perf_counter()
        oracle.run(probe)
        dt = time.perf_counter() - t0
        if best is None or dt < best[0]:
            best = (dt, nt)
        if dt > 3.0:
            break
    torch.set_num_threads(best[1])
    filt = {}

    def filters_for(cam):
        if cam not in filt:
            cfg = camera_config(cam, args.model)
            fs = [ConfidenceOracle(cfg), AreaOracle(cfg)]
            if 'mask' in cfg:
                fs.append(MaskOracle(cfg))
            filt[cam] = fs
        return filt[cam]

    def run(img, cam):
        b, cl, s, n = oracle.run(img)
        rows = to_detections(b, cl, s, img.shape)
        dets = [Det(r[0], r[1], tuple(r[2:])) for r in rows]
        apply_predicates(dets, filters_for(cam))
        return n
    return run, best[1], host


def run_reference(args, rank):
    if rank != 0:
        return
    model, model_desc = load_model(args.model)
    run, cores, host_cores = oracle_step_fn(model, args)
    cams = args.cameras
    frames = [make_frames(args.frames, c, 2) for c in range(cams)]
    t0 = time.perf_counter()
    run(frames[0][0], 0)
    run(frames[0][1], 0)
    per_frame = (time.perf_counter() - t0) / 2
    budget = 150.0
    per_step = max(1, min(cams, int(budget / max(1e-3, per_frame * (args.steps + args.warmup)))))
    k = 0

    def step():
        nonlocal k
        for i in range(per_step):
            c = (k + i) % cams
            run(frames[c][(k // cams) % 2], c)
        k += per_step
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    fps = per_step * args.steps / dt
    sample = '%d frame(s) of the %d-camera batch per step, %d steps' % (per_step, cams, args.steps)
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': fps, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': 1e3 * dt / args.steps, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': workload_name(args), 'model': model_desc, 'frames': args.frames,
                   'note': 'CPU restatement of the reference TF graph + watsor filters (oracle/), not TensorFlow: '
                           'TensorFlow is not installable offline'},
        'cpu_baseline': {'value': fps, 'unit': UNIT, 'cores': cores, 'host_cores': host_cores, 'kind': 'port',
                         'sample': sample},
        'e2e': {'value': fps, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------- our arm
class Arm:
    """One detector (model + camera tables) on this rank's GPU plus its input rings, and the two timed loops."""

    def __init__(self, args, model_kind, rank, local_rank, world, torch, dist):
        from watsor_b200.detection.b200 import B200ObjectDetector
        from watsor_b200.parallel import camera_shard
        from watsor_b200.stream.share import Detection
        self.args, self.rank, self.world, self.torch, self.dist = args, rank, world, torch, dist
        self.model_kind = model_kind
        self.model, self.model_desc = load_model(model_kind)
        self.C = C = args.cameras
        self.precision = {'fp32': 0, 'bf16': 1, 'tf32x3': 2}[args.precision]
        self.det = B200ObjectDetector(None, device=local_rank, max_batch=C, precision=self.precision,
                                      model_blob=self.model.to_blob())
        for c in range(C):
            self.det.configure_camera(c, W, H, camera_config(c, model_kind))
        self.cam_ids = list(range(C))
        # input ring: distinct frames per camera, total > L2, so each step's input comes from HBM
        self.frame_bytes = W * H * 3
        self.ring = ring = max(4, -(-int(1.4 * L2_BYTES) // (C * self.frame_bytes)))
        self.base = [make_frames(args.frames, g, min(ring, 6)) for g in camera_shard(rank, world, C)]
        self.host_ring = torch.empty((ring, C, H, W, 3), dtype=torch.uint8).pin_memory()
        rng = np.random.default_rng(1234 + rank)
        for r in range(ring):
            for c in range(C):
                img = self.base[c][r % len(self.base[c])]
                if r >= len(self.base[c]):          # distinct bytes per ring slot: roll the picture a little
                    img = np.roll(img, shift=int(rng.integers(1, 40)), axis=1)
                self.host_ring[r, c] = torch.from_numpy(np.ascontiguousarray(img))
        self.dev_ring = self.host_ring.cuda()
        torch.cuda.synchronize()
        self.NS = NS = max(1, min(6, args.inflight))
        self.out_rows = [[(Detection * 100)() for _ in range(C)] for _ in range(NS)]
        self.out_verd = [[np.zeros(100, np.uint32) for _ in range(C)] for _ in range(NS)]
        self.stream = torch.cuda.Stream()
        self.scatter_buf = None
        self.scatter_events = []
        self.comm_ready = False

    def close(self):
        self.det.engine.close()

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def reduce_max(self, x):
        from watsor_b200.parallel import max_over_ranks
        return max_over_ranks(x, device='cuda')

    # ---- device-resident frames (optionally delivered by the NCCL scatter from rank 0)
    def enable_scatter(self):
        torch = self.torch
        self.scatter_buf = [torch.empty((self.C, H, W, 3), dtype=torch.uint8, device='cuda') for _ in range(self.NS)]
        if self.rank == 0:
            self.all_ring = [self.dev_ring.clone() for _ in range(self.world)]
        if self.args.scatter_impl == 'cabi' and not self.comm_ready:
            from watsor_b200.parallel import init_engine_comm
            init_engine_comm(self.det.engine, self.rank, self.world)
            self.comm_ready = True

    def dev_ptrs(self, step, slot, time_scatter=False):
        from watsor_b200.parallel import engine_scatter_frames
        from watsor_b200.parallel import scatter_frames as torch_scatter_frames
        if self.args.scatter_impl == 'cabi':
            def scatter_frames(recv, per_rank, src=0):
                engine_scatter_frames(self.det.engine, recv, per_rank, root=src, cuda_stream=self.stream.cuda_stream)
        else:
            scatter_frames = torch_scatter_frames
        r = step % self.ring
        if self.scatter_buf is not None:
            # the engine's frame scatter: rank 0 owns every camera's frame and NCCL-scatters each rank's
            # batch over NVLink; slot `slot` was collected before, so its buffer is free to overwrite
            src = [self.all_ring[g][r] for g in range(self.world)] if self.rank == 0 else None
            if time_scatter:
                e0, e1 = self.torch.cuda.Event(enable_timing=True), self.torch.cuda.Event(enable_timing=True)
                e0.record(self.stream)
                scatter_frames(self.scatter_buf[slot], src, src=0)
                e1.record(self.stream)
                self.scatter_events.append((e0, e1))
            else:
                scatter_frames(self.scatter_buf[slot], src, src=0)
            self.det.engine.stream_fence(self.stream.cuda_stream, 0)
            return [self.scatter_buf[slot][c].data_ptr() for c in range(self.C)]
        return [self.dev_ring[r, c].data_ptr() for c in range(self.C)]

    def run_device_steps(self, n_steps, first, time_scatter=False):
        det, NS = self.det, self.NS
        for i in range(n_steps):
            s = i % NS
            if i >= NS:
                det.collect(s, self.out_rows[s], self.out_verd[s])
            det.submit(s, self.dev_ptrs(first + i, s, time_scatter), self.cam_ids, fuse_filters=True,
                       frames_on_device=True)
        for i in range(max(0, n_steps - NS), n_steps):
            det.collect(i % NS, self.out_rows[i % NS], self.out_verd[i % NS])

    def outputs(self, slot):
        """What a caller of submit/collect received for the batch collected into `slot`, one row per camera: the
        Detection[100] block field by field and the filter verdict bits, as float64 arrays (exact for every field)."""
        rows = np.stack([np.frombuffer(bytes(r), dtype=DETECTION_DTYPE) for r in self.out_rows[slot]])
        return {'detection_label': rows['label'], 'detection_zones': rows['zones'],
                'detection_confidence': rows['confidence'], 'detection_box': rows['box'],
                'filter_verdicts': np.stack(self.out_verd[slot])}

    def time_device(self, steps, first):
        """CUDA events on a torch stream fenced against the library's slot streams on both sides; max over ranks.
        The wall clock stops before the closing barrier (the NCCL barrier is not part of the loop)."""
        torch = self.torch
        self.barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_wall0 = time.perf_counter()
        ev0.record(self.stream)
        self.det.engine.stream_fence(self.stream.cuda_stream, 0)
        self.run_device_steps(steps, first, time_scatter=self.scatter_buf is not None)
        self.det.engine.stream_fence(self.stream.cuda_stream, 1)
        ev1.record(self.stream)
        torch.cuda.synchronize()
        t_wall = time.perf_counter() - t_wall0
        self.barrier()
        dev_ms = self.reduce_max(ev0.elapsed_time(ev1))
        return dev_ms, t_wall

    # ---- host frames in pinned memory through the public API
    def run_host_steps(self, n_steps, first):
        det, NS = self.det, self.NS
        for i in range(n_steps):
            s = i % NS
            if i >= NS:
                det.collect(s, self.out_rows[s], self.out_verd[s])
            r = (first + i) % self.ring
            det.submit(s, [self.host_ring[r, c].data_ptr() for c in range(self.C)], self.cam_ids, fuse_filters=True,
                       frames_on_device=False)
        for i in range(max(0, n_steps - NS), n_steps):
            det.collect(i % NS, self.out_rows[i % NS], self.out_verd[i % NS])

    def time_host(self, steps, first):
        self.barrier()
        t0 = time.perf_counter()
        self.run_host_steps(steps, first)
        self.torch.cuda.synchronize()
        return self.reduce_max(time.perf_counter() - t0)

    def measure(self, want_long=True):
        """-> dict with value / e2e (+ *_long when the K-step region is shorter than --min-seconds)."""
        args, world, C = self.args, self.world, self.C
        self.torch.cuda.set_stream(self.stream)
        warm = max(self.NS, args.warmup)
        # prime: CUDA graphs of all slots instantiated, clocks and the L2 in their steady state (a 20-step timed region
        # is ~10 ms: a cold start shows up as a 25 % lower number); then the W warm-up steps proper
        t_prime, primed = time.perf_counter(), 0
        while time.perf_counter() - t_prime < 0.3:
            self.run_device_steps(2 * self.NS, primed)
            primed += 2 * self.NS
        self.prime_steps = primed
        if world > 1:
            # ranks finish priming at different times (process start-up differs by 100s of ms); without this the early
            # ranks would sit idle in the timed region's opening barrier, clock down, and the maximum over ranks of a
            # short K-step region would measure their ramp-up.  Aligned here, the W warm-up steps below run on every
            # rank right before that barrier, which then costs microseconds.
            self.barrier()
        self.run_device_steps(warm, 0)
        launches = self.det.engine.last_launch_count()
        dev_ms, t_wall = self.time_device(args.steps, args.warmup)
        self.last_outputs = self.outputs((args.steps - 1) % self.NS)
        out = {'value': world * C * args.steps / (dev_ms / 1e3), 'ms_per_step': dev_ms / args.steps,
               'launches_per_step': launches, 'wall_ms_per_step_device_loop': 1e3 * t_wall / args.steps,
               'prime_steps': self.prime_steps,
               'detections_per_frame': float(np.mean([sum(1 for r in range(100) if rows[r].confidence > 0)
                                                      for rows in self.out_rows[0]])),
               'passed_filters_per_frame': float(np.mean([int(np.count_nonzero(v & 16)) for v in self.out_verd[0]]))}
        long_steps = int(min(20000, max(args.steps, args.min_seconds * 1e3 / max(1e-3, out['ms_per_step']))))
        if want_long and long_steps > args.steps:
            ms, _ = self.time_device(long_steps, args.warmup + args.steps)
            out['value_long'] = {'value': world * C * long_steps / (ms / 1e3), 'steps': long_steps,
                                 'ms_per_step': ms / long_steps}
        self.run_host_steps(warm, 0)
        e2e_s = self.time_host(args.steps, args.warmup)
        out['e2e_k'] = {'value': world * C * args.steps / e2e_s, 'steps': args.steps,
                        'ms_per_step': 1e3 * e2e_s / args.steps}
        e2e_steps = int(min(20000, max(args.steps, args.min_seconds / max(1e-6, e2e_s / args.steps))))
        if want_long and e2e_steps > args.steps:
            e2e_s = self.time_host(e2e_steps, args.warmup + args.steps)
        else:
            e2e_steps = args.steps
        out['e2e'] = {'value': world * C * e2e_steps / e2e_s, 'unit': UNIT, 'h2d_bytes_per_step': C * self.frame_bytes,
                      'd2h_bytes_per_step': C * 100 * (72 + 4), 'ms_per_step': 1e3 * e2e_s / e2e_steps,
                      'steps': e2e_steps,
                      'api': 'watsor_b200.detection.b200.B200ObjectDetector.submit/collect (%d slots in flight), '
                             'wall clock between barriers, max over ranks; timed over max(K, %.1f s) steps, '
                             'the K-step figure is e2e_k' % (self.NS, args.min_seconds)}
        return out

    def measure_scatter(self, ms_per_step):
        """The same device loop with every tick's frames NCCL-scattered from rank 0 (north star: 'NCCL over
        NVLink only for the engine's frame scatter')."""
        args, world, C = self.args, self.world, self.C
        self.enable_scatter()
        self.run_device_steps(max(self.NS, args.warmup), 0)
        steps = int(min(5000, max(args.steps, 0.5e3 / max(1e-3, ms_per_step))))   # >= 0.5 s
        self.scatter_events = []
        dev_ms, _ = self.time_device(steps, args.warmup)
        us = [1e3 * a.elapsed_time(b) for a, b in self.scatter_events]
        rec = {'value': world * C * steps / (dev_ms / 1e3), 'steps': steps, 'ms_per_step': dev_ms / steps,
               'nvlink_bytes_per_tick': (world - 1) * C * self.frame_bytes,
               'scatter_us_median': float(np.median(us)) if us else None,
               'scatter_us_p90': float(np.percentile(us, 90)) if us else None,
               'collective': ('wb_scatter_frames (C-ABI; grouped ncclSend/ncclRecv on the library\'s own communicator)'
                              if args.scatter_impl == 'cabi' else
                              'torch.distributed.scatter (ncclScatter: grouped send/recv)') +
                             ' of [C,H,W,3] u8 per rank from rank 0; the kernels read the receive buffer in place'}
        self.scatter_buf = None
        return rec


def main():
    args = parse_args()
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    set_frame_size(args)
    if args.impl == 'reference':
        run_reference(args, rank)
        return

    # NUMA: bind this rank to the CPUs next to its GPU before any pinned allocation or thread creation
    from watsor_b200.parallel import bind_to_gpu_numa
    numa = bind_to_gpu_numa(local_rank)

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit('bench.py --impl b200 needs a B200; there is no CPU fallback')
    # with several batches in flight the persistent GEMM should not pin every SM: leaving ~20 % of them to the
    # other streams' kernels measured +4 % (148 -> 116 CTAs); single-stream users keep the default (all SMs)
    os.environ.setdefault('WB_PERSIST_CTAS', '116')
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))

    sampler = ClockSampler(local_rank)
    sampler.start()
    arm = Arm(args, args.model, rank, local_rank, world, torch, dist)
    if args.ingest == 'scatter' and world > 1:
        arm.enable_scatter()
    m = arm.measure()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, arm.last_outputs, rank if world > 1 else None)
    scatter = None
    if world > 1 and args.ingest == 'local' and not args.no_scatter:
        scatter = arm.measure_scatter(m['ms_per_step'])
        scatter['vs_local_ingest'] = scatter['value'] / (m.get('value_long') or m)['value']
    # keep the GPU loaded until nvidia-smi has a few samples (its first line takes ~0.3 s)
    t_load = time.perf_counter()
    extra = 0
    while time.perf_counter() - t_load < 1.0:
        arm.run_host_steps(20, 0)
        extra += 20
    clocks = sampler.stop()
    clocks['window'] = 'warm-up + every timed loop of the headline model + %d extra e2e steps (100 ms period)' % extra

    # ---------------- roofline of the dominant kernel + per-layer times (rank 0)
    roofline = None
    layer_table = None
    if rank == 0 and not args.no_roofline:
        roofline, layer_table = measure_roofline(arm.det, arm.model, arm.dev_ring, arm.C, arm.cam_ids, arm.precision)

    worker = None
    if rank == 0 and not args.no_worker:
        worker = measure_worker(args, local_rank, m)

    effects = None
    if rank == 0 and world == 1 and not args.no_effects:
        effects = measure_effects(args, local_rank, torch)

    cpu_baseline = None
    if rank == 0 and not args.no_cpu_baseline:
        run, cores, host_cores = oracle_step_fn(arm.model, args)
        C = arm.C
        pool = [(arm.base[c][f], c) for f in range(2) for c in range(C)]
        run(*pool[0])
        t0 = time.perf_counter()
        done = 0
        while done < 2000 and (time.perf_counter() - t0 < 12.0 or done < 4):
            run(*pool[done % len(pool)])
            done += 1
        dt = time.perf_counter() - t0
        cpu_baseline = {'value': done / dt, 'unit': UNIT, 'cores': cores, 'host_cores': host_cores,
                        'kind': 'port',
                        'sample': '%d frames (cycling the first ring slots of the %d cameras), batch 1, %.1f s of CPU work, torch threads calibrated; '
                                  'CPU restatement of the reference TF graph (oracle/), not TensorFlow'
                                  % (done, C, dt)}
    arm.close()

    # ---------------- second record: the only model with real weights (round 1's headline configuration)
    real = None
    if args.model not in ('shapes', 'inception') and not args.no_real_weights:
        arm2 = Arm(args, 'shapes', rank, local_rank, world, torch, dist)
        r = arm2.measure()
        real = {'model': arm2.model_desc, 'workload': 'same frames; porch.png mask on camera 0, 3 labels',
                'value': r['value'], 'ms_per_step': r['ms_per_step'], 'value_long': r.get('value_long'),
                'e2e': r['e2e']['value'], 'e2e_steps': r['e2e']['steps'], 'launches_per_step': r['launches_per_step'],
                'detections_per_frame': r['detections_per_frame']}
        arm2.close()

    if rank == 0:
        C = args.cameras
        line = {
            'metric': METRIC, 'value': m['value'], 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': m['ms_per_step'], 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'bf16' if arm.precision == 1 else 'f32', 'data': 'synthetic',
            'config': {
                'workload': workload_name(args), 'cameras_per_gpu': C, 'global_batch': world * C,
                'frame': '%dx%dx3 u8' % (W, H), 'model': arm.model_desc, 'frames': args.frames, 'ingest': args.ingest,
                'num_classes': arm.model.num_classes, 'score_threshold': arm.model.score_thr,
                'masks': 'one per camera (cam 0: porch.png, 2 zones; cams 1..%d: synthetic RGBA, 1 + cam %% 4 zones)'
                         % (C - 1) if args.model != 'shapes' else 'porch.png on camera 0',
                'camera_to_gpu': 'camera c -> rank c // %d (contiguous blocks; BASELINE.md suggests c mod G, '
                                 'equivalent for independent cameras)' % C,
                'precision': args.precision, 'batches_in_flight': arm.NS,
                'persistent_gemm_ctas': int(os.environ.get('WB_PERSIST_CTAS', '0')),
                'l2': 'input ring of %d distinct frames per camera (%.0f MB per GPU) > 126 MB L2; no flush needed'
                      % (arm.ring, arm.ring * C * arm.frame_bytes / 1e6),
                'detections_per_frame': m['detections_per_frame'],
                'passed_filters_per_frame': m['passed_filters_per_frame'],
                'wall_ms_per_step_device_loop': m['wall_ms_per_step_device_loop'],
                'prime_steps_before_warmup': m['prime_steps'],
                'numa': numa,
                'real_weights': real,
                'per_layer_ms': layer_table,
            },
            'value_long': m.get('value_long'),
            'e2e': m['e2e'],
            'e2e_k': m['e2e_k'],
            'e2e_worker': worker,
            'effects': effects,
            'scatter': scatter,
            'gpu_launches': m['launches_per_step'] * args.steps,
            'gpu_launches_per_step': m['launches_per_step'],
            'clocks': clocks,
            'roofline': roofline,
            'cpu_baseline': cpu_baseline,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out_dir, arrays, rank=None):
    """DIR/<name>.npy per array (DIR/<name>_rank<r>.npy with several ranks), float64."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        if rank is not None:
            name = '%s_rank%d' % (name, rank)
        np.save(os.path.join(out_dir, name + '.npy'), np.ascontiguousarray(a, dtype=np.float64))


def measure_effects(args, local_rank, torch):
    """Auxiliary record (SURVEY.md 8 (f)4, not part of the headline): the output stage's effect chain of main.py:302-312
    -- BlendEffect + DrawEffectWithContours -- for the same 8 masked cameras as one `wb_fx_render` per tick, with 8
    labelled detections per frame.  `value`: frames resident on the device, kernels only (CUDA events inside the
    library); `e2e`: host frames in, host frames out, wall clock.  HBM roofline: 3 B read + 3 B written per pixel
    plus the alpha channel (1 B) and the zone-outline raster (4 B)."""
    try:
        from tests.fx_cases import random_rows
        from watsor_b200.filter.mask import get_alpha_channel
        from watsor_b200.output.effects import (WB_FX_BLEND, WB_FX_CONTOURS, WB_FX_DRAW, WB_FX_ON_DEVICE,
                                                EffectsEngine, contour_bits)
        C = args.cameras
        rng = np.random.default_rng(3)
        t0 = time.perf_counter()
        eng = EffectsEngine(local_rank)
        init_s = time.perf_counter() - t0
        cams, rows, imgs = [], [], []
        for c in range(C):
            cfg = camera_config(c, args.model)
            alpha = cont = None
            if 'mask' in cfg:
                alpha, _ = get_alpha_channel(cfg['mask'], W, H)
                cont = contour_bits(alpha)
            cams.append(eng.add_camera(W, H, alpha, cont))
            rows.append(random_rows(rng, W, H, 8, n_zones=1))
            imgs.append(make_frames(args.model, c, 1)[0])
        flags = WB_FX_BLEND | WB_FX_DRAW | WB_FX_CONTOURS
        d_in = [torch.from_numpy(np.ascontiguousarray(i)).cuda() for i in imgs]
        d_out = [torch.empty_like(t) for t in d_in]
        torch.cuda.synchronize()
        pin, pout = [t.data_ptr() for t in d_in], [t.data_ptr() for t in d_out]
        for _ in range(5):
            eng.render(pin, pout, cams, rows, flags | WB_FX_ON_DEVICE)
        ms = [eng.render(pin, pout, cams, rows, flags | WB_FX_ON_DEVICE) for _ in range(200)]
        med = float(np.median(ms))
        # host frames in pinned memory, like the shared frame buffers the worker registers (wb_register_host)
        pinned_in = [torch.from_numpy(np.ascontiguousarray(i)).pin_memory() for i in imgs]
        pinned_out = [torch.empty_like(t).pin_memory() for t in pinned_in]
        imgs, outs = [t.numpy() for t in pinned_in], [t.numpy() for t in pinned_out]
        for _ in range(3):
            eng.render(imgs, outs, cams, rows, flags)
        t0 = time.perf_counter()
        reps = 30
        for _ in range(reps):
            eng.render(imgs, outs, cams, rows, flags)
        wall = (time.perf_counter() - t0) / reps
        eng.close()
        alg = C * W * H * 11
        peak = 6650.0
        pk = os.path.join(ROOT, 'MEASURED_PEAKS.json')
        if os.path.isfile(pk):
            peak = json.load(open(pk)).get('hbm_gbs', peak)
        rec = {'value': C / (med / 1e3), 'unit': 'frames/s', 'ms_per_tick': med, 'frames_per_tick': C,
               'drawn_detections_per_frame': 8, 'chain': 'BlendEffect + DrawEffectWithContours (CopyImageEffect + '
               'DrawEffect on cameras without a mask), one wb_fx_render per tick',
               'algorithmic_bytes_per_tick': alg, 'achieved_gbps': alg / (med / 1e3) / 1e9,
               'e2e': {'value': C / wall, 'unit': 'frames/s', 'h2d_bytes_per_tick': C * W * H * 3 + C * 7200,
                       'd2h_bytes_per_tick': C * W * H * 3}, 'engine_init_s': init_s}
        if peak:
            rec['hbm_frac'] = rec['achieved_gbps'] / peak
        return rec
    except Exception as e:          # auxiliary: never takes the headline down
        return {'error': '%s: %s' % (type(e).__name__, e)}


def measure_worker(args, local_rank, headline):
    """e2e through the drop-in worker (watsor_b200.detection.detector.ObjectDetector) on multiprocessing shared
    frames; implemented in watsor_b200/bench_worker.py when present."""
    try:
        from watsor_b200.bench_worker import run_worker_bench
    except ImportError:
        return None
    try:
        return run_worker_bench(args, local_rank, camera_config, load_model, make_frames, width=W, height=H)
    except Exception as e:          # the headline number must not die with the auxiliary one
        return {'error': '%s: %s' % (type(e).__name__, e)}


def measure_roofline(det, model, dev_ring, C, cam_ids, precision):
    """Per-layer CUDA-event times (un-graphed run, median of 5) -> the kernel family with the largest
    share of the step is the dominant kernel; its roofline uses SURVEY.md 8(d) algorithmic FLOPs/bytes."""
    from watsor_b200.model import OP_ADD, OP_CONV, OP_DW, OP_HEAD, OP_NAMES, OP_PW, OP_STEM
    runs = []
    for rep in range(6):
        ptrs = [dev_ring[rep % dev_ring.shape[0], c].data_ptr() for c in range(C)]
        runs.append(det.engine.profile_layers(ptrs, cam_ids))
    ms = np.median(np.array([[t for _, t in r] for r in runs[1:]]), axis=0)
    kinds = [k for k, _ in runs[0]]
    elem = 2 if precision == 1 else 4
    fam = {}
    table = []
    for i, (k, t) in enumerate(zip(kinds, ms)):
        if k == 100:
            name, flops, byts = 'post', 0.0, C * (model.num_anchors * (5 + model.num_classes) * 4 + 7200.0)
        else:
            l = model.layers[i]
            name = OP_NAMES[k]
            flops = 2.0 * l.macs * C
            w_bytes = 4.0 * l.kh * l.kw * (l.in_c if k != OP_DW else 1) * l.out_c
            in_b = (W * H * 3) if k == OP_STEM else l.in_h * l.in_w * l.in_c * elem * (2 if k == OP_ADD else 1)
            out_b = l.out_h * l.out_w * l.out_c * (4 if k == OP_HEAD else elem)
            byts = C * (in_b + out_b) + w_bytes
            if k in (OP_PW, OP_CONV, OP_HEAD):
                name = 'gemm'
        f = fam.setdefault(name, {'ms': 0.0, 'flops': 0.0, 'bytes': 0.0, 'launches': 0})
        f['ms'] += float(t)
        f['flops'] += flops
        f['bytes'] += byts
        if float(t) > 0:
            f['launches'] += 1 if k != 100 else 3
        table.append([name if k == 100 else model.layers[i].name[-28:], round(float(t), 4)])
    total = sum(f['ms'] for f in fam.values())
    dom = max(fam, key=lambda n: fam[n]['ms'])
    d = fam[dom]
    peaks = {}
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.isfile(p):
        peaks = json.load(open(p))
    hbm = peaks.get('hbm_gbs', 6650.0)
    tf = peaks.get('bf16_tflops_sustained', 1400.0)
    src = 'measured (MEASURED_PEAKS.json)' if peaks else 'fallback (B200_PROFILING.md)'
    if dom == 'gemm':
        ach = d['flops'] / (d['ms'] / 1e3) / 1e12
        roof = {'bound': 'tensor', 'achieved': ach, 'peak': tf, 'unit': 'TFLOP/s', 'frac': ach / tf}
    else:
        ach = d['bytes'] / (d['ms'] / 1e3) / 1e9
        roof = {'bound': 'hbm', 'achieved': ach, 'peak': hbm, 'unit': 'GB/s', 'frac': ach / hbm}
    # DRAM bytes per launch of the dominant family from the committed ncu --set full capture of this model
    # (profiles/r02_traffic.json: {model name: {precision: {family: {dram_bytes_per_launch}}}}), batch 8 only
    traffic = None
    prec_name = {0: 'fp32', 1: 'bf16', 2: 'tf32x3'}[precision]
    tp = os.path.join(ROOT, 'profiles', 'r02_traffic.json')
    if os.path.isfile(tp) and C == 8:
        t = json.load(open(tp)).get(model.name, {}).get(prec_name, {}).get(dom)
        if t:
            traffic = t['dram_bytes_per_launch']
    roof.update({'traffic': traffic, 'traffic_unit': 'bytes of DRAM read+write per launch (ncu capture in profiles/, batch 8)',
                 'algorithmic_bytes_per_launch': d['bytes'] / max(1, d['launches']),
                 'kernel': {'gemm': 'tcgen05 GEMM family: k_gemm_tc / k_gemm_tc_persist / fused kernels (1x1 convs, 3x3 extras, heads)',
                            'dw': 'k_dw_strip', 'stem': 'k_stem', 'add': 'k_add',
                            'post': 'k_decode_scores+k_nms+k_merge_filter'}.get(dom, dom),
                 'peak_source': src, 'share_of_step': d['ms'] / total, 'launches_per_step': d['launches'],
                 'algorithmic_gflop_per_step': d['flops'] / 1e9, 'algorithmic_mb_per_step': d['bytes'] / 1e6,
                 'avg_launch_us': 1e3 * d['ms'] / max(1, d['launches']),
                 'frac_of_mode_ceiling': (roof['achieved'] / (tf / {0: 1e9, 1: 1.0, 2: 6.0}[precision])
                                          if roof['bound'] == 'tensor' else None),
                 'families_ms': {n: round(f['ms'], 4) for n, f in fam.items()},
                 'families_hbm_frac': {n: round(f['bytes'] / (f['ms'] / 1e3) / 1e9 / hbm, 4) for n, f in fam.items()
                                       if f['ms'] > 0},
                 'note': 'per-layer CUDA events, every layer launched 10x back to back (median of 5 runs); '
                         'TF32X3 issues 3 TF32 MMAs per product, so its tensor ceiling is bf16 peak/6 (frac_of_mode_ceiling); '
                         'traffic from ncu is in profiles/'})
    return roof, table


if __name__ == '__main__':
    main()
