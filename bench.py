#!/usr/bin/env python
"""bench.py -- frames/s of the heatmap -> 3D keypoint path on N B200s (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A step is one pass of the hot path (K1 peaks, K3/K4 grouping + 3D lift; for N > 1 the grouping kernel also
stores every frame's 3D keypoint record into the gathering rank's buffer over NVLink) over one batch of synthetic network outputs that is
already resident in HBM. Frames shard independently: every rank decodes its own `frames` frames
(weak scaling), `value` is the whole-job frames/s = N * frames / max-over-ranks step time.

Workloads (BASELINE.json configs; SURVEY.md section 8d):
  config4_180x320  4096 valve frames [1,3] of 180x320 per GPU, 8 objects per frame   (default)
  config4_64x64    4096 valve frames of 64x64 per GPU, 2 objects per frame
  config2_cups     128 cups frames [1,1,1] of 64x64 (64 stereo pairs), 1-4 objects

One JSON line is printed by rank 0.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    'config4_180x320': dict(cfg=[1, 3], size=(180, 320), frames=4096, grid=(4, 2), config='valve.json'),
    'config4_64x64': dict(cfg=[1, 3], size=(64, 64), frames=4096, grid=(2, 1), config='valve.json'),
    'config2_cups': dict(cfg=[1, 1, 1], size=(64, 64), frames=128, grid=(2, 2), config='cups.json'),
}
METRIC = "frames/sec heatmap->3D keypoints"
UNIT = "frames/s"


def measured_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f), 'measured'
    return {'hbm_gbs': 6650.0, 'sm_max_mhz': 1965.0}, 'fallback'       # B200_PROFILING.md fallback


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled while the timed region runs."""
    FIELDS = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
              'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
              'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index = index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.FIELDS}', '--format=csv,noheader,nounits',
                                          '-lms', '100', '-i', str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        sm, sm_max, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for line in self.lines:
            parts = [p.strip() for p in line.split(',')]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                sm_max.append(float(parts[1]))
            except ValueError:
                continue
            for name, value in zip(names, parts[3:7]):
                if value.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': statistics.median(sm) if sm else None, 'sm_max_mhz': max(sm_max) if sm_max else None,
                'reasons': sorted(reasons), 'samples': len(sm)}


def workload_config(workload, world, exchange='gather'):
    """The `config` object of the JSON line -- the SAME dict for both arms (ours / reference), so that the driver's
    same_config check holds: it names the workload, not how an arm samples it (that is in `cpu_baseline.sample` / `e2e`)."""
    w = WORKLOADS[workload]
    H, W = w['size']
    C = 1 + len(w['cfg'])
    heat_bytes = w['frames'] * C * H * W * 4
    return {'workload': workload, 'keypoint_config': w['config'], 'frames_per_gpu': w['frames'],
            'prediction_size': [H, W], 'objects_per_frame': w['grid'][0] * w['grid'][1],
            'l2': f"inputs {heat_bytes / 1e6:.0f} MB heatmaps per step exceed the 126 MB L2; no flush needed",
            'parallelism': f"frames sharded over {world} GPU(s); per step one "
                           f"{'gather to rank 0' if exchange == 'gather' else 'all_gather'} of the 3D keypoint records"}


PARITY_INT = ('peak_count', 'peak_yx', 'peak_object', 'n_objects', 'flags', 'kp_assigned', 'kp_count', 'kp_peak', 'n_votes')
PARITY_F32 = ('peak_score', 'peak_xy', 'peak_conf', 'kp_xy')


def parity_mismatches(got, want):
    """Frames of `got` (GPU tables, NumPy) that differ from the oracle's `want` under the parity rules: integer tables and
    flags equal, float32 tables bitwise, votes equal, 3D points <= 1e-4 relative. -> (frames compared, frames differing)."""
    import numpy as np
    n = want['n_objects'].shape[0]
    bad = np.zeros(n, bool)
    for key in PARITY_INT:
        bad |= (got[key][:n].reshape(n, -1) != want[key].reshape(n, -1)).any(axis=1)
    for key in PARITY_F32:
        bad |= (got[key][:n].view(np.uint32).reshape(n, -1) != want[key].view(np.uint32).reshape(n, -1)).any(axis=1)
    for key in ('peak_vote', 'votes'):
        bad |= (got[key][:n].reshape(n, -1) != want[key].reshape(n, -1)).any(axis=1)
    scale = np.maximum(np.linalg.norm(want['kp_point'], axis=-1), 1e-9)
    err = np.linalg.norm(got['kp_point'][:n] - want['kp_point'], axis=-1)
    bad |= (err > 1e-4 * scale + 1e-12).reshape(n, -1).any(axis=1)
    return n, int(bad.sum())


DUMP_BYTES = 60_000_000


def dump_outputs(directory, tables, budget=DUMP_BYTES):
    """Writes decode tables (NumPy, as DecodeTables.numpy() returns them) as DIR/<table>.npy, float32 tables as they are and
    the integer tables and flags as float64 (exact), so that two builds can be compared output for output. When all frames
    would take more than `budget` bytes, a fixed seeded sample of frames is written; frame_index.npy lists the frames."""
    import numpy as np
    n = tables['n_objects'].shape[0]
    per_frame = sum(int(np.prod(v.shape[1:])) * (4 if v.dtype == np.float32 else 8) for v in tables.values())
    keep = min(n, budget // max(per_frame, 1))
    frames = np.arange(n) if keep == n else np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, 'frame_index.npy'), frames.astype(np.float64))
    for name, value in tables.items():
        np.save(os.path.join(directory, f'{name}.npy'), value[frames].astype(np.float32 if value.dtype == np.float32 else np.float64))


def make_inputs(workload, device, seed):
    import torch
    from object_keypoints_b200 import synthetic
    w = WORKLOADS[workload]
    if workload == 'config2_cups':
        batch = synthetic.make_batch(w['frames'], w['cfg'], w['size'], seed=1002 + seed, objects=(1, 4))
        return (torch.from_numpy(batch.heat).to(device), torch.from_numpy(batch.depth).to(device),
                torch.from_numpy(batch.centers).to(device))
    heat, depth, centers, _ = synthetic.torch_grid_batch(w['frames'], w['cfg'], w['size'], seed=1004 + seed,
                                                         grid=w['grid'], device=device)
    return heat, depth, centers


def cpu_baseline(workload, heat, depth, centers, budget_s=12.0):
    """The C oracle (OpenMP, every host core) on a bounded sample of the very same frames."""
    from object_keypoints_b200 import synthetic
    from oracle import c_oracle
    w = WORKLOADS[workload]
    camera = synthetic.default_camera(w['size'])
    cores = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else c_oracle.max_threads()
    probe = min(64, heat.shape[0])
    h, d, c = heat[:probe].cpu().numpy(), depth[:probe].cpu().numpy(), centers[:probe].cpu().numpy()
    c_oracle.decode(h, d, c, w['cfg'], camera, threads=cores)                       # warm-up (thread pool, page faults)
    t0 = time.perf_counter()
    c_oracle.decode(h, d, c, w['cfg'], camera, threads=cores)
    rate = probe / (time.perf_counter() - t0)
    sample = int(max(probe, min(heat.shape[0], rate * budget_s)))
    h, d, c = heat[:sample].cpu().numpy(), depth[:sample].cpu().numpy(), centers[:sample].cpu().numpy()
    t0 = time.perf_counter()
    want = c_oracle.decode(h, d, c, w['cfg'], camera, threads=cores)
    elapsed = time.perf_counter() - t0
    return {'value': sample / elapsed, 'unit': UNIT, 'cores': cores, 'kind': 'port',
            'sample': f"first {sample} frames of {workload} (C/OpenMP restatement oracle/okp_oracle.c, {elapsed:.2f} s)"}, want


def run_reference(args):
    """--impl reference: the reference's CPU algorithm (the C/OpenMP port; the Python original cannot
    travel to the GPU box) on every host core, same workload/metric; rank 0 only."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    import torch
    from object_keypoints_b200 import synthetic
    from oracle import c_oracle
    w = WORKLOADS[args.workload]
    camera = synthetic.default_camera(w['size'])
    sample = min(w['frames'], 512 if w['size'] != (64, 64) else 2048)
    if w['size'] == (64, 64) and args.workload == 'config2_cups':
        batch = synthetic.make_batch(w['frames'], w['cfg'], w['size'], seed=1002, objects=(1, 4))
        heat, depth, centers = batch.heat, batch.depth, batch.centers
    else:
        device = 'cuda' if torch.cuda.is_available() else 'cpu'
        h, d, c, _ = synthetic.torch_grid_batch(sample, w['cfg'], w['size'], seed=1004, grid=w['grid'], device=device, chunk=64)
        heat, depth, centers = h.cpu().numpy(), d.cpu().numpy(), c.cpu().numpy()
    sample = heat.shape[0]
    # every host core, whatever OMP_NUM_THREADS says (torchrun sets it to 1 for its workers)
    cores = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
    for _ in range(max(args.warmup, 1)):
        c_oracle.decode(heat, depth, centers, w['cfg'], camera, threads=cores)
    times = []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        out = c_oracle.decode(heat, depth, centers, w['cfg'], camera, threads=cores)
        times.append(time.perf_counter() - t0)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out)
    ms = 1e3 * sum(times) / len(times)
    value = sample / (ms / 1e3)
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32', 'data': 'synthetic',
        'config': workload_config(args.workload, args.gpus, args.exchange),
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': cores, 'kind': 'port',
                         'sample': f"{sample} frames of {args.workload} per step, C/OpenMP port of perception/pipeline.py"},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line))


def time_decode(decoder, inputs, tables, steps, warmup=3):
    """ms per decode_batch over `steps` back-to-back calls (CUDA events on the launching stream, after warm-up)."""
    import torch
    for _ in range(warmup):
        decoder.decode_batch(*inputs, tables=tables)
    torch.cuda.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(steps):
        decoder.decode_batch(*inputs, tables=tables)
    stop.record()
    torch.cuda.synchronize()
    return start.elapsed_time(stop) / steps


def secondary_64x64(device, peaks, steps):
    """The network's real output resolution (SURVEY.md 8: KeypointNet emits 64x64): 32768 valve frames of 64x64 (1.61 GB of
    float32 heatmaps, far above the 126 MB L2), float32 and bfloat16, whole step = peak kernel + overflow fix-up + grouping
    kernel, lean tables (only valid slots are written: at this size clearing the tables would be a quarter of the DRAM
    traffic). Parity of this workload: tests/test_gpu_decode.py::test_headline_bench_workload_is_bitwise_the_oracle."""
    import torch
    from object_keypoints_b200 import KeypointDecoder, synthetic
    w = WORKLOADS['config4_64x64']
    frames = 32768
    heat, depth, centers, n_obj = synthetic.torch_grid_batch(frames, w['cfg'], w['size'], seed=1004, grid=w['grid'], device=device)
    camera = synthetic.default_camera(w['size'])
    out = []
    for dtype, esize, lean in (('f32', 4, True), ('f32', 4, False), ('bf16', 2, True)):
        decoder = KeypointDecoder(w['cfg'], w['size'], camera=camera, device=device, lean_tables=lean)
        inputs = (heat, depth, centers) if dtype == 'f32' else tuple(t.to(torch.bfloat16) for t in (heat, depth, centers))
        tables = decoder.tables(frames)
        ms = time_decode(decoder, inputs, tables, steps)
        found = float((tables['n_objects'] == n_obj).float().mean())
        assert found > 0.99, f"64x64 {dtype}: only {found:.3f} of the frames decoded to {n_obj} objects"
        nbytes = frames * 3 * 64 * 64 * esize
        out.append({'workload': 'config4_64x64', 'dtype': dtype, 'frames': frames, 'lean_tables': lean, 'ms': ms, 'kernel_ms': ms,
                    'frames_per_s': frames / (ms / 1e3), 'algorithmic_bytes': nbytes,
                    'achieved_gbs': nbytes / (ms / 1e3) / 1e9, 'frac': nbytes / (ms / 1e3) / 1e9 / peaks['hbm_gbs']})
        del decoder, tables, inputs
    del heat, depth, centers
    torch.cuda.empty_cache()
    return out


def secondary_config3(device, reps=5):
    """BASELINE config 3: valve sequence of ~900 frames (30 s at 30 fps), 8 objects, 16 viewpoints per point: decode ->
    cross-view association -> robust multi-view triangulation (object_keypoints_b200/sequence.py), everything on the device.
    Parity: tests/test_sequence.py (bit-equal matches / masks, points <= 1e-4 relative against oracle/sequence_oracle.py)."""
    import numpy as np
    import torch
    from object_keypoints_b200 import KeypointDecoder, sequence, synthetic, targets
    camera = synthetic.default_camera((180, 320))
    seq = sequence.synthetic_sequence(900)
    keypoints, depths = sequence.project_sequence(seq, camera)
    heat, depth, centers = targets.rasterise_targets(keypoints, depths, [1, 3], (180, 320), device=device)
    decoder = KeypointDecoder([1, 3], (180, 320), camera=camera, device=device)
    tables = decoder.tables(900)
    chain = sequence.SequenceTriangulator(camera, views=16, device=device)
    prepared = chain.prepare(seq['T_CW'])
    events = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    decode_ms = chain_ms = 0.0
    out = None
    for rep in range(reps + 2):
        events[0].record()
        decoder.decode_batch(heat, depth, centers, tables=tables)
        events[1].record()
        out = chain(tables, prepared)
        events[2].record()
        torch.cuda.synchronize()
        if rep >= 2:
            decode_ms += events[0].elapsed_time(events[1]) / reps
            chain_ms += events[1].elapsed_time(events[2]) / reps
    points = out['points'].cpu().numpy()
    ok = ~np.isnan(points[..., 0])
    truth = seq['scene'].reshape(-1, 3)
    error = np.linalg.norm(points[ok][:, None] - truth[None], axis=2).min(axis=1)
    observed, valid = out['observed'].cpu().numpy()[ok], out['valid'].cpu().numpy()[ok]
    return {'workload': 'config3_sequence: 900 valve frames 180x320, 8 objects, 16 views per point', 'frames': 900,
            'tracks': int(ok.sum()), 'views': 16, 'decode_ms': decode_ms, 'association_triangulation_ms': chain_ms,
            'frames_per_s': 900 / ((decode_ms + chain_ms) / 1e3), 'points_per_s': int(ok.sum()) / (chain_ms / 1e3),
            'objects_per_frame': float(tables['n_objects'].float().mean()),
            'views_observed_mean': float(observed.sum(axis=1).mean()), 'views_dropped_by_the_filter': int(observed.sum() - valid.sum()),
            'median_error_m': float(np.median(error)), 'within_1cm': float((error < 1e-2).mean())}


def secondary_config5(device, batch=256, reps=3):
    """BASELINE config 5: random-init CornerNet-Squeeze forward in bf16 at batch 256 (plain PyTorch / cuDNN: the input
    producer, not the product) whose three head outputs stay on the device and go straight into okp_decode_bf16.
    Random-init heatmaps sit at ~0.5: about a hundred noise peaks per map, every map overflows the fast path."""
    import torch
    from object_keypoints_b200 import KeypointDecoder, producer, synthetic
    cfg = [1, 3]
    torch.backends.cudnn.benchmark = True
    net = producer.build_producer(cfg, device=device, dtype=torch.bfloat16, seed=0)
    generator = torch.Generator(device=device).manual_seed(0)
    frames = torch.randn(batch, 3, 511, 511, device=device, dtype=torch.bfloat16, generator=generator).contiguous(memory_format=torch.channels_last)
    decoder = KeypointDecoder(cfg, (64, 64), camera=synthetic.default_camera((64, 64)), device=device, max_peaks=128, max_objects=128,
                              max_votes=64)
    tables = decoder.tables(batch)
    events = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    net_ms = dec_ms = 0.0
    with torch.no_grad():
        for rep in range(reps + 2):
            events[0].record()
            heat, depth, centers = net(frames)
            events[1].record()
            decoder.decode_batch(heat, depth, centers, tables=tables)
            events[2].record()
            torch.cuda.synchronize()
            if rep >= 2:
                net_ms += events[0].elapsed_time(events[1]) / reps
                dec_ms += events[1].elapsed_time(events[2]) / reps
    out = {'workload': 'config5: CornerNet-Squeeze bf16 forward (PyTorch) -> okp_decode_bf16, random-init weights', 'batch': batch,
           'network_ms': net_ms, 'decode_ms': dec_ms, 'frames_per_s': batch / ((net_ms + dec_ms) / 1e3),
           'decode_share': dec_ms / (net_ms + dec_ms), 'mean_peaks_per_map': float(tables['peak_count'].float().mean()),
           'overflow_frames': int((tables['flags'] & 1).ne(0).sum()), 'dtype': 'bf16'}
    del net, frames
    torch.cuda.empty_cache()
    return out


def host_read_ceiling(device, nbytes=1 << 30):
    """Measured ceilings of the e2e path on this box: (a) the DMA engine reading pinned host memory into HBM, (b) every
    host core of this rank reading the same pinned buffer (the host pass's access pattern). GB/s."""
    import numpy as np
    import torch
    host = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    host.fill_(1)
    dev = torch.empty(nbytes, dtype=torch.uint8, device=device)
    for _ in range(2):
        dev.copy_(host, non_blocking=True)
    torch.cuda.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(3):
        dev.copy_(host, non_blocking=True)
    stop.record()
    torch.cuda.synchronize()
    h2d = 3 * nbytes / (start.elapsed_time(stop) / 1e3) / 1e9
    view = host.numpy().view(np.float32)
    threads = torch.get_num_threads()
    t0 = time.perf_counter()
    total = float(torch.from_numpy(view).sum())            # a streaming read by torch's intra-op threads
    read = nbytes / (time.perf_counter() - t0) / 1e9
    del host, dev
    return {'h2d_pinned_gbs': h2d, 'host_read_gbs': read, 'host_read_threads': threads, 'checksum': total != 0.0}


def run_ours(args):
    import torch
    import torch.distributed as dist
    from object_keypoints_b200 import KeypointDecoder, synthetic, sharding
    from object_keypoints_b200.sharding import RecordExchange

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    device = torch.device('cuda', local_rank)
    if world > 1:
        import datetime
        # a protocol bug must cost minutes, not the watchdog's default ten
        dist.init_process_group('nccl', device_id=device, timeout=datetime.timedelta(seconds=180))
    w = WORKLOADS[args.workload]
    frames = w['frames']
    H, W = w['size']
    C = 1 + len(w['cfg'])
    camera = synthetic.default_camera(w['size'])
    heat, depth, centers = make_inputs(args.workload, device, seed=rank)
    decoder = KeypointDecoder(w['cfg'], w['size'], camera=camera, device=device)
    tables = decoder.tables(frames)
    root = 0 if args.exchange == 'gather' else None
    exchange = RecordExchange(decoder, frames, world=world, rank=rank, transport=args.transport, root=root) if world > 1 else None
    gathered = None

    def step():
        """One pass of the hot path: the peak kernel (K1) + its no-op overflow fix-up, then the grouping / 3D-lift kernel,
        which for N > 1 also stores every frame's compact record straight into the gathering rank's buffer over NVLink."""
        sink = exchange.begin() if world > 1 else None
        decoder.decode_batch(heat, depth, centers, tables=tables, records=sink)
        return exchange.end()[0] if world > 1 else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        gathered = step()
    barrier()

    # ---- timed region: exactly K steps, device time, the decode bracketed by its own events ----
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.2)
    # K1 is timed inside the timed region, in every K1_EVERY-th step: the two events around the kernel's launch sit between
    # kernels that otherwise overlap their launch latencies (programmatic dependent launches), which costs ~15 us per
    # instrumented step (r02v: 513 us per step with every step instrumented, 495 us with none)
    k1_every = max(1, args.k1_every)
    k1_events = {i: (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
                 for i in range(0, args.steps, k1_every)}
    for pair in k1_events.values():                     # torch creates a CUDA event at its first record: not inside the region
        for event in pair:
            event.record()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    start.record()
    phase_events = {i: (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for i in k1_events}
    for i in range(args.steps):
        if i in phase_events:
            phase_events[i][0].record()                 # before the exchange's admission wait (N > 1) and the counter memset
        sink = exchange.begin() if world > 1 else None
        decoder.decode_batch(heat, depth, centers, tables=tables, records=sink, peaks_done=k1_events.get(i))
        if i in phase_events:
            phase_events[i][1].record()                 # behind the grouping kernel
        if world > 1:
            gathered, _ = exchange.end()
    if world > 1:
        exchange.finish()                               # every completion of the K steps is inside the timed region
    stop.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    elapsed_ms = start.elapsed_time(stop)
    k1_ms = sum(a.elapsed_time(b) for a, b in k1_events.values()) / len(k1_events)
    # where an instrumented step's time goes on this rank: in front of K1 (admission wait of the exchange, counter memset),
    # K1, behind it (overflow fix-up, grouping + record stores, launch gaps)
    lead_ms = sum(phase_events[i][0].elapsed_time(k1_events[i][0]) for i in k1_events) / len(k1_events)
    tail_ms = sum(k1_events[i][1].elapsed_time(phase_events[i][1]) for i in k1_events) / len(k1_events)
    if args.dump_outputs and rank == 0:                 # the tables of the last timed step, before anything else reuses them
        dump_outputs(args.dump_outputs, tables.numpy())

    # ---- sustained behaviour: ~1 s of back-to-back steps (the K timed steps above last ~10 ms), clocks sampled throughout ----
    sustained = None
    if not args.no_sustained:
        count = max(args.steps, args.sustained_steps)          # the SAME on every rank: each step is a cross-rank exchange
        sampler2 = ClockSampler(local_rank)
        if rank == 0:
            sampler2.start()
        barrier()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for _ in range(count):
            step()
        if world > 1:
            exchange.finish()
        s1.record()
        barrier()
        ms = torch.tensor([s0.elapsed_time(s1) / count], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        if rank == 0:
            sustained = {'steps': count, 'ms_per_step': float(ms), 'frames_per_s': world * frames / (float(ms) / 1e3),
                         'clocks': sampler2.stop()}

    # ---- parity, outside the timed region ----
    # N > 1: the gathered rows of EVERY rank against a re-pack of that rank's own tables (plain torch + NCCL all_gather)
    gathered_check = None
    if world > 1:
        mine = sharding.unpack_compact_records(sharding.pack_compact_records(tables, w['cfg']), decoder.params.max_objects, w['cfg'])
        want = {}
        for key, value in mine.items():
            parts = [torch.empty_like(value) for _ in range(world)]
            dist.all_gather(parts, value.contiguous())
            want[key] = torch.cat(parts)
        if rank == 0 or args.exchange == 'allgather':
            back = sharding.unpack_compact_records(gathered, decoder.params.max_objects, w['cfg'])
            bad = torch.zeros(world * frames, dtype=torch.bool, device=device)
            for key in want:
                bad |= (back[key] != want[key]).reshape(world * frames, -1).any(dim=1)
            gathered_check = {'rows': world * frames, 'mismatches': int(bad.sum()),
                              'objects': int(back['n_objects'].sum())}
            assert gathered_check['mismatches'] == 0, f"gathered records differ from the ranks' tables: {gathered_check}"
            assert gathered_check['objects'] > 0.99 * world * frames * w['grid'][0] * w['grid'][1]
    # every rank: a sample of its own frames against the C oracle
    parity = None
    if not args.no_cpu_baseline:
        from oracle import c_oracle
        sample = frames if world == 1 else min(frames, 128)
        cores = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else 1
        if world == 1:
            baseline, want_tables = cpu_baseline(args.workload, heat, depth, centers)
        else:
            baseline = None
            want_tables = c_oracle.decode(heat[:sample].cpu().numpy(), depth[:sample].cpu().numpy(), centers[:sample].cpu().numpy(),
                                          w['cfg'], camera, threads=max(1, cores // world))
        compared, differing = parity_mismatches(tables.numpy(), want_tables)
        counts = torch.tensor([compared, differing], dtype=torch.int64, device=device)
        if world > 1:
            dist.all_reduce(counts)
        parity = {'frames': int(counts[0]), 'mismatches': int(counts[1]), 'against': 'oracle/okp_oracle.c on the same frames',
                  'rules': 'integer + float32 tables bitwise, 3D points <= 1e-4 relative'}
        if gathered_check is not None:
            parity['gathered'] = gathered_check
        assert parity['mismatches'] == 0, f"{parity['mismatches']} of {parity['frames']} frames differ from the oracle"

    # ---- strong scaling (N > 1): BASELINE config 4 as worded -- 4096 frames TOTAL sharded over the N GPUs, one CUDA graph
    # replay = `depth` steps (decode + record stores + completion barrier on a forked stream), so that a 512-frame step is not
    # bound by launch overhead. Rank 0 then decodes all 4096 frames alone for the single-GPU reference of the same run. ----
    strong = None
    if world > 1 and frames % world == 0:
        strong = strong_scaling(args, decoder, exchange.transport, heat, depth, centers, frames, world, rank, device, root, barrier)

    # ---- end to end through the public API with HOST buffers (pinned), copies inside the timed region ----
    e2e = end_to_end(args, decoder, heat, depth, centers, frames, world, rank, device, barrier)

    phases = torch.tensor([lead_ms, k1_ms, tail_ms, elapsed_ms / args.steps], dtype=torch.float64, device=device)
    per_rank = [torch.empty_like(phases) for _ in range(world)] if world > 1 else [phases]
    if world > 1:
        dist.all_gather(per_rank, phases)
    per_rank = [[round(float(v), 4) for v in row.cpu()] for row in per_rank]
    times = torch.tensor([elapsed_ms, k1_ms], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    elapsed_ms, k1_ms = [float(v) for v in times.cpu()]

    # sanity: the decode found the objects that were drawn (guards against timing an empty kernel)
    found = float((tables['n_objects'] > 0).float().mean())
    assert found > 0.99, f"only {found:.3f} of the frames produced objects"

    if rank == 0:
        peaks, peak_kind = measured_peaks()
        ms_per_step = elapsed_ms / args.steps
        value = world * frames / (ms_per_step / 1e3)
        algorithmic_bytes = frames * C * H * W * 4                 # every heatmap byte exactly once (SURVEY 8d)
        achieved = algorithmic_bytes / (k1_ms / 1e3) / 1e9
        traffic = None
        for name in ('r02_k1_traffic.json', 'r01_k1_traffic.json'):
            ncu_summary = os.path.join(ROOT, 'profiles', name)
            if os.path.exists(ncu_summary):
                with open(ncu_summary) as f:
                    traffic = json.load(f).get(args.workload)
                break
        line = {
            'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': max(args.warmup, 3),
            'ms_per_step': ms_per_step, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f32', 'data': 'synthetic',
            'config': workload_config(args.workload, world, args.exchange),
            'exchange': (f"{exchange.transport}{'/staged' if getattr(exchange, 'staged', False) else ''}: " +
                         ('the grouping kernel writes every frame\'s compact record into a local buffer, the exchange stream pushes '
                          'the buffer into the gathering rank with one peer copy over NVLink (copy engine, no SM); completion = a '
                          'device-side barrier' if getattr(exchange, 'staged', False) else
                          'the grouping kernel stores every frame\'s compact record straight into the gathering rank over NVLink; '
                          'completion = a device-side barrier' if exchange.transport == 'peer' else 'compact records + NCCL')
                         + ", overlapped with the next step's decode") if world > 1 else None,
            'roofline': {'bound': 'hbm', 'achieved': achieved, 'peak': peaks['hbm_gbs'], 'unit': 'GB/s',
                         'frac': achieved / peaks['hbm_gbs'], 'traffic': traffic, 'peak_source': peak_kind,
                         'kernel': 'okp_peaks_stream_kernel<float>: box sum + NMS + threshold + raster order + centroid of every map; '
                                   'kernel_ms = CUDA events recorded on the launching stream right before and right after its '
                                   f'launch (okp_extract_peaks_events_f32) in every {k1_every}th of the timed steps',
                         'kernel_ms': k1_ms, 'algorithmic_bytes': algorithmic_bytes},
            'e2e': e2e,
            'gpu_launches': args.steps * 3,
            'clocks': clocks,
        }
        if parity is not None:
            line['parity'] = parity
        if strong is not None:
            line['strong'] = strong
        if sustained is not None:
            line['sustained'] = sustained
        line['phases_per_rank'] = {'columns': ['ms in front of K1 (exchange admission wait, counter memset)', 'K1 ms',
                                               'ms behind K1 (overflow fix-up, grouping + record stores, gaps)', 'ms per step'],
                                   'instrumented_steps': sorted(k1_events), 'ranks': per_rank}
        if not args.no_cpu_baseline and world == 1:
            line['cpu_baseline'] = baseline
        if world == 1 and not args.no_secondary:
            line['secondary'] = secondary_64x64(device, peaks, max(5, min(args.steps, 20)))
            line['secondary'].append(secondary_config3(device))
            line['secondary'].append(secondary_config5(device))
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def strong_scaling(args, decoder, transport, heat, depth, centers, frames, world, rank, device, root, barrier):
    import torch
    import torch.distributed as dist
    from object_keypoints_b200.sharding import RecordExchange
    share = frames // world
    inputs = (heat[:share], depth[:share], centers[:share])
    tables = decoder.tables(share)
    exchange = RecordExchange(decoder, share, world=world, rank=rank, transport=transport, root=root)
    steps_per_graph = exchange.depth

    def eager_steps(count):
        for _ in range(count):
            sink = exchange.begin()
            decoder.decode_batch(*inputs, tables=tables, records=sink)
            exchange.end()

    eager_steps(exchange.depth)                                # warm-up (allocations, module loads) before the capture
    exchange.finish()
    barrier()
    graph, how = None, 'eager launches'
    try:
        exchange.calls = 0
        side = torch.cuda.Stream(device=device)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=side):
                eager_steps(steps_per_graph)                   # LAG < depth: every event waited on is recorded inside the capture
                exchange.finish()
        torch.cuda.current_stream().wait_stream(side)
        how = f"one CUDA graph replay = {steps_per_graph} steps"
    except Exception as error:                                 # e.g. a collective that cannot be captured on this build
        graph, how = None, f"eager launches (graph capture failed: {type(error).__name__})"
        torch.cuda.synchronize()
        exchange.calls = 0
    replays = max(1, (args.steps * 4 + steps_per_graph - 1) // steps_per_graph)

    def run(count):
        for _ in range(count):
            if graph is not None:
                graph.replay()
            else:
                eager_steps(steps_per_graph)
                exchange.finish()

    run(2)
    barrier()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    run(replays)
    stop.record()
    barrier()
    ms = torch.tensor([start.elapsed_time(stop) / (replays * steps_per_graph)], dtype=torch.float64, device=device)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms)
    single_ms = None
    if rank == 0:                                              # the single-GPU time of the same 4096 frames, same run, same GPU
        single_ms = time_decode(decoder, (heat, depth, centers), decoder.tables(frames), max(5, args.steps))
    barrier()
    if rank != 0:
        return None
    return {'frames_total': frames, 'frames_per_gpu': share, 'ms_per_step': ms, 'frames_per_s': frames / (ms / 1e3),
            'single_gpu_ms_per_step': single_ms, 'efficiency_vs_n1': (single_ms / ms) / world,
            'launch': how, 'steps_timed': replays * steps_per_graph}


def end_to_end(args, decoder, heat, depth, centers, frames, world, rank, device, barrier):
    import torch
    import torch.distributed as dist
    e2e_frames = min(frames, args.e2e_frames)
    host = [t[:e2e_frames].cpu().pin_memory() for t in (heat, depth, centers)]
    e2e_steps = max(1, min(args.steps, args.e2e_steps))

    def timed(**options):
        out = None
        for _ in range(2):
            out = decoder.decode_host_batch(*host, out=out, **options)
        barrier()
        t_start, t_stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_start.record()
        for _ in range(e2e_steps):
            out = decoder.decode_host_batch(*host, out=out, **options)
        t_stop.record()
        barrier()
        ms = torch.tensor([t_start.elapsed_time(t_stop) / e2e_steps], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms), out, decoder.host_bytes_copied, decoder.host_chunks_sparse, getattr(decoder, 'host_marked_fraction', None)

    e2e_ms, result_host, h2d, sparse_chunks, marked = timed()
    dense_ms, _, dense_h2d, _, _ = timed(sparse=False)
    d2h = sum(v.numel() * v.element_size() for v in result_host.values())
    out = {'value': world * e2e_frames / (e2e_ms / 1e3), 'unit': UNIT, 'h2d_bytes_per_step': h2d,
           'd2h_bytes_per_step': d2h, 'frames_per_step': e2e_frames, 'steps': e2e_steps,
           'host_input_bytes_per_step': sum(t.numel() * t.element_size() for t in host),
           'sparse_chunks': sparse_chunks, 'marked_tile_fraction': marked,
           'e2e_dense': {'value': world * e2e_frames / (dense_ms / 1e3), 'h2d_bytes_per_step': dense_h2d,
                         'note': 'sparse=False: every heatmap byte crosses PCIe (what a caller gets on dense maps)'},
           'host_threads_per_rank': getattr(decoder, 'host_pack_threads', None),
           'note': 'pinned host tensors in, pinned host tables out, chunks of 128 frames pipelined (host pass / PCIe / '
                   'decode). Heatmaps: a host pass (OpenMP, inside the timed region) marks the 4x16-pixel tiles '
                   'within reach of a value above threshold / 25 and only those cross PCIe (bit-identical tables, '
                   'csrc/okp_sparse.cuh; dense copy when more than half of a chunk is marked). Depth and centre maps '
                   '(gather-only) are read in place from pinned host memory over PCIe'}
    if rank == 0 and not args.no_cpu_baseline:
        pageable = [t.clone() for t in (h.cpu() for h in (heat[:e2e_frames], depth[:e2e_frames], centers[:e2e_frames]))]
        decoder.decode_host_batch(*pageable)
        t0 = time.perf_counter()
        decoder.decode_host_batch(*pageable)
        out['pageable_inputs'] = {'value': e2e_frames / (time.perf_counter() - t0),
                                  'note': 'one rank, pageable CPU tensors (what InferenceComponent.cpu() hands over in the reference): '
                                          'every map is copied, nothing is gathered in place'}
        out['ceilings'] = host_read_ceiling(device)
    barrier()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='config4_180x320', choices=sorted(WORKLOADS))
    ap.add_argument('--frames', type=int, default=0, help="frames per GPU (default: the workload's)")
    ap.add_argument('--e2e-frames', type=int, default=2048)
    ap.add_argument('--e2e-steps', type=int, default=5)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-secondary', action='store_true', help="skip the 64x64 / config 3 / config 5 lines (N = 1)")
    ap.add_argument('--k1-every', type=int, default=4, help="time K1 with events in every n-th timed step")
    ap.add_argument('--no-sustained', action='store_true', help="skip the ~1 s sustained run")
    ap.add_argument('--sustained-steps', type=int, default=2000)
    ap.add_argument('--exchange', default='gather', choices=['gather', 'allgather'],
                    help="N > 1: gather the records to rank 0 (north_star) or to every rank")
    ap.add_argument('--transport', default='auto', choices=['auto', 'peer', 'nccl'],
                    help="N > 1: how the keypoint records are gathered (sharding.RecordExchange)")
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help="write the tables of the last timed step (rank 0's when N > 1) to DIR/<table>.npy as float32 / float64, "
                         "at most 60 MB (a fixed seeded sample of frames beyond that)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.frames:
        WORKLOADS[args.workload] = dict(WORKLOADS[args.workload], frames=args.frames)
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
