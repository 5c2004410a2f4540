#!/usr/bin/env python
"""bench.py -- frames/s of the deephar forward hot path on B200 (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            (ours; torchrun for N > 1)
  python bench.py --impl reference --gpus N --steps K --warmup W   (CPU arm, see below)

Headline workload (config.workload): ReceptionNet 2-D pose, the model of BASELINE.json configs[1]
(`reception.build((256,256,3), 16, dim=2, num_blocks=8, num_context_per_joint=2, ksize=(5,5))`,
exp/mpii/eval_mpii_singleperson.py:42-49) on the headline batch: 32 clips x 16 frames of 256x256x3 = 512 frames
per step (TimeDistributed folds clips into frames), synthetic uniform[-1,1] frames and seeded synthetic weights
(no datasets / checkpoints offline).

  scaling : STRONG (SURVEY.md 8e): the fixed 32-clip batch is split contiguously over the N ranks
            (`dist.shard_range`: 32 / 16 / 8 / 4 clips per GPU), weights replicated, no data-path collective; the one
            exchange step is a fixed-shape all-gather of the last block's (pose, visibility) over NCCL.  The weak
            number (512 frames on every GPU) is reported under secondary.weak.
  value   : frames/s, inputs resident in HBM, CUDA-event timed, max over ranks.  Forwards are CUDA-graph replays.
  e2e     : frames/s through Model.predict() with pinned HOST input, H2D + D2H inside the timed region.
  roofline: the dominant kernel of the step (CUDA events around every launch of one extra step): algorithmic
            FLOPs / launch time vs the measured bf16 peak; `traffic` = DRAM bytes of that kernel from the committed
            ncu capture (profiles/r2_traffic.json, written by tools/ncu_traffic.py from the raw ncu CSV).
  secondary: the other BASELINE configs on the same box -- C3 (H36M 3-D, b32), C4 (PennAction SPNet, 16 clips),
            C5 (NTU SPNet, 64 clips, action all-gather) -- and the soft-argmax 2-D / 3-D HBM micro-benchmarks.
  --impl reference : the reference's Keras/TF forward cannot run here (no tensorflow/keras in the image,
            SURVEY.md 8c); the arm times the CPU port of the same graph (oracle/, torch-CPU fp32): one step =
            32 frames through the C2 model (a 32-frame sample of the 512-frame step), plus the C1 (b1) latency,
            medians over the timed iterations (SURVEY.md 8d).  Thread count (up to all physical cores) and predict
            batch size (32, or 4 x 8) are the fastest of a short calibration, reported in the line.
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

MODEL_KW = dict(num_joints=16, dim=2, num_context_per_joint=2, num_blocks=8, ksize=(5, 5),
                concat_pose_confidence=False)
C3_KW = dict(num_joints=17, dim=3, num_blocks=8, ksize=(5, 5), concat_pose_confidence=False)
CLIPS, FRAMES = 32, 16
METRIC = 'frames/sec (256x256, 16-frame clips, b32)'
HEADLINE = 'reception2d_8blk_k5_j16 (BASELINE configs[1] model) x 32 clips x 16 frames'


_T0 = time.time()


def note(msg):
    """progress line on stderr (the JSON line on stdout stays alone)"""
    print('[bench %6.1fs] %s' % (time.time() - _T0, msg), file=sys.stderr, flush=True)


def measured_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {'hbm_gbs': p['hbm_gbs'], 'bf16_tflops': p['bf16_tflops'],
                'bf16_tflops_sustained': p.get('bf16_tflops_sustained', p['bf16_tflops']),
                'source': 'measured'}
    return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0, 'bf16_tflops_sustained': 1400.0, 'source': 'fallback'}


def ncu_traffic():
    """{kernel label: {'bytes_per_frame', 'source'}} from the committed ncu capture (tools/ncu_traffic.py)."""
    path = os.path.join(ROOT, 'profiles', 'r2_traffic.json')
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f)
    return {}


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
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
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [s.strip() for s in ln.split(',')]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[5:9]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        if not sm:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['no samples']}
        return {'sm_mhz': float(np.median(sm)), 'sm_max_mhz': float(max(mx)), 'reasons': sorted(reasons),
                'samples': len(sm)}


# ------------------------------------------------------------------------------------------------------------------
# workloads
# ------------------------------------------------------------------------------------------------------------------
def build_workload(name):
    """-> (model, clip_model: bool, label).  Frames are 256x256x3; clip models take (clips, 16, 256, 256, 3)."""
    if name in ('reception2d', 'reception3d'):
        from deephar_b200 import reception
        kw = MODEL_KW if name == 'reception2d' else C3_KW
        label = HEADLINE if name == 'reception2d' else 'reception3d_8blk_k5_j17 (BASELINE configs[2] model, H36M 3-D)'
        return reception.build((256, 256, 3), **kw).init_synthetic_weights(1234), False, label
    from deephar_b200 import spnet
    from deephar_b200.config import ModelConfig, pa16j2d, pa17j3d
    if name == 'spnet_penn':
        cfg = ModelConfig((FRAMES, 256, 256, 3), pa16j2d, num_actions=[15], num_pyramids=6, action_pyramids=[5, 6],
                          num_levels=4, pose_replica=True, num_pose_features=160, num_visual_features=160)
        label = 'spnet PennAction multitask (BASELINE configs[3] model), 16-frame clips'
    else:
        cfg = ModelConfig((FRAMES, 256, 256, 3), pa17j3d, num_actions=[60], num_pyramids=2, action_pyramids=[1, 2],
                          num_levels=4, num_pose_features=192, num_visual_features=192)
        label = 'spnet NTU 3D multitask (BASELINE configs[4] model), 16-frame clips'
    return spnet.build(cfg).init_synthetic_weights(1234), True, label


def shard_plan(items_global, item_frames, rank, world, micro_frames, clip_model):
    """Host arithmetic of one rank's share of a step (no device): the contiguous shard of the global batch
    (`dist.shard_range`), the leading extent of its input tensor -- clips for clip models, frames otherwise -- and how it
    is cut into forward calls of at most `micro_frames` frames.  -> dict(first, items_local, frames_local, lead,
    micro_items, spans)."""
    from deephar_b200.dist import shard_range
    a, b = shard_range(items_global, rank, world)
    items_local = b - a
    frames_local = items_local * item_frames
    lead = items_local if clip_model else frames_local
    per = FRAMES if clip_model else 1
    micro_items = max(1, min(micro_frames // per, lead)) if lead else 1
    spans = [(i, min(i + micro_items, lead)) for i in range(0, lead, micro_items)]
    return {'first': a, 'items_local': items_local, 'frames_local': frames_local, 'lead': lead,
            'micro_items': micro_items, 'spans': spans}


class Runner(object):
    """One workload on this rank's shard of a global batch of `items` (clips, or frames for b32-of-frames configs)."""

    def __init__(self, torch, model, clip_model, items_global, item_frames, rank, world, micro_frames, precision=3):
        self.torch, self.model, self.world = torch, model, world
        model.precision = precision
        plan = shard_plan(items_global, item_frames, rank, world, micro_frames, clip_model)
        self.items_global, self.items_local, self.item_frames = items_global, plan['items_local'], item_frames
        self.frames_local = plan['frames_local']
        self.clip_model = clip_model
        shape = ((plan['lead'], FRAMES, 256, 256, 3) if clip_model else (plan['lead'], 256, 256, 3))
        gen = torch.Generator().manual_seed(1000 + plan['first'])
        self.x_host = torch.empty(*shape, dtype=torch.float32).pin_memory()
        if self.x_host.numel():
            self.x_host.uniform_(-1.0, 1.0, generator=gen)
        self.x_dev = self.x_host.cuda()
        self.micro_items, self.spans = plan['micro_items'], plan['spans']
        self.comm = None            # dist.Comm: the all-gather through the C ABI (set by main for world > 1)

    def forward_all(self, keep=False):
        """Every micro-batch of this rank's shard; returns the last one's outputs (views into the model's buffers).
        keep: also hold a copy of every micro-batch's outputs, concatenated, in self.kept (--dump-outputs)."""
        last, kept = None, []
        for (i, j) in self.spans:
            last = self.model.forward_device(self.x_dev[i:j])
            if keep:
                kept.append([o.clone() for o in last])
        if keep:
            self.kept = [self.torch.cat(parts) for parts in zip(*kept)]
        return last

    def exchange(self, outs, which):
        """The one exchange step of the data-parallel path (SURVEY.md 8e): all-gather of the final outputs."""
        if self.world == 1 or outs is None:
            return outs
        from deephar_b200.dist import gather_outputs
        torch = self.torch
        if which == 'pose':         # reception: last block's (pose, visibility) of the LAST micro-batch
            local = torch.cat([outs[-2], outs[-1]], dim=-1)
            return gather_outputs(local.contiguous(), self.world, comm=self.comm)
        local = torch.stack([o for o in outs if o.dim() == 2], dim=1)    # action probabilities (B_local, n_pred, n_act)
        return gather_outputs(local.contiguous(), self.world, comm=self.comm)

    def step(self, which, keep=False):
        return self.exchange(self.forward_all(keep), which)


def timed_steps(torch, dist, world, fn, steps, warmup, last_fn=None):
    """W warm-ups, then K steps bracketed by barrier + synchronize, CUDA events, max over ranks -> ms per step.
    last_fn: run instead of fn as the last timed step."""
    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    for _ in range(warmup):
        fn()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        (last_fn if last_fn is not None and i == steps - 1 else fn)()
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], device='cuda')
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item()) / steps


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(directory, outs):
    """The outputs of every micro-batch of this rank's shard in the last timed step, as DIR/out<i>.npy (float32, the
    model's output order, items in input order), so that two builds can be compared output for output: the inputs and
    weights are seeded, so the same arguments give the same inputs on every run.  Above DUMP_LIMIT_BYTES in all, every
    array keeps the same fixed, seeded sample of its leading rows (DIR/rows.npy lists them)."""
    arrays = [o.detach().float().cpu().numpy() for o in outs]
    total = sum(a.nbytes for a in arrays)
    os.makedirs(directory, exist_ok=True)
    if total > DUMP_LIMIT_BYTES:
        n = arrays[0].shape[0]
        rows = np.sort(np.random.default_rng(0).choice(n, max(1, n * DUMP_LIMIT_BYTES // total), replace=False))
        arrays = [a[rows] for a in arrays]
        np.save(os.path.join(directory, 'rows.npy'), rows)
    names = ['out%02d' % i for i in range(len(arrays))]
    for name, a in zip(names, arrays):
        np.save(os.path.join(directory, name + '.npy'), a)
    return names


# ------------------------------------------------------------------------------------------------------------------
# CPU arm (SURVEY.md 8d)
# ------------------------------------------------------------------------------------------------------------------
def cpu_port(iters_b32, iters_b1, warm_b32=1, warm_b1=3, calibrate=True):
    """torch-CPU (oneDNN) fp32 port of the Keras graph (oracle/), all host threads: C2 (b32) and C1 (b1) medians."""
    import torch
    from deephar_b200 import reception
    from oracle import ops_torch, synth
    from oracle import reception as oracle_reception
    # all PHYSICAL cores, set explicitly: torchrun exports OMP_NUM_THREADS=1 (round 1's arm ran single-threaded under
    # it), and one thread per hyper-thread (os.cpu_count() = 128 on the B200 hosts) makes oneDNN ~100x slower
    cores = os.cpu_count() or 1
    try:
        import psutil
        threads = psutil.cpu_count(logical=False) or max(1, cores // 2)
    except Exception:
        threads = max(1, cores // 2)
    if hasattr(os, 'sched_getaffinity'):
        threads = max(1, min(threads, len(os.sched_getaffinity(0))))
    m = reception.build((256, 256, 3), **MODEL_KW).init_synthetic_weights(1234)
    table = m.get_weights()

    def run(batch, warm, iters, chunk=None):
        """`iters` timed passes over `batch` frames, `chunk` frames per forward (keras predict(x, batch_size=chunk))"""
        x = synth.synth_frames(batch, seed=0)
        chunk = chunk or batch
        times = []
        for i in range(warm + iters):
            t0 = time.perf_counter()
            for j in range(0, batch, chunk):
                oracle_reception.forward(ops_torch, table, x[j:j + chunk], **MODEL_KW)
            dt = time.perf_counter() - t0
            if i >= warm:
                times.append(dt)
        return times

    # thread count and predict() batch size by calibration (a few seconds): on the many-core GPU hosts one oneDNN
    # thread per physical core is not necessarily the fastest setting (round 2 measured 5.1 frames/s on 64 threads
    # where an 8-core container gives 10.5), and one 32-frame forward is slower per frame than four 8-frame ones when
    # the 134 MB intermediates fall out of the allocator's cache.  The arm reports the best the host does.
    calib, chunk = {}, 32
    if calibrate:
        for c in sorted({c for c in (4, 8, 16, 32, threads // 2, threads) if 1 <= c <= threads}):
            torch.set_num_threads(c)
            calib['%d threads, b8' % c] = (8.0 / min(run(8, 1, 1)), c)
        threads = max(calib.values())[1]
        torch.set_num_threads(threads)
        calib['%d threads, b32' % threads] = (32.0 / min(run(32, 0, 1)), threads)
        if calib['%d threads, b8' % threads][0] > calib['%d threads, b32' % threads][0]:
            chunk = 8
    torch.set_num_threads(threads)
    t1 = run(1, warm_b1, iters_b1) if iters_b1 else []
    t32 = run(32, warm_b32, iters_b32, chunk=chunk)
    return {'b32_times': t32, 'b1_times': t1, 'cores': cores, 'threads': torch.get_num_threads(), 'chunk': chunk,
            'calibration': {k: round(v[0], 2) for k, v in calib.items()}}


def headline_config(world, frames_local, micro):
    return {'workload': HEADLINE, 'global_batch_frames': CLIPS * FRAMES, 'frames_per_gpu': frames_local,
            'micro_batch': micro, 'parallelism': 'dp%d' % world,
            'l2': 'inputs (%.0f MB per GPU per step) + 7 GB of activations per forward >> 126 MB L2; no flush needed'
                  % (frames_local * 256 * 256 * 3 * 4 / 1e6)}


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    from deephar_b200.dist import shard_range
    r = cpu_port(iters_b32=args.steps, iters_b1=10, warm_b32=max(args.warmup, 1), warm_b1=3)
    med32 = float(np.median(r['b32_times']))
    fps = 32.0 / med32
    a, b = shard_range(CLIPS, 0, args.gpus)
    frames_local = (b - a) * FRAMES
    sample = ('32 frames of the C2 model per step (32 of the 512 frames; predict batch_size=%d), median of %d timed '
              'steps = %.2f s; C1 (b1) latency median of 10 = %.3f s; torch-CPU fp32 port of the Keras graph (oracle/), '
              '%d threads (threads and batch size: the fastest of thread_calibration_frames_per_s)'
              % (r['chunk'], len(r['b32_times']), med32, float(np.median(r['b1_times'])), r['threads']))
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': fps, 'unit': 'frames/s', 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1000.0 * med32,
        'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': headline_config(args.gpus, frames_local, min(args.micro_batch, frames_local)),
        'cpu_baseline': {'value': fps, 'unit': 'frames/s', 'cores': r['threads'], 'kind': 'port', 'sample': sample,
                         'c1_b1_latency_s': float(np.median(r['b1_times'])), 'host_cpu_count': r['cores'],
                         'thread_calibration_frames_per_s': r['calibration'],
                         'implementation': 'CPU port of the Keras graph; keras 2.1.4 / tensorflow 1.6 are not '
                                           'installable in this image (SURVEY.md 8c)'},
        'e2e': {'value': fps, 'unit': 'frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------------
# micro-benchmarks: soft-argmax heads (BASELINE metric: "softargmax HBM GB/s")
# ------------------------------------------------------------------------------------------------------------------
def _time_launch(torch, launch, reps=10):
    for _ in range(3):
        launch()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        launch()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def softargmax_microbench(torch, model, peaks):
    """dh_softargmax2d_ctx_f32 on 4096 frames of (32,32,48) = 805 MB (6x L2): achieved HBM GB/s."""
    import ctypes as C
    from deephar_b200 import _ffi
    n = 4096
    g = torch.Generator(device='cuda').manual_seed(0)
    h = torch.randn(n, 32, 32, 48, device='cuda', generator=g) * 3.0
    pose = torch.empty(n, 16, 2, device='cuda')
    vis = torch.empty(n, 16, 1, device='cuda')
    hv = _ffi.dh_view(h.data_ptr(), n, 32, 32, 48, 48)
    lib, ctx = _ffi.lib(), model._ctx.handle
    st = torch.cuda.current_stream().cuda_stream

    def launch():
        _ffi.check(lib.dh_softargmax2d_ctx_f32(ctx, C.byref(hv), 16, 2, C.c_float(0.8), pose.data_ptr(),
                                               vis.data_ptr(), st), 'softargmax')
    ms = _time_launch(torch, launch)
    bytes_ = n * (32 * 32 * 48 * 4 + 16 * 3 * 4)
    gbs = bytes_ / ms / 1e6
    return {'kernel': 'softargmax2d_ctx (32x32x48 maps, %d frames, %.0f MB > L2)' % (n, bytes_ / 1e6),
            'bound': 'hbm', 'achieved': gbs, 'peak': peaks['hbm_gbs'], 'unit': 'GB/s',
            'frac': gbs / peaks['hbm_gbs'], 'us_per_launch': ms * 1000.0, 'peak_source': peaks['source']}


def softargmax3d_microbench(torch, model, peaks):
    """dh_softargmax3d_f32 on C3's volume: 256 frames x (32,32,16*17) = 285 MB (32 frames x 8 blocks of the b32 step)."""
    import ctypes as C
    from deephar_b200 import _ffi
    n, nj, d = 256, 17, 16
    g = torch.Generator(device='cuda').manual_seed(0)
    h = torch.randn(n, 32, 32, nj * d, device='cuda', generator=g) * 3.0
    pose = torch.empty(n, nj, 3, device='cuda')
    vis = torch.empty(n, nj, 1, device='cuda')
    hv = _ffi.dh_view(h.data_ptr(), n, 32, 32, nj * d, nj * d)
    lib, ctx = _ffi.lib(), model._ctx.handle
    st = torch.cuda.current_stream().cuda_stream

    def launch():
        _ffi.check(lib.dh_softargmax3d_f32(ctx, C.byref(hv), nj, d, pose.data_ptr(), vis.data_ptr(), st), 'softargmax3d')
    ms = _time_launch(torch, launch)
    bytes_ = n * (32 * 32 * nj * d * 4 + nj * 4 * 4)
    gbs = bytes_ / ms / 1e6
    return {'kernel': 'softargmax3d (32x32x272 volumes, %d frames, %.0f MB > L2)' % (n, bytes_ / 1e6),
            'bound': 'hbm', 'achieved': gbs, 'peak': peaks['hbm_gbs'], 'unit': 'GB/s',
            'frac': gbs / peaks['hbm_gbs'], 'us_per_launch': ms * 1000.0, 'peak_source': peaks['source']}


def single_frame_latency(torch, model):
    """BASELINE configs[0] (C1): one 256x256 frame through the 8-block ReceptionNet -- the reference's own CPU-runnable
    case.  Device-resident latency (CUDA events over 50 graph replays) and end-to-end latency of the public call
    (host frame in, host pose out)."""
    import time
    g = torch.Generator().manual_seed(7)
    x_host = torch.empty(1, 256, 256, 3).uniform_(-1.0, 1.0, generator=g).pin_memory()
    x_dev = x_host.cuda()
    ms = _time_launch(torch, lambda: model.forward_device(x_dev), reps=50)
    x_np = x_host.numpy()
    for _ in range(3):
        model.predict(x_np, batch_size=1)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(20):
        model.predict(x_np, batch_size=1)
    torch.cuda.synchronize()
    e2e = (time.perf_counter() - t0) / 20
    return {'config': 'MPII single-person 2-D pose, 1 frame (BASELINE configs[0])', 'latency_ms': ms,
            'frames_per_s': 1000.0 / ms, 'e2e_latency_ms': e2e * 1000.0, 'e2e_frames_per_s': 1.0 / e2e}


def preprocess_microbench(torch):
    """SURVEY 8 f4: 32 decoded 480x640 uint8 frames -> crop -> bilinear 256x256 -> normalize, through
    deephar_b200.preprocess.FramePipeline with HOST images (pinned upload inside the timed region)."""
    import time
    from deephar_b200 import preprocess
    rng = np.random.default_rng(0)
    imgs = [rng.integers(0, 256, (480, 640, 3), dtype=np.uint8) for _ in range(32)]
    objpos = rng.uniform(200, 300, (32, 2))
    wins = rng.uniform(250, 500, 32)
    pipe = preprocess.FramePipeline((256, 256))
    out = torch.empty(32, 256, 256, 3, device='cuda')
    for _ in range(3):
        pipe(imgs, objpos, wins, out=out)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    reps = 10
    for _ in range(reps):
        pipe(imgs, objpos, wins, out=out)
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / reps
    return {'workload': '32 x 480x640x3 uint8 -> 256x256x3 fp32 (crop + Pillow-exact bilinear + normalize)',
            'value': 32.0 / dt, 'unit': 'frames/s', 'ms_per_batch': dt * 1000.0, 'h2d_bytes_per_batch': pipe.h2d_bytes,
            'launches_per_batch': 2, 'timing': 'wall clock around the public call incl. host planning + upload'}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--micro-batch', type=int, default=256, help='frames per forward call')
    ap.add_argument('--workload', default='reception2d', choices=['reception2d', 'reception3d', 'spnet_penn', 'spnet_ntu'],
                    help='reception2d = BASELINE configs[1] model (headline); others: configs[2]/[3]/[4] models')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-secondary', action='store_true')
    ap.add_argument('--no-graph', action='store_true', help='plain launches instead of CUDA-graph replays')
    ap.add_argument('--precision', type=int, default=3)
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the outputs of every micro-batch of the last timed step (rank 0\'s shard) to DIR/out<i>.npy; '
                         'that step also copies them on the device; above 64 MB, a fixed sample of rows')
    ap.add_argument('--emulate-world', type=int, default=0,
                    help='analysis only (1 GPU): run rank 0 shard of a W-GPU strong-scaling job without the exchange step')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.impl == 'reference':
        return run_reference(args)
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm')
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))

    peaks = measured_peaks()
    note('building %s' % args.workload)
    model, clip_model, wl_name = build_workload(args.workload)
    model.use_cuda_graph = not args.no_graph
    items_global = CLIPS
    item_frames = FRAMES
    if args.emulate_world > 1:
        assert world == 1, '--emulate-world is a single-process analysis mode'
        run = Runner(torch, model, clip_model, items_global, item_frames, 0, args.emulate_world, args.micro_batch, args.precision)
        run.world = 1
    else:
        run = Runner(torch, model, clip_model, items_global, item_frames, rank, world, args.micro_batch, args.precision)
    comm = None
    if world > 1:               # the exchange step goes through the C ABI (dh_comm_init / dh_allgather_f32)
        from deephar_b200.dist import Comm
        model._ensure_device_weights()
        comm = Comm(model._ctx, rank, world)
        run.comm = comm
    which = 'action' if clip_model else 'pose'
    n_frames = CLIPS * FRAMES                       # global frames per step (strong scaling: fixed)
    micro = run.micro_items * (FRAMES if clip_model else 1)

    note('model built, shard %d frames, micro-batch %d' % (run.frames_local, micro))
    # ---- value: device-resident, CUDA events, max over ranks ------------------------------------------------------
    for _ in range(2):
        run.step(which)                             # first uses: plain launches, then the graph capture
    model.launch_total = 0
    sampler = ClockSampler(local)
    sampler.start()
    ms_step = timed_steps(torch, dist, world, lambda: run.step(which), args.steps, args.warmup,
                          last_fn=(lambda: run.step(which, keep=True)) if args.dump_outputs else None)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        note('outputs of the last timed step -> %s/{%s}.npy' % (args.dump_outputs, ','.join(
            dump_outputs(args.dump_outputs, run.kept))))
    run.kept = None
    launches = int(getattr(model, 'launch_total', 0)) * args.steps // max(1, args.steps + args.warmup)
    value = n_frames / (ms_step / 1000.0)

    note('value: %.1f frames/s (%.2f ms/step)' % (value, ms_step))
    # ---- e2e: public API, pinned host input, H2D + D2H inside the timed region ----------------------------------------
    x_np = run.x_host.numpy()
    bs = run.micro_items
    for _ in range(2):
        model.predict(x_np, batch_size=bs)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        outs = model.predict(x_np, batch_size=bs)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    t = torch.tensor([dt], device='cuda')
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_fps = n_frames * args.steps / float(t.item())
    outs = outs if isinstance(outs, list) else [outs]
    d2h = sum(int(np.prod(o.shape)) * 4 for o in outs)

    note('e2e: %.1f frames/s' % e2e_fps)
    # ---- per-kernel profile (CUDA events around every launch of one extra step) ------------------------------------
    xs = run.x_dev[run.spans[0][0]:run.spans[0][1]]
    prof = model.profile(xs)
    conv_flops = model.conv_flops_per_frame()
    top = max(prof.values(), key=lambda r: r['ms'])
    total_ms = sum(r['ms'] for r in prof.values())
    tf = top['flops'] / (top['ms'] / top['launches'] / 1000.0) / 1e12 if top['flops'] else 0.0
    traffic = ncu_traffic().get(top['label'])
    roofline = {
        'kernel': top['label'], 'bound': 'tensor', 'achieved': tf, 'peak': peaks['bf16_tflops_sustained'],
        'unit': 'TFLOP/s', 'frac': tf / peaks['bf16_tflops_sustained'],
        'traffic': traffic['bytes_per_frame'] * micro if traffic else None,
        'traffic_source': traffic['source'] if traffic else None,
        'share_of_step': top['ms'] / total_ms, 'us_per_launch': 1000.0 * top['ms'] / top['launches'],
        'frames_per_launch': micro,
        'peak_source': peaks['source'] + ' bf16 dense (sustained); kernel math: ' + model.math_mode() +
                       ' (executed tensor FLOPs = 3x the algorithmic ones counted here)',
        'whole_forward_tflops': conv_flops * n_frames / (ms_step / 1000.0) / 1e12 / world,
    }
    if traffic:
        hbm = traffic['bytes_per_frame'] * micro / (top['ms'] / top['launches'] / 1000.0) / 1e9
        roofline['hbm_gbs'] = hbm
        roofline['hbm_frac'] = hbm / peaks['hbm_gbs']
    line = {
        'metric': METRIC, 'value': value, 'unit': 'frames/s', 'n_gpus': world, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': ms_step, 'higher_is_better': True, 'scaling': 'strong',
        'vs_baseline': None, 'dtype': model.math_mode(), 'data': 'synthetic',
        'config': headline_config(world, run.frames_local, micro) if args.workload == 'reception2d' else
        dict(headline_config(world, run.frames_local, micro), workload=wl_name + ' x 32 clips'),
        'clocks': clocks,
        **({'emulated_world': args.emulate_world, 'shard_ms': ms_step,
            'note': 'ANALYSIS ONLY: rank-0 shard of a %d-GPU job on one GPU, no exchange step; value = predicted aggregate'
                    % args.emulate_world} if args.emulate_world > 1 else {}),
        'e2e': {'value': e2e_fps, 'unit': 'frames/s', 'h2d_bytes_per_step': n_frames * 256 * 256 * 3 * 4,
                'd2h_bytes_per_step': d2h * world},
        'gpu_launches': launches * world,
        'launch_mode': ('plain launches of %d kernels per forward' if args.no_graph else
                        'CUDA-graph replay of %d kernels per forward') % len(model._bind(micro).calls),
        'roofline': roofline,
        'kernel_profile': sorted(([r['label'], round(r['ms'], 3), r['launches']] for r in prof.values()),
                                 key=lambda r: -r[1])[:10],
    }

    note('kernel profile done')
    # ---- secondary: soft-argmax micro-benchmarks, the other BASELINE configs, the weak-scaling number ---------------
    if not args.no_secondary:
        sec = {}
        if rank == 0:
            line['softargmax'] = softargmax_microbench(torch, model, peaks)
            sec['softargmax3d'] = softargmax3d_microbench(torch, model, peaks)
            sec['input_pipeline'] = preprocess_microbench(torch)
            sec['C1'] = single_frame_latency(torch, model)
        if world > 1:       # weak scaling: the full 512 frames on every GPU (round-1 mode), device-resident
            wrun = Runner(torch, model, clip_model, CLIPS * world, FRAMES, rank, world, args.micro_batch, args.precision)
            wrun.comm = comm
            ms = timed_steps(torch, dist, world, lambda: wrun.step(which), 3, 2)
            sec['weak'] = {'value': world * n_frames / (ms / 1000.0), 'unit': 'frames/s', 'frames_per_gpu': n_frames,
                           'ms_per_step': ms, 'scaling': 'weak'}
            del wrun
        del run
        model._bound = {}
        torch.cuda.empty_cache()
        if args.workload == 'reception2d':
            for key, wl, items, per, desc in (
                    ('C3', 'reception3d', 32, 1, 'H36M 3-D pose, b32 frames (BASELINE configs[2])'),
                    ('C4', 'spnet_penn', 16, FRAMES, 'PennAction pose+action, 16 clips x 16 frames (BASELINE configs[3])'),
                    ('C5', 'spnet_ntu', 64, FRAMES, 'NTU 3-D pose+action, 64 clips x 16 frames, action all-gather (BASELINE configs[4])')):
                note('secondary %s: building %s' % (key, wl))
                m2, clip2, name2 = build_workload(wl)
                m2.use_cuda_graph = not args.no_graph
                r2 = Runner(torch, m2, clip2, items, per, rank, world, args.micro_batch, args.precision)
                r2.comm = comm          # one communicator per process (it lives on the headline model's context)
                w2 = 'action' if clip2 else 'pose'
                assert r2.items_local > 0, 'every rank needs a shard (the exchange step is a collective)'
                ms = timed_steps(torch, dist, world, lambda: r2.step(w2), 3, 3)
                note('secondary %s: %.2f ms/step' % (key, ms))
                fr = items * per
                sec[key] = {'config': desc, 'model': name2, 'frames_per_step': fr, 'frames_per_gpu': r2.frames_local,
                            'value': fr / (ms / 1000.0), 'unit': 'frames/s', 'ms_per_step': ms,
                            'conv_tflops': m2.conv_flops_per_frame() * fr / (ms / 1000.0) / 1e12 / world,
                            'launches_per_forward': len(m2._bind(r2.micro_items * (FRAMES if clip2 else 1)).calls)}
                del r2, m2
                torch.cuda.empty_cache()
        line['secondary'] = sec

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        note('cpu baseline (torch-CPU port, %d host CPUs)' % (os.cpu_count() or 1))
        r = cpu_port(iters_b32=3, iters_b1=5, warm_b32=1, warm_b1=2)
        med32, med1 = float(np.median(r['b32_times'])), float(np.median(r['b1_times']))
        line['cpu_baseline'] = {'value': 32.0 / med32, 'unit': 'frames/s', 'cores': r['threads'], 'kind': 'port',
                                'sample': 'C2 model, 32 frames (predict batch_size=%d): median of 3 (after 1 warm-up) = '
                                          '%.2f s; C1 (b1) latency median of 5 = %.3f s; torch-CPU fp32 port of the Keras '
                                          'graph (oracle/), %d threads on %d host CPUs (threads and batch size: the '
                                          'fastest of thread_calibration_frames_per_s)'
                                          % (r['chunk'], med32, med1, r['threads'], r['cores']),
                                'c1_b1_latency_s': med1, 'thread_calibration_frames_per_s': r['calibration']}
    note('done')
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        try:
            dist.barrier()
            dist.destroy_process_group()
        except Exception as e:      # the JSON line is already out; never fail the run on teardown
            print('teardown: %r' % (e,), file=sys.stderr)


if __name__ == '__main__':
    main()
