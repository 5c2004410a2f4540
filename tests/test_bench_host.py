"""bench.py's host logic without a device: the strong-scaling shard arithmetic of every workload at N = 1, 2, 4, 8, the
nvidia-smi clock parser, and the contract keys of the reference-arm line (the CPU port itself is stubbed: it is timed for
real by the driver)."""
import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402

# (global items, frames per item, clip model) of the headline and the secondary configs (bench.py main)
WORKLOADS = {'headline': (32, 16, False), 'weak x8': (32 * 8, 16, False), 'C3': (32, 1, False), 'C4': (16, 16, True),
             'C5': (64, 16, True)}


@pytest.mark.parametrize('world', [1, 2, 4, 8])
@pytest.mark.parametrize('name', sorted(WORKLOADS))
def test_every_rank_gets_a_contiguous_non_empty_shard(name, world):
    items, per, clip = WORKLOADS[name]
    plans = [bench.shard_plan(items, per, r, world, 256, clip) for r in range(world)]
    assert [p['first'] for p in plans] == list(np.cumsum([0] + [p['items_local'] for p in plans[:-1]]))
    assert sum(p['items_local'] for p in plans) == items and all(p['items_local'] > 0 for p in plans)
    for p in plans:
        assert p['frames_local'] == p['items_local'] * per
        assert p['lead'] == (p['items_local'] if clip else p['frames_local'])
        frames_per_call = p['micro_items'] * (bench.FRAMES if clip else 1)
        assert 1 <= frames_per_call <= 256
        assert p['spans'][0][0] == 0 and p['spans'][-1][1] == p['lead']
        assert all(a1 == b0 for (_, b0), (a1, _) in zip(p['spans'], p['spans'][1:]))
    if name == 'headline':                  # SURVEY 8e: 32 / 16 / 8 / 4 clips per GPU
        assert plans[0]['items_local'] == 32 // world and plans[0]['frames_local'] == 512 // world


def test_clock_sampler_parses_nvidia_smi_lines():
    s = bench.ClockSampler(0)
    s.proc = type('P', (), {'terminate': lambda self: None, 'wait': lambda self, timeout=None: 0, 'kill': lambda self: None})()
    s.lines = ['0, 1890, 1965, 830.1, 0x0000000000000004, Not Active, Not Active, Not Active, Active',
               '0, 1905, 1965, 790.0, 0x0000000000000000, Not Active, Not Active, Not Active, Not Active',
               '0, 1875, 1965, 845.5, 0x0000000000000004, Not Active, Not Active, Not Active, Active',
               'garbage', '0, [N/A], 1965, 1, 0, Not Active, Not Active, Not Active, Not Active']
    got = s.stop()
    assert got == {'sm_mhz': 1890.0, 'sm_max_mhz': 1965.0, 'reasons': ['sw_power_cap'], 'samples': 3}
    empty = bench.ClockSampler(0)
    assert empty.stop()['reasons'] == ['nvidia-smi unavailable']


def test_reference_arm_line_has_the_contract_keys(monkeypatch, capsys):
    monkeypatch.setattr(bench, 'cpu_port', lambda **kw: {'b32_times': [3.0, 3.2, 2.8], 'b1_times': [0.1] * 10, 'cores': 128,
                                                          'threads': 16, 'chunk': 8, 'calibration': {'16 threads, b8': 11.0}})
    monkeypatch.setenv('RANK', '0')
    args = type('A', (), {'steps': 3, 'warmup': 1, 'gpus': 4, 'micro_batch': 256})()
    bench.run_reference(args)
    line = json.loads(capsys.readouterr().out.strip())
    assert line['impl'] == 'reference' and line['metric'] == bench.METRIC and line['unit'] == 'frames/s'
    assert line['value'] == pytest.approx(32.0 / 3.0) and line['ms_per_step'] == pytest.approx(3000.0)
    assert line['n_gpus'] == 4 and line['higher_is_better'] is True and line['vs_baseline'] is None
    assert line['e2e'] == {'value': line['value'], 'unit': 'frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
    assert line['cpu_baseline']['kind'] == 'port' and line['cpu_baseline']['cores'] == 16
    assert line['cpu_baseline']['value'] == line['value'] and 'predict batch_size=8' in line['cpu_baseline']['sample']
    # same `config` as the product arm prints for the same N (the driver compares them)
    assert line['config'] == bench.headline_config(4, 128, 128)
    monkeypatch.setenv('RANK', '1')             # the other ranks of a torchrun launch print nothing
    bench.run_reference(args)
    assert capsys.readouterr().out == ''


@pytest.mark.timeout(600)
@pytest.mark.parametrize('world', [1, 8])
def test_bench_control_flow_on_the_stand_in_device(world, tmp_path):
    """bench.py from its first line to its JSON line on tests/fake_cuda.py (host memory as device memory, inert streams /
    events / graphs, gloo for NCCL, every device entry point of the C library a no-op): model builds, buffer binding,
    CUDA-graph branch, the copy-pipelined predict of the e2e leg, the per-kernel profile, the exchange step through
    dist.Comm, the weak-scaling and C3 / C4 / C5 secondary runs with their shards, at N = 1 and N = 8 ranks.  The numbers
    mean nothing; the contract keys and the shard sizes do."""
    import socket
    import subprocess
    fake = os.path.join(ROOT, 'tests', 'fake_cuda.py')
    tail = [fake, os.path.join(ROOT, 'bench.py'), '--gpus', str(world), '--steps', '1', '--warmup', '3', '--no-cpu-baseline',
            '--dump-outputs', str(tmp_path / 'outs')]
    if world == 1:
        cmd = [sys.executable] + tail
    else:
        s = socket.socket()
        s.bind(('127.0.0.1', 0))
        port = s.getsockname()[1]
        s.close()
        cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', str(world),
               '--master-addr', '127.0.0.1', '--master-port', str(port)] + tail
    env = {k: v for k, v in os.environ.items() if k not in ('RANK', 'WORLD_SIZE', 'LOCAL_RANK')}
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=580, cwd=ROOT, env=env)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith('{')]
    assert len(lines) == 1, 'exactly one JSON line, from rank 0'
    d = json.loads(lines[0])
    assert d['metric'] == bench.METRIC and d['unit'] == 'frames/s' and d['n_gpus'] == world and d['scaling'] == 'strong'
    assert d['steps'] == 1 and d['warmup'] == 3 and d['higher_is_better'] is True and d['vs_baseline'] is None
    assert d['value'] > 0 and d['ms_per_step'] > 0 and d['data'] == 'synthetic' and 'bf16x3' in d['dtype']
    assert d['config'] == bench.headline_config(world, 512 // world, min(256, 512 // world))
    assert set(d['clocks']) >= {'sm_mhz', 'sm_max_mhz', 'reasons'}
    assert d['e2e']['value'] > 0 and d['e2e']['h2d_bytes_per_step'] == 512 * 256 * 256 * 3 * 4 and d['e2e']['d2h_bytes_per_step'] > 0
    assert d['gpu_launches'] >= 127 * world and '127 kernels per forward' in d['launch_mode']
    assert set(d['roofline']) >= {'kernel', 'bound', 'achieved', 'peak', 'unit', 'frac', 'traffic'}
    # the last timed step's outputs: per block (pose, visibility) of every frame of rank 0's shard -- both 256-frame
    # forwards at N = 1
    dumped = sorted(os.listdir(tmp_path / 'outs'))
    assert dumped == ['out%02d.npy' % i for i in range(16)]
    shapes = [np.load(tmp_path / 'outs' / f).shape for f in dumped]
    assert shapes == [(512 // world, 16, 2), (512 // world, 16, 1)] * 8
    assert len(d['kernel_profile']) == 10 and 'cpu_baseline' not in d
    sec = d['secondary']
    assert set(sec) >= {'softargmax3d', 'input_pipeline', 'C1', 'C3', 'C4', 'C5'} and ('weak' in sec) == (world > 1)
    assert (sec['C3']['frames_per_gpu'], sec['C4']['frames_per_gpu'], sec['C5']['frames_per_gpu']) == \
        (32 // world, 256 // world, 1024 // world)
    assert (sec['C3']['launches_per_forward'], sec['C4']['launches_per_forward'], sec['C5']['launches_per_forward']) == (134, 345, 237)
    if world > 1:
        assert sec['weak']['frames_per_gpu'] == 512 and sec['weak']['scaling'] == 'weak'
