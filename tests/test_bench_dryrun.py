"""bench.py's GPU arm driven on the CPU: the real Workload / Trainer / Engine / schedule compiler with the NumPy kernel
emulation (tests/fake_kernels.py) and stubbed CUDA events, at toy sizes -- catches host-side bugs of the bench (JSON keys,
config plumbing, the separate profiling pass) before a GPU minute is spent.  The numbers it prints mean nothing."""
import io
import json
import sys
import time
from contextlib import redirect_stdout

import numpy as np
import pytest
import torch

import bench
from fake_kernels import FakeKernels
from macaronicusermodeling_b200 import engine


class _Event(object):
    def __init__(self, enable_timing=False):
        self.t = None

    def record(self):
        self.t = time.perf_counter()

    def synchronize(self):
        pass

    def elapsed_time(self, other):
        return max((other.t - self.t) * 1e3, 1e-3)


CONFIGS = {'c3': [], 'c4': ['--config', 'c4', '--users', '3', '--sentences-per-user', '4'],
           'c4_adapt': ['--config', 'c4', '--users', '3', '--sentences-per-user', '4', '--user-adapt'],
           'c5': ['--config', 'c5', '--V', '96', '--sweeps', '4'], 'c3_strong': ['--scaling', 'strong', '--msg-passes', '3']}


def dry_run(monkeypatch, extra, steps=2, warmup=1):
    monkeypatch.setattr(engine, 'Kernels', FakeKernels)
    monkeypatch.setattr(torch.cuda, 'set_device', lambda *_: None)
    monkeypatch.setattr(torch.cuda, 'synchronize', lambda *_: None)
    monkeypatch.setattr(torch.cuda, 'Event', _Event)
    real_tensor = torch.tensor
    monkeypatch.setattr(torch, 'tensor', lambda *a, **k: real_tensor(*a, **{x: y for x, y in k.items() if x != 'device'}))
    monkeypatch.setattr(sys, 'argv', ['bench.py', '--steps', str(steps), '--warmup', str(warmup), '--sentences', '6', '--V', '96',
                                      '--Vd', '12', '--k', '4', '--no-cpu-baseline'] + extra)
    buf = io.StringIO()
    with redirect_stdout(buf):
        bench.ours(bench.parse())
    return json.loads(buf.getvalue().strip().splitlines()[-1])


@pytest.mark.parametrize('extra', list(CONFIGS.values()), ids=list(CONFIGS))
def test_bench_gpu_arm_dry_run(monkeypatch, extra):
    line = dry_run(monkeypatch, extra)
    for key in ('metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling', 'vs_baseline',
                'dtype', 'data', 'config', 'clocks', 'e2e', 'gpu_launches', 'roofline', 'hbm_kernels', 'cpu_baseline', 'host',
                'message_rows'):
        assert key in line, key
    assert line['gpu_launches'] > 0 and line['value'] > 0 and line['e2e']['value'] > 0
    assert line['e2e']['h2d_bytes_per_step'] > 0 and line['e2e']['d2h_bytes_per_step'] == 128
    assert set(line['roofline']) >= {'bound', 'achieved', 'peak', 'unit', 'frac', 'traffic', 'by_passes'}
    assert line['scaling'] == ('strong' if ('c4' in extra or 'strong' in extra) else 'weak')
    assert 'workload' in line['config']


@pytest.mark.parametrize('name', ['c3', 'c4_adapt', 'c5'])
def test_bench_dump_outputs_are_the_last_timed_step(monkeypatch, tmp_path, name):
    """--dump-outputs writes, as float64, what the last of exactly --steps timed steps returned; a second run with the same
    arguments sees the same inputs and writes the same arrays"""
    steps, warmup = 3, 2
    finish, seen = bench.Workload._finish, []

    def record(self, red):
        seen.append(np.array(finish(self, red)))
        return seen[-1]
    monkeypatch.setattr(bench.Workload, '_finish', record)
    runs = []
    for i in range(2):
        del seen[:]
        line = dry_run(monkeypatch, CONFIGS[name] + ['--dump-outputs', str(tmp_path / str(i))], steps=steps, warmup=warmup)
        runs.append({p.stem: np.load(p) for p in (tmp_path / str(i)).iterdir()})
        assert len(line['message_rows']['ranks_switched_to_three_passes_per_step']) == steps
        np.testing.assert_array_equal(runs[-1]['reduced'], seen[warmup + steps - 1])
    want = {'c3': {'reduced', 'theta'}, 'c4_adapt': {'reduced', 'theta', 'user_theta'}, 'c5': {'reduced'}}[name]
    assert set(runs[0]) == want
    for k in want:
        assert runs[0][k].dtype == np.float64
        np.testing.assert_array_equal(runs[0][k], runs[1][k])
    assert runs[0]['reduced'].shape == (16,) and runs[0]['reduced'][14] == (12 if name == 'c4_adapt' else 6)
    if 'theta' in want:
        np.testing.assert_allclose(runs[0]['theta'], line['message_rows']['theta_after_each_step'][warmup + steps - 1], atol=6e-4)
    if name == 'c4_adapt':
        assert runs[0]['user_theta'].shape == (3, 9)


def test_bench_rejects_zero_steps(monkeypatch):
    monkeypatch.setattr(sys, 'argv', ['bench.py', '--steps', '0'])
    with pytest.raises(SystemExit):
        bench.parse()
