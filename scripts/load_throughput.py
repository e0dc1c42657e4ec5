"""Time Model.from_text (K8, the device text parser) against the np.loadtxt path train_cli used before it, from the same files.

    python scripts/load_throughput.py --V 10000 --Vd 2000 --out profiles/r4a_load_throughput.jsonl

Writes V x V (pmi, pmi_w1) and V x Vd (ed, ped) matrices as np.savetxt's default '%.18e' text to a temporary directory
(setup, not timed: 200 distinct random rows, repeated, so that generating ~6 GB of text takes seconds; the parser's work does
not depend on which rows repeat).  In one process the two paths then run alternately (device, np.loadtxt, device) and their
planes and ranges are checked to be identical.  The peak host RSS of each path is measured in a subprocess of its own.
Prints and appends one JSON line: wall seconds and text MB/s per path, the K8 kernel time (CUDA events around every launch),
the file-read and H2D-copy split, the hard-field count, peak RSS (VmHWM; the RSS after torch and the CUDA context are up is
reported beside it), and the card's name and power limit.  The files are read from the page cache (they were just written)."""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, 'tests'))


def write_matrix(path, rows, cols, seed, distinct=200):
    rng = np.random.default_rng(seed)
    lines = []
    for _ in range(distinct):
        a = rng.standard_normal(cols) * 10.0 ** rng.integers(-3, 4, size=cols)
        lines.append((' '.join('%.18e' % x for x in a) + '\n').encode())
    with open(path, 'wb') as f:
        for r in range(rows):
            f.write(lines[(r * 7919) % distinct])


def load(arm, paths, V, Vd):
    import torch
    from macaronicusermodeling_b200.engine import Model
    t0 = time.perf_counter()
    if arm == 'device':
        m = Model.from_text(*paths, V, Vd, 'cuda')
    else:
        from text_load_cases import loadtxt_model
        m = loadtxt_model(Model, paths, 'cuda')
    torch.cuda.synchronize()
    return m, time.perf_counter() - t0


def _status_gb(field):
    with open('/proc/self/status') as f:
        for line in f:
            if line.startswith(field + ':'):
                return int(line.split()[1]) / 2.0 ** 20
    return float('nan')


def child(arm, paths, V, Vd):
    import torch
    torch.zeros(1, device='cuda')                 # CUDA context and torch before the baseline
    base = _status_gb('VmRSS')
    _, dt = load(arm, paths, V, Vd)
    print(json.dumps({'seconds': dt, 'peak_rss_gb': _status_gb('VmHWM'), 'baseline_rss_gb': base}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--V', type=int, default=10000)
    ap.add_argument('--Vd', type=int, default=2000)
    ap.add_argument('--out', default='')
    ap.add_argument('--tmp', default=None)
    ap.add_argument('--child', default='')
    ap.add_argument('--paths', nargs=4)
    a = ap.parse_args()
    if a.child:
        return child(a.child, a.paths, a.V, a.Vd)
    import torch
    from macaronicusermodeling_b200 import build
    from macaronicusermodeling_b200.engine import Kernels, Model
    from macaronicusermodeling_b200.textload import TextLoader
    from text_load_cases import assert_same_model
    assert torch.cuda.is_available(), 'needs a B200'
    build.build()
    tmp = tempfile.mkdtemp(dir=a.tmp)
    try:
        paths = [os.path.join(tmp, n + '.txt') for n in ('pmi', 'pmi_w1', 'ed', 'ped')]
        t0 = time.perf_counter()
        for i, (p, shape) in enumerate(zip(paths, ((a.V, a.V), (a.V, a.V), (a.V, a.Vd), (a.V, a.Vd)))):
            write_matrix(p, shape[0], shape[1], seed=i)
        gen = time.perf_counter() - t0
        nbytes = sum(os.path.getsize(p) for p in paths)
        rss = {}                                  # first, while this process is small: a child's peak starts from ours
        for arm in ('device', 'loadtxt'):
            r = subprocess.run([sys.executable, os.path.abspath(__file__), '--child', arm, '--V', str(a.V), '--Vd', str(a.Vd),
                                '--paths'] + paths, capture_output=True, text=True, check=True)
            rss[arm] = json.loads(r.stdout.strip().splitlines()[-1])
        torch.cuda.set_device(0)
        runs = {'device': [], 'loadtxt': []}
        models = {}
        for arm in ('device', 'loadtxt', 'device'):
            m, dt = load(arm, paths, a.V, a.Vd)
            runs[arm].append(dt)
            models[arm] = m
            if arm == 'device':
                stats = m.load_stats
        assert_same_model(models['device'], models['loadtxt'])
        del models
        # the K8 launches alone (CUDA events around each mlbp_parse_float_text call) and the H2D copies, on one more pass
        k = Kernels()
        kernel_s = [0.0]
        orig = k.call

        def timed(name, *args):
            if name != 'mlbp_parse_float_text':
                return orig(name, *args)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            orig(name, *args)
            e1.record()
            e1.synchronize()
            kernel_s[0] += e0.elapsed_time(e1) / 1e3
        k.call = timed
        loader = TextLoader(k)
        for p, (rows, cols) in zip(paths, ((a.V, a.V), (a.V, a.V), (a.V, a.Vd), (a.V, a.Vd))):
            out = torch.zeros((rows, cols), dtype=torch.float32, device='cuda')
            assert not isinstance(loader.parse(p, rows, cols, out, cols), str)
        pinned = torch.empty(256 << 20, dtype=torch.uint8, pin_memory=True)
        dev = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')
        for rep in range(2):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            dev.copy_(pinned, non_blocking=True)
            e1.record()
            e1.synchronize()
            h2d_gbs = (256 << 20) / (e0.elapsed_time(e1) / 1e3) / 1e9
        smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True,
                             text=True).stdout.strip().splitlines()[0]
        rec = {'what': 'load_throughput', 'V': a.V, 'Vd': a.Vd, 'format': '%.18e', 'text_bytes': nbytes,
               'generate_seconds': round(gen, 1),
               'device_seconds': [round(x, 3) for x in runs['device']], 'loadtxt_seconds': [round(x, 2) for x in runs['loadtxt']],
               'device_MBps': round(nbytes / min(runs['device']) / 1e6, 1),
               'loadtxt_MBps': round(nbytes / min(runs['loadtxt']) / 1e6, 1),
               'k8_kernel_seconds': round(kernel_s[0], 4), 'k8_GBps': round(nbytes / kernel_s[0] / 1e9, 2),
               'file_read_seconds': round(loader.stats['read_seconds'], 3),
               'h2d_seconds_at_measured_rate': round(nbytes / (h2d_gbs * 1e9), 3), 'h2d_GBps_pinned_256MB': round(h2d_gbs, 1),
               'hard_fields': stats['hard_fields'], 'chunks': stats['chunks'],
               'peak_rss_gb': {arm: round(rss[arm]['peak_rss_gb'], 2) for arm in rss},
               'rss_before_load_gb': {arm: round(rss[arm]['baseline_rss_gb'], 2) for arm in rss},
               'page_cache': 'files just written: read from the page cache, not from disk',
               'subprocess_seconds': {arm: round(rss[arm]['seconds'], 2) for arm in rss},
               'gpu': smi}
        line = json.dumps(rec)
        print(line)
        if a.out:
            with open(a.out, 'a') as f:
                f.write(line + '\n')
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == '__main__':
    main()
