#!/usr/bin/env python
"""LBP training throughput on B200 (BASELINE.json metric) next to the CPU path.

    python bench.py --gpus N --steps K --warmup W            our arm (torchrun launches N ranks for N > 1)
    python bench.py --impl reference --gpus N --steps K ...  the CPU arm: the oracle port of the reference's path
                                                             (one process with threaded BLAS AND a train_mp.py-style pool of
                                                             forked single-threaded workers; the faster one is the value)
    python bench.py ... --dump-outputs DIR                   also writes the last timed step's outputs as DIR/<name>.npy

A step = one synchronous minibatch SGD step of the hot path over one batch of synthetic macaronic sentences:
table build for the current theta (K2), unary products (K1), 3 sweeps of level-batched message passing
(K3 + K4), gradient (K4 + K6), marginals / log-posterior / precision counts (K5), the 16-float64 all-reduce and
the theta update.  Workload at N = 1 is BASELINE config C3 (4096 sentences, V = 10 000, Vd = 2 000, k = 20
predicted tokens, 3 sweeps); with N > 1 every rank gets its own 4096 sentences (weak scaling, no data-path
collective besides the theta-gradient all-reduce).

`value` is measured with the sentence index arrays already resident in HBM; `e2e` re-measures the same steps
through the public API with HOST sentence arrays (H2D of the index arrays and schedules, D2H of the reduced
gradient inside the timed region).  The feature planes are model state (the reference loads them once,
train.py:589-612) and stay resident in both.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

METRIC = 'LBP sentences/sec (train, 3 iters, V=10k)'
UNIT = 'sentences/s'


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=3)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--sentences', type=int, default=4096, help='sentences per GPU per step')
    ap.add_argument('--V', type=int, default=10000)
    ap.add_argument('--Vd', type=int, default=2000)
    ap.add_argument('--k', type=int, default=20)
    ap.add_argument('--g', type=int, default=0)
    ap.add_argument('--sweeps', type=int, default=3)
    ap.add_argument('--workspace-gb', type=float, default=96.0)
    ap.add_argument('--cpu-sample', type=int, default=6, help='sentences timed on the CPU for cpu_baseline')
    ap.add_argument('--ref-sample', type=int, default=0, help='sentences per step of the process-pool CPU variant (0 = one per host core)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-literal', action='store_true', help='CPU arm: skip the timed sample of the literal (per-message) reference restatement')
    ap.add_argument('--gemm-slice-pairs', type=int, default=None, help='M pairs per three-pass K4 launch (default: Engine rule; 0 = one launch per level, A/B probe)')
    ap.add_argument('--gemm-impl', type=int, default=0, help='K4 variant / flags (include/mlbp.h; A/B probes)')
    ap.add_argument('--grad-b-terms', type=int, default=1, help='2 = keep the table lo half in the gradient rows (A/B probe)')
    ap.add_argument('--msg-passes', type=int, default=None, help='2 / 3 = two- / three-pass message rows (A/B probes); default: Engine rule (one pass where V >= 4096)')
    ap.add_argument('--config', default='c3', choices=['c3', 'c4', 'c5'],
                    help='BASELINE config: c3 batched training (the headline metric), c4 multi-user training (512 users x 100 '
                         'sentences, users sharded), c5 inference-only belief sweep (V=50k, 10 sweeps)')
    ap.add_argument('--scaling', default='weak', choices=['weak', 'strong'],
                    help='c3 / c5: weak = --sentences per GPU, strong = --sentences in total; c4 is always strong (fixed users)')
    ap.add_argument('--users', type=int, default=512)
    ap.add_argument('--sentences-per-user', type=int, default=100)
    ap.add_argument('--user-adapt', action='store_true', help='c4: every user owns a theta pair (train.py --user_adapt)')
    ap.add_argument('--traffic-file', default='r2_k4_traffic.json', help='profiles/<file>: DRAM bytes per K4 launch from the committed ncu capture')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='GPU arm: write what the last timed step returned as DIR/<name>.npy (float64), to compare two builds on '
                         'the same seeded inputs')
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error('--steps must be at least 1 and --warmup at least 0')
    if a.dump_outputs and a.impl != 'ours':
        ap.error('--dump-outputs writes the outputs of the GPU arm (--impl ours)')
    if a.config == 'c5':                                             # run-predictions.sh:12 at the size BASELINE names
        d = ap.parse_args([])
        if a.V == d.V: a.V = 50000
        if a.sweeps == d.sweeps: a.sweeps = 10
        if a.sentences == d.sentences: a.sentences = 64
        if a.workspace_gb == d.workspace_gb: a.workspace_gb = 40.0
    return a


def workload_name(a):
    if a.config == 'c4':
        return ('C4 multi-user training: %d users x %d sentences per step (one pass over every user), users sharded over the GPUs, '
                'V=%d, Vd=%d, k=%d predicted + %d given tokens, %d sweeps, %s' % (
                    a.users, a.sentences_per_user, a.V, a.Vd, a.k, a.g, a.sweeps,
                    'per-user theta (--user_adapt: one table build per user)' if a.user_adapt else 'shared theta'))
    if a.config == 'c5':
        return ('C5 inference-only belief sweep: %d sentences%s/step, V=%d, Vd=%d, k=%d predicted + %d given tokens, %d sweeps, '
                'marginals + top-1 + log-posterior + precision counts' % (a.sentences, '' if a.scaling == 'strong' else '/GPU',
                                                                           a.V, a.Vd, a.k, a.g, a.sweeps))
    return ('C3 batched training: %d sentences%s/step, V=%d, Vd=%d, k=%d predicted + %d given tokens, %d sweeps, '
            'shared pairwise tables' % (a.sentences, ' in total' if a.scaling == 'strong' else '/GPU', a.V, a.Vd, a.k, a.g, a.sweeps))


def metric_name(a):
    if a.config == 'c5':
        return 'LBP sentences/sec (inference, %d iters, V=%dk)' % (a.sweeps, a.V // 1000)
    return METRIC


def scaling_name(a):
    return 'strong' if (a.config == 'c4' or a.scaling == 'strong') else 'weak'


def make_inputs(a, rank, n_sent):
    from macaronicusermodeling_b200 import synth
    model = synth.make_model(a.V, a.Vd, seed=1234, dtype=np.float32)
    sents = synth.make_corpus(model, n_sent, k=a.k, g=a.g, seed=1234 + 7919 * rank)
    return model, sents


def theta0():
    # mid-training magnitudes (theta = 0, the reference's start, makes every potential 1 and every belief tie)
    return np.array([0.8, 0.5, -0.3]), np.array([1.0, -0.6, 0.5, 0.3, 0.4, -0.2])


def local_roots(corpus, sweeps, rng):
    k = np.diff(corpus.var_off)
    return (rng.random((corpus.n_sent, 1 + sweeps)) * k[:, None]).astype(np.int32)


# ----------------------------------------------------------------------------------------------- clocks
class ClockSampler(object):
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.idx), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '200'], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, r[5:9]):
                if v.lower().startswith('active') and not v.lower().startswith('not'):
                    reasons.add(n)
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': sorted(reasons), 'samples': len(sm)}


# ----------------------------------------------------------------------------------------------- CPU arm
def cpu_run(a, n_sent, model=None, sents=None):
    """the oracle's fast evaluator (hoisted potentials, closed-form gradient, level-batched BLAS) -- the strongest
    fair CPU variant of the reference's path (BASELINE.md §3), all host threads"""
    from oracle import lbp_oracle as orc
    from macaronicusermodeling_b200 import synth
    if model is None:
        model, sents = make_inputs(a, 0, n_sent)
    m64 = {k: (np.asarray(v, dtype=np.float64) if hasattr(v, 'dtype') else v) for k, v in model.items()}
    te, td = theta0()
    roots = synth.draw_roots(sents[:n_sent], a.sweeps, seed=5)
    t0 = time.perf_counter()
    tb = orc.Tables(m64, te, td)
    t_tables = time.perf_counter() - t0
    t0 = time.perf_counter()
    for s, r in zip(sents[:n_sent], roots):
        orc.run_fast(tb, s, r, a.sweeps)
    t_sent = time.perf_counter() - t0
    return t_tables, t_sent, tb


def host_threads():
    try:
        from threadpoolctl import threadpool_info
        n = [p.get('num_threads', 1) for p in threadpool_info() if p.get('user_api') == 'blas']
        if n:
            return int(max(n))
    except Exception:
        pass
    return os.cpu_count() or 1


# train_mp.py-style CPU variant (train_mp.py:634-649: a multiprocessing.Pool, one sentence per task): the workers are
# forked AFTER the theta-only tables exist, so they inherit them copy-on-write instead of unpickling 4.8 GB per task
# (SURVEY.md section 8(d) names this deviation), and every worker runs single-threaded BLAS.
_POOL = {}


def _pool_init():
    from threadpoolctl import threadpool_limits
    _POOL['limit'] = threadpool_limits(limits=1, user_api='blas')


def _pool_sentence(i):
    _POOL['orc'].run_fast(_POOL['tb'], _POOL['sents'][i], _POOL['roots'][i], _POOL['sweeps'])
    return i


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def literal_reference_sample(a, m64, te, td):
    """SURVEY.md section 8(d) variant (i): the reference's path as it stands (train.py:357-397 -> LBP.py), restated op for op by
    oracle.run_literal -- potentials exp(phi . theta) rebuilt per sentence (train.py:218-253), one V x V dgemv per message
    (LBP.py:509 / :518), dense pairwise beliefs per factor (LBP.py:566-610).  A k = 20 sentence of the workload takes minutes
    that way, so two SHORT sentences of the same model (3 and 4 predicted tokens: 3 and 6 pairwise factors) are timed and the
    workload's sentence is extrapolated linearly in the number of pairwise factors (k (k - 1) / 2): every message update and
    every belief belongs to one factor, the potentials are a per-sentence constant."""
    from oracle import lbp_oracle as orc
    from macaronicusermodeling_b200 import synth
    try:
        t = {}
        for k in (3, 4):
            sents = synth.make_corpus({'V': a.V, 'Vd': a.Vd}, 1, k=k, g=0, seed=99)
            roots = synth.draw_roots(sents, a.sweeps, seed=5)
            t0 = time.perf_counter()
            orc.run_literal(m64, sents[0], te, td, roots[0], a.sweeps, keep_messages=False)
            t[k] = time.perf_counter() - t0
        per_factor = max((t[4] - t[3]) / 3.0, 0.0)
        per_sentence = t[3] - 3.0 * per_factor
        n_pair = a.k * (a.k - 1) // 2
        est = per_sentence + n_pair * per_factor
        return {'value': 1.0 / est, 'unit': UNIT, 'kind': 'port (literal: oracle.run_literal, op for op)', 'extrapolated': True,
                'threads': host_threads(), 'measured_s': {'k=3 (3 pairwise factors)': t[3], 'k=4 (6 pairwise factors)': t[4]},
                'per_pairwise_factor_s': per_factor, 'per_sentence_constant_s': per_sentence,
                'seconds_per_workload_sentence': est,
                'note': 'k = %d: %d pairwise factors; linear in the factor count, measured on two short sentences at V = %d' % (a.k, n_pair, a.V)}
    except Exception as e:                                      # never lose the arm's line over the slow variant
        return {'value': None, 'error': str(e)[:200]}


def reference_arm(a):
    """Two CPU variants of the same port are timed over the same K steps and the FASTER one is the arm's value:
    `blas_threads` = one process, every level's dgemm threaded by the BLAS; `process_pool` = train_mp.py's layout,
    one worker process per host core, one sentence per task."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    if a.config == 'c5':
        return reference_arm_c5(a)
    import multiprocessing as mp
    from oracle import lbp_oracle as orc
    from macaronicusermodeling_b200 import synth
    workers = host_cores()
    n_thr = 2
    n_pool = a.ref_sample if a.ref_sample > 0 else workers
    model, sents = make_inputs(a, 0, max(n_pool, n_thr))
    m64 = {k: (np.asarray(v, dtype=np.float64) if hasattr(v, 'dtype') else v) for k, v in model.items()}
    te, td = theta0()
    roots = synth.draw_roots(sents, a.sweeps, seed=5)

    try:                                                        # torchrun exports OMP_NUM_THREADS=1: give the BLAS every host core back
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=workers, user_api='blas')
    except Exception:
        pass

    # theta changes once per SGD step, so the theta-only tables are rebuilt once per step of a.sentences sentences;
    # the bounded sample below is charged its share of that build (n / a.sentences), like the GPU arm amortises K2
    t0 = time.perf_counter()
    tb = orc.Tables(m64, te, td)
    t_tab = time.perf_counter() - t0

    def timed(step, n):
        for _ in range(a.warmup):
            step()
        t0 = time.perf_counter()
        for _ in range(a.steps):
            step()
        dt = time.perf_counter() - t0 + a.steps * t_tab * n / float(a.sentences)
        return n * a.steps / dt, dt

    def step_threads():
        for s, r in zip(sents[:n_thr], roots[:n_thr]):
            orc.run_fast(tb, s, r, a.sweeps)

    v_thr, dt_thr = timed(step_threads, n_thr)
    blas_threads = host_threads()

    _POOL.update(orc=orc, tb=tb, sents=sents, roots=roots, sweeps=a.sweeps)
    with mp.get_context('fork').Pool(workers, initializer=_pool_init) as pool:
        v_pool, dt_pool = timed(lambda: pool.map(_pool_sentence, range(n_pool), chunksize=1), n_pool)

    literal = None if a.no_literal else literal_reference_sample(a, m64, te, td)

    if v_pool >= v_thr:
        v, dt, n, variant, cores = v_pool, dt_pool, n_pool, 'process_pool', workers
    else:
        v, dt, n, variant, cores = v_thr, dt_thr, n_thr, 'blas_threads', blas_threads
    line = {'impl': 'reference', 'metric': METRIC, 'value': v, 'unit': UNIT, 'n_gpus': a.gpus, 'steps': a.steps,
            'warmup': a.warmup, 'ms_per_step': 1e3 * dt / a.steps, 'higher_is_better': True, 'scaling': scaling_name(a),
            'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
            'config': {'workload': workload_name(a),
                       'note': 'CPU arm: oracle port of the reference path, fast variant (potentials hoisted to once '
                               'per step, closed-form gradient, level-batched dgemm); each step is a bounded sample of '
                               '%d sentences of the workload; the literal per-message reference restatement is ~100x '
                               'slower (cpu_baseline.variants.literal: timed on two short sentences, extrapolated)' % n},
            'cpu_baseline': {'value': v, 'unit': UNIT, 'cores': cores, 'kind': 'port', 'variant': variant,
                             'variants': {'process_pool': {'value': v_pool, 'workers': workers, 'blas_threads_per_worker': 1,
                                                           'sentences_per_step': n_pool},
                                          'blas_threads': {'value': v_thr, 'threads': blas_threads, 'sentences_per_step': n_thr},
                                          'literal': literal},
                             'sample': '%d sentences x %d steps (%s: %s) + the amortised share of one %.1f s table build per '
                                       '%d-sentence step' % (n, a.steps, variant,
                                                             'train_mp.py-style pool of %d forked single-threaded workers' % workers
                                                             if variant == 'process_pool' else 'one process, %d BLAS threads' % blas_threads,
                                                             t_tab, a.sentences)},
            'e2e': {'value': v, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    print(json.dumps(line), flush=True)


def reference_arm_c5(a):
    """C5 on the host: the oracle's chunked evaluator (V = 50 000 float64 tables do not fit: 20 GB each), all host threads,
    a bounded sample of sentences advanced in lock step through ONE pass over the feature planes per schedule level."""
    from oracle import lbp_oracle as orc
    from macaronicusermodeling_b200 import synth
    n = a.ref_sample if a.ref_sample > 0 else 4
    model = synth.make_model_large(a.V, a.Vd, seed=1234)
    sents = synth.make_corpus({'V': a.V, 'Vd': a.Vd}, n, k=a.k, g=a.g, seed=1234)
    roots = synth.draw_roots(sents, a.sweeps, seed=5)
    te, td = theta0()
    t0 = time.perf_counter()
    orc.run_chunked(model, sents, te, td, roots, a.sweeps)
    dt = time.perf_counter() - t0
    v = n / dt
    line = {'impl': 'reference', 'metric': metric_name(a), 'value': v, 'unit': UNIT, 'n_gpus': a.gpus, 'steps': 1, 'warmup': 0,
            'ms_per_step': 1e3 * dt, 'higher_is_better': True, 'scaling': scaling_name(a), 'vs_baseline': None, 'dtype': 'f64',
            'data': 'synthetic', 'config': {'workload': workload_name(a), 'note': 'CPU arm: chunked float64 oracle, one untimed-warm-up-free pass'},
            'cpu_baseline': {'value': v, 'unit': UNIT, 'cores': host_cores(), 'kind': 'port', 'variant': 'chunked',
                             'sample': '%d sentences advanced in lock step, tables rebuilt on the fly per schedule level (%.0f s)' % (n, dt)},
            'e2e': {'value': v, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}, 'gpu_launches': 0}
    print(json.dumps(line), flush=True)


def cpu_baseline_subprocess(a):
    """cpu_baseline of the GPU arm = the reference arm run in a FRESH interpreter (no CUDA context, no NCCL threads in the
    process that forks the worker pool), one timed step after one warm-up step."""
    cmd = [sys.executable, os.path.abspath(__file__), '--impl', 'reference', '--steps', '1', '--warmup', '1',
           '--sentences', str(a.sentences), '--V', str(a.V), '--Vd', str(a.Vd), '--k', str(a.k), '--g', str(a.g),
           '--sweeps', str(a.sweeps), '--ref-sample', str(a.ref_sample), '--config', a.config, '--scaling', a.scaling,
           '--users', str(a.users), '--sentences-per-user', str(a.sentences_per_user)] + (['--user-adapt'] if a.user_adapt else []) + \
        (['--no-literal'] if a.no_literal else [])
    env = {k: v for k, v in os.environ.items() if k not in ('RANK', 'LOCAL_RANK', 'WORLD_SIZE', 'LOCAL_WORLD_SIZE')}
    out = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900, env=env, check=True).stdout
    for ln in reversed(out.splitlines()):
        if ln.startswith('{'):
            return json.loads(ln)['cpu_baseline']
    raise RuntimeError('no JSON line from the CPU arm')


# ----------------------------------------------------------------------------------------------- GPU arm
class Workload(object):
    """One rank's share of a BASELINE config: builds the inputs, exposes step() (index arrays resident) and step_e2e()
    (fresh host arrays every step)."""

    def __init__(self, a, rank, world, eng_kw):
        import torch
        from macaronicusermodeling_b200 import synth
        from macaronicusermodeling_b200.engine import Corpus, Engine, Kernels, Model
        from macaronicusermodeling_b200.trainer import AdaptTrainer, Trainer
        self.a, self.rank, self.world, self.Corpus = a, rank, world, Corpus
        self.rng = np.random.default_rng(99 + rank)
        self.train = a.config != 'c5'
        if a.config == 'c5':
            model = synth.make_model_large(a.V, a.Vd, seed=1234)
        else:
            model = synth.make_model(a.V, a.Vd, seed=1234, dtype=np.float32)
        k = Kernels()
        self.eng = Engine(Model.from_dict(model, k.device), kernels=k, workspace_bytes=int(a.workspace_gb * (1 << 30)), **eng_kw)
        small = {'V': a.V, 'Vd': a.Vd}
        del model
        if a.config == 'c4':
            users = ['user%03d' % u for u in range(a.users)]
            self.mine = users[rank::world]                                  # users are the unit of sharding
            per_user = {u: synth.make_corpus(small, a.sentences_per_user, k=a.k, g=a.g, seed=1000 + 17 * users.index(u), users=[u])
                        for u in self.mine}
            self.n_global = a.users * a.sentences_per_user
            self.n_local = len(self.mine) * a.sentences_per_user
            if a.user_adapt:
                self.tr = AdaptTrainer(self.eng, self.mine, reg_param=0.2, ua_scale=0.5, N=self.n_global, sweeps=a.sweeps)
                for u in self.mine:
                    self.tr.domain2theta[u] = tuple(x.copy() for x in theta0())
                self.batches = [(u, Corpus(per_user[u])) for u in self.mine]
                self.corpus = None
            else:
                self.tr = Trainer(self.eng, reg_param=0.2, N=self.n_global, sweeps=a.sweeps)
                self.corpus = Corpus([s for u in self.mine for s in per_user[u]])
            self.lr = 0.01 / self.n_global                                  # small steps: theta stays in the benchmark's regime
        else:
            per_rank = a.sentences // world if a.scaling == 'strong' else a.sentences
            self.n_local = per_rank
            self.n_global = per_rank * world
            seed = 1234 + 7919 * rank
            self.corpus = Corpus(synth.make_corpus(small, per_rank, k=a.k, g=a.g, seed=seed))
            self.tr = Trainer(self.eng, reg_param=0.2, N=self.n_global, sweeps=a.sweeps)
            self.lr = 0.1 / float(self.n_global)    # minibatch sum of gradients: the reference's 0.1 per sentence, averaged
        self.tr.theta_ee, self.tr.theta_ed = theta0()
        self.parts = self.eng.prepare(self.corpus, a.sweeps, self.train) if self.corpus is not None else None
        self._next_roots = None
        self.peaked = []                                                    # red[15] of every step
        self.all_peaked = []
        self.thetas = []

    def roots(self, corpus):
        return local_roots(corpus, self.a.sweeps, self.rng)

    def _finish(self, red):
        if self.train:
            h = self.tr.apply(red, self.lr)
        else:
            h = red.cpu().numpy()                                           # the step's device -> host read
        self.peaked.append(float(h[15]))
        self.all_peaked.append(float(h[15]))
        self.thetas.append([round(float(x), 3) for x in list(self.tr.theta_ee) + list(self.tr.theta_ed)])
        self.last = h
        return h

    def outputs(self):
        """What the last step handed its caller: the reduced 16-vector (Trainer.step) and, when training, theta after the update
        (theta_ee then theta_ed) and, with per-user theta, this rank's users' theta in user order."""
        out = {'reduced': self.last}
        if self.train:
            out['theta'] = np.concatenate([self.tr.theta_ee, self.tr.theta_ed])
        if self.corpus is None:
            out['user_theta'] = np.array([np.concatenate(self.tr.domain2theta[u]) for u in self.mine])
        return {k: np.array(v, dtype=np.float64) for k, v in out.items()}

    def step(self):
        if self.corpus is None:                                             # c4 --user-adapt: one engine pass per user
            return self._finish(self.tr.step_domains([(u, c, self.roots(c)) for u, c in self.batches], self.lr))
        # the roots of the NEXT step are drawn now (they do not depend on theta): the trainer compiles that step's first
        # micro-batch schedule in the background while the host waits for this step's all-reduce
        roots = self._next_roots if self._next_roots is not None else self.roots(self.corpus)
        self._next_roots = self.roots(self.corpus)
        if self.train:
            return self._finish(self.tr.step(self.parts, roots, self.lr, next_roots=self._next_roots))
        return self._finish(self.tr.eval_step(self.parts, roots, next_roots=self._next_roots))

    def step_e2e(self):
        fresh = lambda c: self.Corpus(**{f: getattr(c, f) for f in self.Corpus.FIELDS})   # nothing cached on the device
        if self.corpus is None:
            keep = [(u, fresh(c)) for u, c in self.batches]
            return keep, self._finish(self.tr.step_domains([(u, c, self.roots(c)) for u, c in keep], self.lr))
        c = fresh(self.corpus)
        if self.train:
            return c, self._finish(self.tr.step(c, self.roots(c), self.lr))
        return c, self._finish(self.tr.eval_step(c, self.roots(c)))

    def index_bytes(self):
        cs = [self.corpus] if self.corpus is not None else [c for _, c in self.batches]
        return sum(getattr(c, f).nbytes for c in cs for f in self.Corpus.FIELDS if f != 'var_pos') + \
            sum(c.n_sent for c in cs) * (1 + self.a.sweeps) * 4


def ours(a):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    lws = int(os.environ.get('LOCAL_WORLD_SIZE', str(world)))
    os.environ.setdefault('MLBP_PLAN_THREADS', str(max(2, min(16, (os.cpu_count() or 8) // max(lws, 1)))))
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    assert world == a.gpus or world == 1, (world, a.gpus)

    w = Workload(a, rank, world, dict(grad_b_terms=a.grad_b_terms, gemm_slice_pairs=a.gemm_slice_pairs, gemm_impl=a.gemm_impl,
                                      msg_passes=a.msg_passes))
    eng = w.eng

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """exactly `steps` calls of fn between two CUDA events on the launching stream, barrier + synchronize on both sides,
        max over ranks"""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device='cuda')
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for _ in range(a.warmup):
        w.step()
    # ---- value: device-timed, index arrays resident, NO per-kernel events inside the timed region
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0, w.peaked = eng.launches, []
    t_plan0 = eng.plan_seconds
    tm0 = (eng.plan_template_hits, eng.plan_template_misses)
    ms = timed(w.step, a.steps)
    clocks = sampler.stop() if rank == 0 else None
    launches = eng.launches - l0
    plan_s_per_step = (eng.plan_seconds - t_plan0) / a.steps
    tm1 = (eng.plan_template_hits, eng.plan_template_misses)
    peaked_value = list(w.peaked)
    value = w.n_global * a.steps / (ms / 1e3)
    if a.dump_outputs and rank == 0:                          # before the e2e and profiling steps move theta on
        os.makedirs(a.dump_outputs, exist_ok=True)
        for name, x in w.outputs().items():
            np.save(os.path.join(a.dump_outputs, name + '.npy'), x)

    # ---- e2e: host sentence arrays in, reduced gradient out, every step
    e2e = None
    if not a.no_e2e:
        w.step_e2e()
        blob0 = eng.blob_bytes
        ms2 = timed(w.step_e2e, a.steps)
        # index arrays of every micro-batch slice + roots are re-uploaded; schedules (plan blobs) are uploaded in both modes
        e2e = {'value': w.n_global * a.steps / (ms2 / 1e3), 'unit': UNIT,
               'h2d_bytes_per_step': int(w.index_bytes() + (eng.blob_bytes - blob0) / a.steps), 'd2h_bytes_per_step': 16 * 8,
               'ms_per_step': ms2 / a.steps}

    # ---- profiling pass (separate from both timed regions): a CUDA-event pair around every kernel launch
    eng.profile_gemm = eng.profile_kernels = True
    eng.gemm_events, eng.kernel_events = [], []
    w.peaked = []
    p_steps = max(1, min(a.steps, 3))

    def prof_step():
        eng.event_tag = len(w.peaked)
        w.step()
    ms_prof = timed(prof_step, p_steps)
    eng.profile_gemm = eng.profile_kernels = False
    pass_stats = eng.pass_stats()
    by_passes = {}
    gemm_ms = gemm_rows = gemm_pass_rows = 0.0
    by_role = {}
    for x, y, r, p, gated, tag, role in eng.gemm_events:
        code = int(w.peaked[tag]) if world == 1 else (3 if w.peaked[tag] else 0)   # bit 0 PEAK, bit 1 SPIKE (summed over ranks: any)
        if gated == 1 and (code & 1):
            p = 3                                          # a message with too many spikes switched the message rows to three passes
        if gated == 2 and (code & 1):
            p = 2                                          # ... and the one-pass gradient rows to two
        t = x.elapsed_time(y)
        d = by_passes.setdefault(p, {'launches': 0, 'rows': 0, 'ms': 0.0})
        d['launches'] += 1; d['rows'] += r; d['ms'] += t
        d = by_role.setdefault('%s rows, %d pass%s' % (role, p, '' if p == 1 else 'es'), {'launches': 0, 'rows': 0, 'ms': 0.0, 'p': p})
        d['launches'] += 1; d['rows'] += r; d['ms'] += t
        gemm_ms += t; gemm_rows += r; gemm_pass_rows += r * p
    n_gemm = len(eng.gemm_events)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = {}
    pk_path = os.path.join(REPO, 'MEASURED_PEAKS.json')
    if os.path.exists(pk_path):
        peaks = json.load(open(pk_path))
    peak_tf = float(peaks.get('bf16_tflops_sustained', 1400.0))
    which = 'measured (MEASURED_PEAKS.json bf16_tflops_sustained)' if peaks else 'fallback 1.4 PFLOP/s sustained (B200_PROFILING.md)'
    flops = 2.0 * gemm_rows * a.V * a.V
    ach = flops / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else 0.0
    traffic, traffic_note, key = None, None, None
    tr_path = os.path.join(REPO, 'profiles', a.traffic_file)
    if os.path.exists(tr_path) and a.V == 10000:
        tj = json.load(open(tr_path))
        key = next((kk for kk in (('one_pass_message_rows',) if 2 not in by_passes and 3 not in by_passes else ()) + ('two_pass_37_pairs', 'three_pass_37_pairs', 'three_pass_big') if kk in tj), None)
    if os.path.exists(tr_path) and a.V == 10000 and key:
        big = tj[key]
        traffic = big['dram_bytes_per_launch']
        traffic_note = ('dram__bytes_read+write of one %s launch of %d rows from the committed ncu --set full capture (%s): %.1fx its '
                        'algorithmic A + D + table bytes; %.0f %% of DRAM peak while the tensor pipe is %.0f %% active; launches of '
                        'this run average %d rows' % (key, big['rows_per_launch_padded'], big.get('source', 'profiles/'), big['ratio'],
                                                      big['dram_pct_of_peak'], big['tensor_pipe_active_pct'], gemm_rows // max(n_gemm, 1)))
    roofline = {'bound': 'tensor', 'kernel': 'gemm_split_f16_pair_kernel (K4, CTA pair, tcgen05.mma.cta_group::2)' if a.V > 2048 else 'gemm_split_f16_kernel (K4)', 'achieved': ach, 'peak': peak_tf, 'unit': 'TFLOP/s',
                'frac': ach / peak_tf, 'traffic': traffic, 'traffic_note': traffic_note, 'peak_source': which,
                'executed_tflops': ach * gemm_pass_rows / max(gemm_rows, 1), 'executed_frac': ach * gemm_pass_rows / max(gemm_rows, 1) / peak_tf,
                'by_passes': {str(p): {'launches': d['launches'], 'rows': d['rows'], 'ms': d['ms'],
                                       'algorithmic_tflops': 2.0 * d['rows'] * a.V * a.V / (d['ms'] / 1e3) / 1e12 if d['ms'] > 0 else 0.0,
                                       'executed_tflops': p * 2.0 * d['rows'] * a.V * a.V / (d['ms'] / 1e3) / 1e12 if d['ms'] > 0 else 0.0}
                              for p, d in sorted(by_passes.items())},
                'by_role': {k: {'launches': d['launches'], 'rows': d['rows'], 'ms': d['ms'], 'share_of_step': d['ms'] / ms_prof,
                                'algorithmic_tflops': 2.0 * d['rows'] * a.V * a.V / (d['ms'] / 1e3) / 1e12 if d['ms'] > 0 else 0.0,
                                'executed_tflops': d['p'] * 2.0 * d['rows'] * a.V * a.V / (d['ms'] / 1e3) / 1e12 if d['ms'] > 0 else 0.0}
                            for k, d in sorted(by_role.items())},
                'launches_timed': n_gemm, 'avg_launch_ms': gemm_ms / max(n_gemm, 1),
                'algorithmic_flops_per_launch': flops / max(n_gemm, 1), 'share_of_step': gemm_ms / ms_prof,
                'measured_in': 'a separate profiling pass of %d steps (CUDA-event pair around every launch, %.1f ms/step); `value` and '
                               '`e2e` are timed without those events' % (p_steps, ms_prof / p_steps),
                'note': 'algorithmic flops 2*rows*V*V counted once; message rows issue ONE fp16 MMA pass (hi*hi: the lo halves of the '
                        'message and of the table are dropped, the spikes of a message get both dropped terms back exactly '
                        '(csrc/spikes.cu) and every near-tied decision is re-scored from the full operands, csrc/rescore.cu), 2 with '
                        '--msg-passes 2 (hi*hi, hi*lo) or 3 (hi*hi, hi*lo, lo*hi) when a message has more spikes than slots or the '
                        'potentials span more than e^3; gradient rows 1 (hi*hi; V >= 4096 and potentials within e^3, else 2 or 3): '
                        '%.2f passes per row on average' % (gemm_pass_rows / max(gemm_rows, 1))}
    # HBM-bound kernels: algorithmic bytes (each input / output row counted once) over the CUDA-event time of every launch
    peak_gbs = float(peaks.get('hbm_gbs', 6500.0))
    hbm = {}
    for name, x, y, nbytes in eng.kernel_events:
        d = hbm.setdefault(name, {'launches': 0, 'ms': 0.0, 'bytes': 0.0})
        d['launches'] += 1; d['ms'] += x.elapsed_time(y); d['bytes'] += nbytes
    for name, d in hbm.items():
        gbs = d['bytes'] / (d['ms'] / 1e3) / 1e9 if d['ms'] > 0 else 0.0
        hbm[name] = {'bound': 'hbm', 'launches': d['launches'], 'achieved': gbs, 'peak': peak_gbs, 'unit': 'GB/s',
                     'frac': gbs / peak_gbs, 'algorithmic_bytes_per_launch': d['bytes'] / max(d['launches'], 1),
                     'avg_launch_ms': d['ms'] / max(d['launches'], 1), 'share_of_step': d['ms'] / ms_prof}
    cpu_baseline = None
    if not a.no_cpu_baseline and world == 1:
        try:
            cpu_baseline = cpu_baseline_subprocess(a)
        except Exception as e:                                   # still report a CPU number: the in-process threaded variant
            if a.config == 'c5':
                cpu_baseline = {'value': None, 'unit': UNIT, 'kind': 'port', 'sample': 'failed: %s' % str(e)[:200]}
            else:
                n = a.cpu_sample
                t_tab, t_sent, _ = cpu_run(a, n)
                per_sent = t_sent / n + t_tab / float(a.sentences)
                cpu_baseline = {'value': 1.0 / per_sent, 'unit': UNIT, 'cores': host_threads(), 'kind': 'port', 'variant': 'blas_threads',
                                'sample': '%d sentences of the workload (%.1f s) + one table build (%.1f s, amortised over %d '
                                          'sentences/step); oracle fast variant, float64, all BLAS threads; the process-pool '
                                          'variant failed: %s' % (n, t_sent, t_tab, a.sentences, str(e)[:200])}
    line = {'metric': metric_name(a), 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': a.steps, 'warmup': a.warmup,
            'ms_per_step': ms / a.steps, 'higher_is_better': True, 'scaling': scaling_name(a), 'vs_baseline': None,
            'dtype': 'f16 x f16 -> f32 (one tensor-core pass per GEMM row, fp32 accumulate; the hi+lo operand split serves the exact re-score, the spike compensation and the three-pass fallback; fp32 message products, f64 sums)', 'data': 'synthetic',
            'config': {'workload': workload_name(a), 'global_sentences_per_step': w.n_global,
                       'parallelism': 'dp%d (%s sharded, 16 x f64 all-reduce per step)' % (world, 'users' if a.config == 'c4' else 'sentences'),
                       'l2': 'inputs larger than L2: table planes %.1f GB, message blocks > 10 GB per micro-batch' % (eng.planes.numel() * 2 / 1e9),
                       'micro_batches_per_step': len(w.parts) if w.parts is not None else len(w.batches),
                       'k4_rows_per_sliced_launch': eng.gemm_slice_rows},
            'clocks': clocks, 'e2e': e2e, 'gpu_launches': launches, 'roofline': roofline, 'hbm_kernels': hbm,
            'host': {'plan_compile_s_per_step': plan_s_per_step, 'plan_threads': int(os.environ.get('MLBP_PLAN_THREADS', '0')),
                     'schedules_compiled_ahead': eng.plan_prefetched,   # next step's first micro-batch, during the wait for the all-reduce
                     'schedule_templates': {'hits_in_timed_steps': tm1[0] - tm0[0], 'compiled_in_timed_steps': tm1[1] - tm0[1],
                                            'note': 'graphs whose schedule was relocated from a cached template vs compiled (csrc/plan.cpp); roots are redrawn every step'}},
            'message_rows': {'passes': pass_stats['msg_passes'], 'reduced_pass_enabled': pass_stats['msg_two_pass'], 'ranks_switched_to_three_passes_per_step': peaked_value,
                             'ranks_switched_all_steps_incl_warmup_e2e_profiling': w.all_peaked, 'max_message_prob_last_step': pass_stats['max_message_prob'],
                             'flag_code': 'bit 0 = a row had more spikes than slots (message rows ran three passes, gradient rows two), bit 1 = a spike was seen and compensated',
                             'spiky_rows_last_batch': pass_stats['spiky_rows_last_batch'], 'theta_after_each_step': w.thetas,
                             'rescore': {k: pass_stats[k] for k in ('rescored', 'skipped_mass_tie', 'skipped_degenerate', 'top1_changed', 'rank_changed')},
                             'rescore_note': 'counters of the LAST step of the profiling pass (reset per theta)'},
            'cpu_baseline': cpu_baseline}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    a = parse()
    if a.impl == 'reference':
        reference_arm(a)
    else:
        ours(a)


if __name__ == '__main__':
    main()
