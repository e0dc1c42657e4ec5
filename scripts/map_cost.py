"""What max-product decoding (Engine.run max_product: K10 mlbp_factor_to_var_maxprod, K11 mlbp_assignment_score) costs:

  1. K10 alone: 16 384 rows x V = 10 000 for each of the four message tables, CUDA events over --launches launches after a
     warm-up; multiply-max/s against the issue bound of the SIMT pipes, 148 SMs x 128 lanes x the SM clock (one FMUL2 + one
     FMNMX3 per two multiply-max);
  2. end to end at V = 10 000, 1 024 sentences, k = 20, 3 sweeps: decode sentences/s next to sum-product inference
     (want_grad=False) in the same process, the two alternated;
  3. the share of the decode step spent in K10, from a separate profiled pass (Engine.profile_kernels).

The card's name, power limit and SM clocks are read with nvidia-smi in the same process and written with the numbers.

    python scripts/map_cost.py [--out profiles/r6a_map_cost.jsonl] [--reps 3] [--launches 20]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from macaronicusermodeling_b200 import build, synth  # noqa: E402
from macaronicusermodeling_b200.engine import Corpus, Engine  # noqa: E402

THETA_EE, THETA_ED = [0.8, 0.5, -0.3], [1.0, -0.6, 0.5, 0.3, 0.4, -0.2]
V, VD, N_SENT, K, ROWS = 10000, 2000, 1024, 20, 16384
LANES = 128                                                     # fp32 SIMT lanes of one SM


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.sm,clocks.max.sm', '--format=csv,noheader,nounits'],
                       capture_output=True, text=True)
    name, power, sm, sm_max = [x.strip() for x in q.stdout.strip().split('\n')[0].split(',')]
    return {'card': name, 'power_limit_w': float(power), 'sm_clock_mhz_at_query': float(sm), 'sm_clock_max_mhz': float(sm_max),
            'sms': torch.cuda.get_device_properties(0).multi_processor_count}


def k10_alone(eng, launches, info):
    """K10 on ROWS random message rows for each table, CUDA events around `launches` launches"""
    rng = np.random.default_rng(3)
    msg = rng.random((ROWS, V)).astype(np.float32)
    msg *= np.float32(2.0 ** 14) / msg.sum(axis=1, keepdims=True)
    A = torch.zeros((2, ROWS, eng.ld), dtype=torch.float16, device='cuda')
    A[0, :, :V] = torch.from_numpy(msg).cuda().half()
    A[1, :, :V] = (torch.from_numpy(msg).cuda() - A[0, :, :V].float()).half()
    D = torch.empty((ROWS, eng.ld), dtype=torch.float32, device='cuda')
    out = {}
    for t in range(4):
        for _ in range(2):
            eng.maxprod_rows(A[0], A[1], ROWS, 0, ROWS, t, D, 0)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(launches):
            eng.maxprod_rows(A[0], A[1], ROWS, 0, ROWS, t, D, 0)
        e1.record()
        torch.cuda.synchronize()
        s = e0.elapsed_time(e1) * 1e-3 / launches
        rate = ROWS * float(V) * V / s
        bound = info['sms'] * LANES * info['sm_clock_max_mhz'] * 1e6
        out['table%d' % t] = {'launch_s': s, 'multiply_max_per_s': rate, 'issue_bound_per_s': bound, 'share_of_bound': rate / bound}
    return out


def end_to_end(eng, model, reps):
    sents = [synth.sentence_to_arrays(synth.make_sentence(model, 'p' * K, seed=7000 + i, n_history=3)) for i in range(N_SENT)]
    corpus = Corpus(sents)
    roots = corpus.roots_from_positions(synth.draw_roots(sents, 3, seed=5))
    parts = eng.prepare(corpus, 3, want_grad=False)

    def run(mp):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        eng.run_prepared(parts, roots, 3, want_grad=False, want_marg=True, max_product=mp)
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    for mp in (False, True):                                      # warm-up of every shape
        run(mp)
    times = {False: [], True: []}
    for _ in range(reps):
        for mp in (False, True):
            times[mp].append(run(mp))
    eng.profile_kernels = True                                    # K10's share, in a pass of its own
    eng.kernel_events = []
    step = run(True)
    torch.cuda.synchronize()
    k10 = [e0.elapsed_time(e1) * 1e-3 for name, e0, e1, _ in eng.kernel_events if name == 'K10 maxprod']
    eng.profile_kernels = False
    rows = sum(int(p[2].n_vars) for p in parts)
    return {'V': V, 'sentences': N_SENT, 'k': K, 'sweeps': 3, 'reps': reps, 'infer_s': times[False], 'decode_s': times[True],
            'infer_sent_per_s': N_SENT / min(times[False]), 'decode_sent_per_s': N_SENT / min(times[True]),
            'profiled_decode_s': step, 'k10_launches': len(k10), 'k10_s': sum(k10), 'k10_share_of_profiled_decode': sum(k10) / step,
            'variables': rows}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join('profiles', 'r6a_map_cost.jsonl'))
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--launches', type=int, default=20)
    a = ap.parse_args()
    assert torch.cuda.is_available(), 'the measurement needs the GPU'
    build.build()
    info = card()
    model = synth.make_model_large(V, VD, seed=1234)
    eng = Engine(model)
    eng.set_theta(THETA_EE, THETA_ED, with_grad=False)
    rec = dict(info, k10_alone=k10_alone(eng, a.launches, info), end_to_end=end_to_end(eng, model, a.reps))
    line = json.dumps(rec)
    print(line, flush=True)
    with open(a.out, 'a') as f:
        f.write(line + '\n')


if __name__ == '__main__':
    main()
