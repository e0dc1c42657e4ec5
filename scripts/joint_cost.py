"""What the joint log-likelihood (Engine.run want_joint, K9 mlbp_joint_logp) costs at inference:

  sentences/s of inference (want_grad=False, marginals) with and without want_joint, alternated in one process, at V = 10 000
  (1 024 sentences, k = 20 predicted tokens) and at V = 50 000 (the C5 sizes of scripts/predict_throughput.py: 64 sentences);
  K9's own CUDA-event time in a separate profiled pass (Engine.profile_kernels), with its algorithmic bytes (16 V per pairwise
  factor: the two variable->factor rows as fp16 hi + lo and the two factor->variable rows as fp32) over that time against the
  7.7 TB/s HBM3e data-sheet figure of one B200.

With want_joint the gradient-stage GEMM rows run as well (they produce the normalisers Z); the sentences/s difference includes
them.  The card's name and power limit are read in the same process and written with the numbers.

    python scripts/joint_cost.py [--out profiles/joint_cost.jsonl] [--cases 10000 50000] [--reps 3]
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

CASES = {10000: dict(V=10000, Vd=2000, n=1024, k=20), 50000: dict(V=50000, Vd=2000, n=64, k=20)}
THETA_EE, THETA_ED = [0.8, 0.5, -0.3], [1.0, -0.6, 0.5, 0.3, 0.4, -0.2]
HBM_BYTES_PER_S = 7.7e12


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return {'card': torch.cuda.get_device_name(), 'nvidia_smi': q.stdout.strip().split('\n')}


def one_case(c, reps):
    model = synth.make_model_large(c['V'], c['Vd'], seed=1234)
    sents = [synth.sentence_to_arrays(synth.make_sentence(model, 'p' * c['k'], seed=7000 + i, n_history=3)) for i in range(c['n'])]
    corpus = Corpus(sents)
    roots = corpus.roots_from_positions(synth.draw_roots(sents, 3, seed=5))
    eng = Engine(model)
    eng.set_theta(THETA_EE, THETA_ED, with_grad=True)
    parts = eng.prepare(corpus, 3, want_grad=True)

    def run(joint):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = eng.run_prepared(parts, roots, 3, want_grad=False, want_marg=True, want_joint=joint)
        torch.cuda.synchronize()
        return time.perf_counter() - t0, res

    for joint in (False, True):                                   # warm-up of every shape
        run(joint)
    times = {False: [], True: []}
    for _ in range(reps):
        for joint in (False, True):
            times[joint].append(run(joint)[0])
    _, res = run(True)
    # K9 alone, in a profiled pass of its own
    eng.profile_kernels = True
    eng.kernel_events = []
    run(True)
    torch.cuda.synchronize()
    k9 = [(e0.elapsed_time(e1) * 1e-3, b) for name, e0, e1, b in eng.kernel_events if name == 'K9 joint_logp']
    eng.profile_kernels = False
    k9_s, k9_bytes = sum(t for t, _ in k9), sum(b for _, b in k9)
    sps = lambda ts: c['n'] / min(ts)
    return {'V': c['V'], 'Vd': c['Vd'], 'sentences': c['n'], 'k': c['k'], 'pairs': corpus.n_pairs, 'reps': reps,
            'infer_s': times[False], 'infer_joint_s': times[True], 'sent_per_s': sps(times[False]),
            'sent_per_s_joint': sps(times[True]), 'k9_launches': len(k9), 'k9_s': k9_s, 'k9_bytes': k9_bytes,
            'k9_bytes_per_s': k9_bytes / k9_s if k9_s > 0 else None,
            'k9_share_of_7p7TBps': (k9_bytes / k9_s) / HBM_BYTES_PER_S if k9_s > 0 else None,
            'mean_logp_joint': float(res[4].mean().item()), 'mean_logp_marginal_sum': float(res[1].mean().item())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    ap.add_argument('--cases', type=int, nargs='+', default=[10000, 50000])
    ap.add_argument('--reps', type=int, default=3)
    a = ap.parse_args()
    assert torch.cuda.is_available(), 'the measurement needs the GPU'
    build.build()
    info = card()
    for v in a.cases:
        rec = dict(one_case(CASES[v], a.reps), **info)
        line = json.dumps(rec)
        print(line, flush=True)
        if a.out:
            with open(a.out, 'a') as f:
                f.write(line + '\n')


if __name__ == '__main__':
    main()
