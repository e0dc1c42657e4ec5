"""What the Gibbs sampler (Engine.sample: K12 mlbp_gibbs_sample + its reduce) costs, and what it shows about loopy BP:

  1. K12 alone at V = 10 000, k = 20, 4 chains, 100 burn-in + 100 kept sweeps, for 1 024 sentences and for the command line's
     64-sentence unit: CUDA events around the launch after a warm-up; updates/s and algorithmic bytes/s (from shapes: a U row
     and two fp16 plane rows per neighbour per update, the 8-byte read-modify-write of the Rao-Blackwell row in kept sweeps)
     against 7.7 TB/s;
  2. the payoff: V = 10 000, k = 20, 256 sentences, the flat and the trained theta of tests/test_gpu_engine.py, 16 chains x
     1 000 kept sweeps: |b_BP(label) - p_hat(label)| (mean, max) of 3-sweep loopy BP against the Monte Carlo estimate, the mean
     across-chain standard error, and the share of variables where the difference exceeds 5 SE.

The card's name, power limit and SM clocks are read with nvidia-smi in the same process and written with the numbers.

    python scripts/gibbs_cost.py [--out profiles/r7a_gibbs_cost.jsonl] [--keep 1000]
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from macaronicusermodeling_b200 import build, synth  # noqa: E402
from macaronicusermodeling_b200.engine import Corpus, Engine  # noqa: E402
from map_cost import card  # noqa: E402

V, VD, K = 10000, 2000, 20
HBM = 7.7e12
REGIMES = {'flat': ([0.9, 0.4, -0.1], [1.1, -0.5, 0.5, 0.3, 0.4, -0.2]),
           'trained': ([-0.003, 0.049, -0.3], [0.101, -0.047, 7.534, 0.3, 0.4, -0.2])}


def corpus_of(model, n, seed):
    sents = [synth.sentence_to_arrays(synth.make_sentence(model, 'p' * K, seed=seed + i, n_history=3)) for i in range(n)]
    return sents, Corpus(sents)


def k12_alone(eng, model, n_sent, chains=4, burn_in=100, n_keep=100):
    _, c = corpus_of(model, n_sent, 7000)
    eng.sample(c, chains=chains, burn_in=1, n_keep=1)            # warm-up of the shapes
    torch.cuda.synchronize()
    eng.profile_kernels, eng.kernel_events = True, []
    t0 = time.perf_counter()
    eng.sample(c, chains=chains, burn_in=burn_in, n_keep=n_keep)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    ev = [(e0.elapsed_time(e1) * 1e-3, nb) for name, e0, e1, nb in eng.kernel_events if name == 'K12 gibbs_sample']
    eng.profile_kernels = False
    s, nbytes = sum(x[0] for x in ev), sum(x[1] for x in ev)
    updates = float(c.n_vars) * chains * (1 + burn_in + n_keep)
    return {'sentences': n_sent, 'k': K, 'chains': chains, 'burn_in': burn_in, 'n_keep': n_keep, 'launches': len(ev), 'k12_s': s,
            'sample_call_s': wall, 'updates_per_s': updates / s, 'algorithmic_bytes': nbytes, 'bytes_per_s': nbytes / s,
            'share_of_7_7_TBps': nbytes / s / HBM}


def payoff(eng, model, regime, n_keep, n_sent=256, chains=16):
    te, td = REGIMES[regime]
    eng.set_theta(te, td, with_grad=False)
    sents, c = corpus_of(model, n_sent, 9000)
    roots = c.roots_from_positions(synth.draw_roots(sents, 3, seed=5))
    b = eng.run(c, roots, 3, want_grad=False, want_beliefs=True)
    bl = b.beliefs[torch.arange(c.n_vars, device='cuda'), torch.from_numpy(c.var_label).long().cuda()].double().cpu().numpy()
    t0 = time.perf_counter()
    r = eng.sample(c, chains=chains, burn_in=100, n_keep=n_keep, seed=1)
    torch.cuda.synchronize()
    s = time.perf_counter() - t0
    p = r.label_prob.cpu().numpy()
    se = p.std(axis=1, ddof=1) / np.sqrt(chains)
    d = np.abs(bl - p.mean(axis=1))
    return {'regime': regime, 'theta_ee': te, 'theta_ed': td, 'sentences': n_sent, 'k': K, 'chains': chains, 'burn_in': 100,
            'n_keep': n_keep, 'sample_s': s, 'mean_abs_diff': float(d.mean()), 'max_abs_diff': float(d.max()),
            'mean_se': float(se.mean()), 'max_se': float(se.max()), 'share_diff_over_5se': float((d > 5 * se).mean()),
            'mean_label_prob_bp': float(bl.mean()), 'mean_label_prob_gibbs': float(p.mean())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join('profiles', 'r7a_gibbs_cost.jsonl'))
    ap.add_argument('--keep', type=int, default=1000)
    a = ap.parse_args()
    assert torch.cuda.is_available(), 'the measurement needs the GPU'
    build.build()
    info = card()
    model = synth.make_model_large(V, VD, seed=1234)
    eng = Engine(model)
    eng.set_theta(*REGIMES['flat'], with_grad=False)
    rec = dict(info, k12_alone=[k12_alone(eng, model, n) for n in (1024, 64)],
               payoff=[payoff(eng, model, reg, a.keep) for reg in ('flat', 'trained')])
    line = json.dumps(rec)
    print(line, flush=True)
    with open(a.out, 'a') as f:
        f.write(line + '\n')


if __name__ == '__main__':
    main()
