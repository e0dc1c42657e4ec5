"""What the pseudo-likelihood (Engine.pseudo_likelihood: K1 + K13 mlbp_pseudo_likelihood + the sums) costs against loopy BP:

  a. K13 alone at C3 size (4 096 sentences, V = 10 000, k = 20, with the gradient): CUDA events around each launch after a
     warm-up, over 5 calls; algorithmic bytes/s (from shapes: the U row and one fp16 plane pair per factor for the product, a
     second table row and one or two gradient rows per factor and given token, the ed / ped rows) against 7.7 TB/s;
  b. Trainer.step sentences/s on the same 4 096-sentence batch with objective='pl' and 'lbp', alternated, each warmed up;
  c. (information only) from theta = 0, the same number of SGD steps with each objective on one 1 024-sentence batch (lr =
     0.05 / variables, no minibatch shuffling), then BP
     prediction (3 sweeps) on a held-out batch with each theta: P@0 and the mean log-probability of the labels.

The card's name, power limit and SM clocks are read with nvidia-smi in the same process and written with the numbers.

    python scripts/pl_cost.py [--out profiles/r8a_pl_cost.jsonl] [--steps 20]
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
from macaronicusermodeling_b200.trainer import Trainer  # noqa: E402
from map_cost import card  # noqa: E402

V, VD, K, N_SENT = 10000, 2000, 20, 4096
HBM = 7.7e12
THETA = ([0.9, 0.4, -0.1], [1.1, -0.5, 0.5, 0.3, 0.4, -0.2])


def corpus_of(model, n, seed):
    sents = [synth.sentence_to_arrays(synth.make_sentence(model, 'p' * K, seed=seed + i, n_history=3)) for i in range(n)]
    return sents, Corpus(sents)


def k13_alone(eng, c, reps=5):
    eng.set_theta(*THETA, with_grad=True)
    eng.pseudo_likelihood(c)                                       # warm-up of the shapes
    torch.cuda.synchronize()
    eng.profile_kernels, eng.kernel_events = True, []
    t0 = time.perf_counter()
    for _ in range(reps):
        eng.pseudo_likelihood(c)
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) / reps
    ev = [(e0.elapsed_time(e1) * 1e-3, nb) for name, e0, e1, nb in eng.kernel_events if name == 'K13 pseudo_likelihood']
    eng.profile_kernels = False
    s, nbytes = sum(x[0] for x in ev) / reps, sum(x[1] for x in ev) / reps
    return {'sentences': c.n_sent, 'k': K, 'V': V, 'launches_per_call': len(ev) // reps, 'k13_s': s, 'pl_call_s': wall,
            'variables_per_s': c.n_vars / s, 'algorithmic_bytes': nbytes, 'bytes_per_s': nbytes / s,
            'share_of_7_7_TBps': nbytes / s / HBM}


def step_rate(eng, sents, c, rounds=3):
    roots = c.roots_from_positions(synth.draw_roots(sents, 3, seed=5))
    trs = {obj: Trainer(eng, reg_param=0.2, N=len(sents), objective=obj) for obj in ('pl', 'lbp')}
    for tr in trs.values():
        tr.theta_ee, tr.theta_ed = np.array(THETA[0]), np.array(THETA[1])
        tr.step(c, roots, 0.0)                                     # warm-up
    torch.cuda.synchronize()
    times = {'pl': [], 'lbp': []}
    for _ in range(rounds):                                        # alternated
        for obj, tr in trs.items():
            t0 = time.perf_counter()
            tr.step(c, roots, 0.0).cpu()
            times[obj].append(time.perf_counter() - t0)
    out = {'sentences': len(sents)}
    for obj, t in times.items():
        out[obj + '_step_s'] = sorted(t)
        out[obj + '_sentences_per_s'] = len(sents) / float(np.median(t))
    out['speedup_pl_over_lbp'] = out['pl_sentences_per_s'] / out['lbp_sentences_per_s']
    return out


def fit_and_predict(eng, model, steps):
    sents, c = corpus_of(model, 1024, 11000)
    lr = 0.05 / c.n_vars                                           # a step of 0.05 times the mean gradient of a variable
    held, ch = corpus_of(model, 512, 13000)
    hroots = ch.roots_from_positions(synth.draw_roots(held, 3, seed=9))
    out = {'train_sentences': len(sents), 'held_out_sentences': len(held), 'steps': steps, 'lr': lr}
    for obj in ('pl', 'lbp'):
        tr = Trainer(eng, reg_param=0.2, N=len(sents), objective=obj)
        rng = np.random.default_rng(3)
        for _ in range(steps):
            roots = c.roots_from_positions(synth.draw_roots(sents, 3, seed=int(rng.integers(1 << 30))))
            tr.apply(tr.step(c, None if obj == 'pl' else roots, lr), lr)
        eng.set_theta(tr.theta_ee, tr.theta_ed, with_grad=False)
        r = eng.run(ch, hroots, 3, want_grad=False)
        p0, _, _, tot = r.precision_counts()
        out[obj] = {'theta_ee': tr.theta_ee.tolist(), 'theta_ed': tr.theta_ed.tolist(), 'bp_p_at_0': p0 / float(tot),
                    'bp_mean_logp_var': float(r.logp_var.mean().item())}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join('profiles', 'r8a_pl_cost.jsonl'))
    ap.add_argument('--steps', type=int, default=20)
    a = ap.parse_args()
    assert torch.cuda.is_available(), 'the measurement needs the GPU'
    build.build()
    info = card()
    model = synth.make_model_large(V, VD, seed=1234)
    eng = Engine(model)
    sents, c = corpus_of(model, N_SENT, 7000)
    rec = dict(info, k13_alone=k13_alone(eng, c), trainer_step=step_rate(eng, sents, c),
               fit_then_bp_prediction=fit_and_predict(eng, model, a.steps))
    line = json.dumps(rec)
    print(line, flush=True)
    os.makedirs(os.path.dirname(a.out) or '.', exist_ok=True)
    with open(a.out, 'a') as f:
        f.write(line + '\n')


if __name__ == '__main__':
    main()
