"""GPU tier: trainer semantics (train.py:357-416, :617-638) and the bench entry points."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from macaronicusermodeling_b200 import build, synth
from macaronicusermodeling_b200.engine import Corpus, Engine
from macaronicusermodeling_b200.trainer import Trainer, batch_sgd_many

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), 'golden')
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope='module', autouse=True)
def _built():
    build.build()


def test_sgd_trajectory_matches_reference():
    """minibatch = 1 sentence on one GPU reproduces train.py's per-sentence SGD trajectory (2 epochs)"""
    z = np.load(os.path.join(GOLDEN, 'sgd_trajectory.npz'), allow_pickle=False)
    model = {'V': z['pmi'].shape[0], 'Vd': z['ed'].shape[1], 'pmi': z['pmi'], 'pmi_w1': z['pmi_w1'], 'ed': z['ed'],
             'ped': z['ped']}
    sents = [synth.sentence_to_arrays(str(s)) for s in z['sentences']]
    roots = z['roots'].tolist()
    eng = Engine(model)
    tr = Trainer(eng, reg_param=0.2, N=len(sents), sweeps=3)
    traj, logps = [], []
    for epoch in range(2):
        lr = tr.lr(epoch)
        for si, s in enumerate(sents):
            c = Corpus([s])
            red = tr.step(c, c.roots_from_positions([roots[epoch][si]]), lr)
            h = tr.apply(red, lr)
            logps.append(h[9])
            traj.append(np.concatenate([tr.theta_ee, tr.theta_ed]))
    np.testing.assert_allclose(np.array(traj), z['traj'], rtol=1e-4, atol=2e-7)
    np.testing.assert_allclose(np.array(logps), z['logps'], rtol=1e-5)


def test_batch_sgd_many_returns_reference_result_lists():
    z = np.load(os.path.join(GOLDEN, 'sgd_trajectory.npz'), allow_pickle=False)
    model = {'V': z['pmi'].shape[0], 'Vd': z['ed'].shape[1], 'pmi': z['pmi'], 'pmi_w1': z['pmi_w1'], 'ed': z['ed'],
             'ped': z['ped']}
    sents = [synth.sentence_to_arrays(str(s)) for s in z['sentences']]
    roots = z['roots'].tolist()[0]
    eng = Engine(model)
    res = batch_sgd_many(eng, sents, np.zeros(3), np.zeros(6), 0.1, roots, reg_param=0.2, N=len(sents))
    # sentence 0 at theta = 0 is the first step of the reference trajectory
    np.testing.assert_allclose(np.concatenate([res[0][2][0], res[0][3][0]]), z['traj'][0], rtol=1e-4, atol=2e-7)
    np.testing.assert_allclose(res[0][1], z['logps'][0], rtol=1e-5)
    assert res[0][2].shape == (1, 3) and res[0][3].shape == (1, 6)


def test_bench_line_small(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(REPO, 'bench.py'), '--steps', '1', '--warmup', '1', '--sentences',
                          '16', '--V', '1024', '--Vd', '128', '--k', '6', '--cpu-sample', '2', '--dump-outputs', str(tmp_path)],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for key in ('metric', 'value', 'unit', 'n_gpus', 'ms_per_step', 'clocks', 'e2e', 'gpu_launches', 'roofline', 'cpu_baseline'):
        assert key in line
    assert line['gpu_launches'] > 0 and line['value'] > 0 and line['e2e']['value'] > 0
    red, theta = np.load(tmp_path / 'reduced.npy'), np.load(tmp_path / 'theta.npy')
    assert red.shape == (16,) and red[14] == 16 and np.isfinite(red).all()
    np.testing.assert_allclose(theta, line['message_rows']['theta_after_each_step'][1], atol=6e-4)   # the second step: the timed one


def test_adapt_trainer_batched_domains_vs_oracle():
    """BASELINE config C4 semantics (users sharded, per-user theta): AdaptTrainer with several sentences per user batch --
    every user's sentences see that user's theta; the base theta receives the sum over all users"""
    from macaronicusermodeling_b200.trainer import AdaptTrainer
    from oracle import lbp_oracle as orc
    model = synth.make_model(96, 20, seed=8)
    users = ['u0', 'u1', 'u2']
    sents = {u: synth.make_corpus(model, 3, k=4, g=1, seed=20 + i) for i, u in enumerate(users)}
    roots = {u: synth.draw_roots(sents[u], 3, seed=30 + i) for i, u in enumerate(users)}
    tr = AdaptTrainer(Engine(model), users, reg_param=0.2, ua_scale=0.5, N=9)
    rng = np.random.default_rng(0)
    for u in users:
        tr.domain2theta[u] = (rng.normal(size=3) * 0.3, rng.normal(size=6) * 0.3)
    before = {u: (tr.domain2theta[u][0].copy(), tr.domain2theta[u][1].copy()) for u in users}
    batches = []
    for u in users:
        c = Corpus(sents[u])
        batches.append((u, c, c.roots_from_positions(roots[u])))
    lr = 0.05
    red = tr.step_domains(batches, lr).cpu().numpy()
    tot = np.zeros(9)
    reg = 0.2 / 9
    for u in users:
        te, td = before[u]
        tb = orc.Tables(model, te, td)
        g = np.zeros(9)
        for s, r in zip(sents[u], roots[u]):
            o = orc.run_fast(tb, s, r, 3)
            g += np.concatenate([o['g_ee_unreg'][0], o['g_ed_unreg'][0]])
        tot += g
        np.testing.assert_allclose(tr.domain2theta[u][0], te + lr * (g[:3] - 3 * reg * 0.5 * te), rtol=1e-4, atol=1e-7)
        np.testing.assert_allclose(tr.domain2theta[u][1], td + lr * (g[3:] - 3 * reg * 0.5 * td), rtol=1e-4, atol=1e-7)
    np.testing.assert_allclose(red[:9], tot, rtol=1e-4, atol=2e-6)
    assert red[14] == 9
