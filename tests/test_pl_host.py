"""CPU tier of the pseudo-likelihood (K13, Engine.pseudo_likelihood, Trainer(objective='pl'), train_cli --objective pl /
--pseudo_likelihood): the float64 model-level reference (tests/pl_oracle.py) against brute-force conditionals of the enumerated
joint, its gradient against central differences, the unbiasedness of the PL score at the true theta (and its failure at another
theta), and the engine, trainer and command line on the emulated kernels (tests/fake_pl_kernels.py)."""
import itertools
import os
import sys

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))

import pl_oracle  # noqa: E402
from fake_pl_kernels import PLKernels  # noqa: E402
from macaronicusermodeling_b200 import build, synth  # noqa: E402
from macaronicusermodeling_b200.engine import Corpus, Engine  # noqa: E402
from map_checks import log_potentials  # noqa: E402

FLAT = ([0.3, -0.2, 0.1], [0.8, -0.5, 0.6, 0.4, 0.3, -0.2])
PEAKED = ([2.0, 1.2, -0.3], [2.0, -1.0, 0.6, 0.4, 0.3, -0.2])
BIAS = (2, 8)


@pytest.fixture(scope='module', autouse=True)
def _built():
    build.build()


def _setup(V, layouts, seed):
    model = synth.make_model(V, 5, seed=seed, dtype=np.float32)
    sents = [synth.sentence_to_arrays(synth.make_sentence(model, l, seed=seed * 10 + i, n_history=2)) for i, l in enumerate(layouts)]
    return model, sents


def _joint_log(model, sent, te, td):
    """log-potential L [V]*k of every assignment of the sentence's predicted tokens (predicted-position order)"""
    var_ids, unary, pair = log_potentials(model, sent, te, td)
    k, V = len(var_ids), model['pmi'].shape[0]
    L = np.zeros((V,) * k)
    for i, v in enumerate(var_ids):
        L = L + unary[v].reshape([V if j == i else 1 for j in range(k)])
    for (a, b), P in pair.items():
        ia, ib = var_ids.index(a), var_ids.index(b)
        L = L + (P if ia < ib else P.T).reshape([V if j in (ia, ib) else 1 for j in range(k)])
    return L


@pytest.mark.parametrize('layouts, V', [(['pp', 'pgp'], 9), (['ppp', 'pgpp'], 7), (['prp', 'pppr'], 5)])
@pytest.mark.parametrize('theta', [FLAT, PEAKED], ids=['flat', 'peaked'])
def test_model_reference_against_brute_force_conditionals(layouts, V, theta):
    model, sents = _setup(V, layouts, seed=V)
    c = Corpus(sents)
    lp, _, probs = pl_oracle.model_reference(c, model, *theta)
    for s, sent in enumerate(sents):
        L = _joint_log(model, sent, *theta)
        lo, hi = int(c.var_off[s]), int(c.var_off[s + 1])
        y = tuple(int(v) for v in c.var_label[lo:hi])
        for i in range(hi - lo):
            row = np.array([L[y[:i] + (x,) + y[i + 1:]] for x in range(V)])
            p = np.exp(row - row.max())
            p /= p.sum()
            np.testing.assert_allclose(probs[lo + i], p, rtol=1e-10, atol=1e-14)
            assert abs(lp[lo + i] - np.log(p[y[i]])) < 1e-10


def _pl(c, model, te, td):
    return pl_oracle.model_reference(c, model, te, td)[0].sum()


@pytest.mark.parametrize('theta', [FLAT, PEAKED], ids=['flat', 'peaked'])
def test_model_gradient_against_central_differences(theta):
    model, sents = _setup(11, ['ppgp', 'pprpp'], seed=4)
    c = Corpus(sents)
    te, td = np.array(theta[0]), np.array(theta[1])
    g = pl_oracle.model_reference(c, model, te, td)[1].sum(axis=0)
    h = 1e-5
    num = []
    for j in range(9):
        d = np.zeros(9)
        d[j] = h
        num.append((_pl(c, model, te + d[:3], td + d[3:]) - _pl(c, model, te - d[:3], td - d[3:])) / (2 * h))
    np.testing.assert_allclose(g, num, rtol=1e-7, atol=1e-8)
    assert g[2] == 0.0 and g[8] == 0.0


def _score_z(model, sent, theta_draw, theta_eval, n=20000, seed=0):
    """|mean PL gradient| / SE over n labels drawn exactly from the enumerated joint at theta_draw, the gradient at theta_eval"""
    L = _joint_log(model, sent, *theta_draw)
    p = np.exp(L - L.max()).ravel()
    p /= p.sum()
    c = Corpus([sent])
    V = model['pmi'].shape[0]
    k = c.n_vars
    G = np.zeros((p.size, 9))
    for idx, y in enumerate(itertools.product(range(V), repeat=k)):
        c.var_label = np.asarray(y, dtype=np.int32)
        G[idx] = pl_oracle.model_reference(c, model, *theta_eval)[1].sum(axis=0)
    cnt = np.random.default_rng(seed).multinomial(n, p)
    mean = cnt.dot(G) / n
    var = cnt.dot((G - mean) ** 2) / (n - 1)
    se = np.sqrt(var / n)
    live = [j for j in range(9) if j not in BIAS and se[j] > 0]
    return np.abs(mean[live]) / se[live]


def test_pl_score_is_unbiased_at_the_true_theta_and_not_elsewhere():
    model, sents = _setup(6, ['pgpr'], seed=8)
    sent = sents[0]
    z = _score_z(model, sent, FLAT, FLAT)
    assert (z < 5).all(), z
    shifted = (np.array(FLAT[0]) + [0.6, 0.4, 0.0], np.array(FLAT[1]) + [0.5, -0.5, 0.0, 0.0, 0.0, 0.0])
    assert (_score_z(model, sent, FLAT, shifted) > 5).any()


# ---------------------------------------------------------------------------------------------------- engine
def _eng(model, **kw):
    eng = Engine(model, kernels=PLKernels(), **kw)
    eng.set_theta(FLAT[0], FLAT[1], with_grad=True)
    return eng


def _outs(r):
    return [x.numpy() for x in (r.grad, r.logp, r.logp_var, r.top1, r.rank, r.beliefs)]


def test_engine_against_the_model_reference_and_batch_order_microbatch_invariance():
    model = synth.make_model(40, 9, seed=3, dtype=np.float32)
    sents = synth.make_corpus(model, 5, k=3, g=1, seed=2) + synth.make_corpus(model, 3, k=5, g=2, seed=7)
    c = Corpus(sents)
    eng = _eng(model)
    r = eng.pseudo_likelihood(c, want_beliefs=True)
    a = _outs(r)
    lp, g, probs = pl_oracle.model_reference(c, model, *FLAT)
    np.testing.assert_allclose(a[2], lp, atol=1e-5)
    gs = np.array([g[c.var_off[s]:c.var_off[s + 1]].sum(axis=0) for s in range(c.n_sent)])
    np.testing.assert_allclose(a[0], gs, rtol=1e-4, atol=2e-6)
    np.testing.assert_allclose(a[5][:, :40], probs, atol=1e-6)
    assert (a[0][:, BIAS] == 0).all()
    np.testing.assert_allclose(a[1], [lp[c.var_off[s]:c.var_off[s + 1]].sum() for s in range(c.n_sent)], atol=1e-4)
    order = list(np.random.default_rng(1).permutation(len(sents)))
    co = Corpus([sents[i] for i in order])
    b = _outs(eng.pseudo_likelihood(co, want_beliefs=True))
    for pos, s in enumerate(order):
        np.testing.assert_array_equal(b[0][pos], a[0][s])
        for j in (2, 3, 4, 5):
            np.testing.assert_array_equal(b[j][co.var_off[pos]:co.var_off[pos + 1]], a[j][c.var_off[s]:c.var_off[s + 1]])
    small = _eng(model, workspace_bytes=4 * eng.ld * 4 * 2)                # 4 variables per micro-batch
    rs = small.pseudo_likelihood(c, want_beliefs=True)
    assert rs.stats['micro_batches'] > 2
    for x, y in zip(a, _outs(rs)):
        np.testing.assert_array_equal(x, y)
    top = eng.pseudo_likelihood(c, want_grad=False, want_topk=5)
    assert top.grad is None and top.beliefs is None
    np.testing.assert_array_equal(top.topk[0].numpy()[:, 0], a[3])


def test_sum_product_outputs_are_bit_identical_around_a_pl_call():
    model = synth.make_model(64, 9, seed=9, dtype=np.float32)
    sents = synth.make_corpus(model, 4, k=4, g=1, seed=3)
    corpus = Corpus(sents)
    roots = corpus.roots_from_positions(synth.draw_roots(sents, 3, seed=4))
    eng = _eng(model)
    kw = dict(want_grad=True, want_marg=True, want_beliefs=True)
    a = eng.run(corpus, roots, 3, **kw)
    eng.pseudo_likelihood(corpus, want_beliefs=True)
    b = eng.run(corpus, roots, 3, **kw)
    for name in ('grad', 'logp', 'logp_var', 'top1', 'rank', 'beliefs'):
        np.testing.assert_array_equal(getattr(a, name).numpy(), getattr(b, name).numpy(), err_msg=name)
    assert 'mlbp_plan_compile' not in eng.k.calls


def test_refusals():
    model = synth.make_model(32, 6, seed=2, dtype=np.float32)
    sents = synth.make_corpus(model, 2, k=3, g=1, seed=5)
    eng = _eng(model)
    for field in ('var_label', 'giv_label'):
        for bad in (-1, 32):
            c = Corpus(sents)
            getattr(c, field)[0] = bad
            with pytest.raises(ValueError):
                eng.pseudo_likelihood(c)
    assert eng.k.calls.count('mlbp_pseudo_likelihood') == 0
    eng.set_theta(FLAT[0], FLAT[1], with_grad=False)
    with pytest.raises(ValueError):
        eng.pseudo_likelihood(Corpus(sents))
    eng.pseudo_likelihood(Corpus(sents), want_grad=False)
    from macaronicusermodeling_b200.trainer import Trainer
    with pytest.raises(ValueError):
        Trainer(eng, objective='bethe')
    with pytest.raises(ValueError):
        Trainer(eng, objective='pl').step(eng.prepare(Corpus(sents)), np.zeros((2, 4), dtype=np.int32), 0.1)
    for kw in (dict(approx_inference=True), dict(approx_beliefs=True)):
        with pytest.raises(ValueError):
            Trainer(eng, objective='pl').step(Corpus(sents), None, 0.1, **kw)
    Trainer(eng, objective='pl').step(Corpus(sents), None, 0.1, approx_inference=False, approx_beliefs=False)


def _trainer_step(sents, N, lr=0.05):
    from macaronicusermodeling_b200.trainer import Trainer
    model = synth.make_model(48, 8, seed=2, dtype=np.float32)
    tr = Trainer(Engine(model, kernels=PLKernels()), reg_param=0.2, N=N, objective='pl')
    tr.theta_ee, tr.theta_ed = np.array(FLAT[0]), np.array(FLAT[1])
    red = tr.step(Corpus(sents), None, lr)
    return model, tr, tr.apply(red, lr)


def test_trainer_pl_step_against_the_model_reference():
    model = synth.make_model(48, 8, seed=2, dtype=np.float32)
    sents = synth.make_corpus(model, 6, k=4, g=1, seed=4)
    _, tr, h = _trainer_step(sents, N=20)
    c = Corpus(sents)
    lp, g, _ = pl_oracle.model_reference(c, model, *FLAT)
    gs = g.sum(axis=0)
    reg = 0.2 / 20
    np.testing.assert_allclose(h[:9], gs, rtol=1e-4, atol=2e-6 * len(sents))
    np.testing.assert_allclose(tr.theta_ee, np.array(FLAT[0]) + 0.05 * (h[:3] - 6 * reg * np.array(FLAT[0])), rtol=1e-15)
    assert h[9] == pytest.approx(lp.sum(), abs=1e-4) and h[13] == c.n_vars and h[14] == 6 and h[15] == 0


def _gloo_worker(rank, world, port, out):
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    model = synth.make_model(48, 8, seed=2, dtype=np.float32)
    sents = synth.make_corpus(model, 6, k=4, g=1, seed=4)
    _, tr, h = _trainer_step(sents[rank::world], N=20)
    out[rank] = h.tolist()
    dist.destroy_process_group()


def test_two_gloo_ranks_give_the_16_vector_of_one():
    model = synth.make_model(48, 8, seed=2, dtype=np.float32)
    sents = synth.make_corpus(model, 6, k=4, g=1, seed=4)
    _, _, want = _trainer_step(sents, N=20)
    out = mp.Manager().dict()
    mp.spawn(_gloo_worker, args=(2, 29600 + os.getpid() % 2000, out), nprocs=2, join=True)
    for r in (0, 1):
        np.testing.assert_allclose(np.array(out[r]), want, rtol=1e-12, atol=1e-12)


# ---------------------------------------------------------------------------------------------------- command line
N_SENT = 40


def _run_cli(argv, rc=0):
    from macaronicusermodeling_b200 import engine, train_cli
    import test_predict_shard_host as sh

    class Kernels(PLKernels, sh.FormatKernels):
        pass

    engine.Kernels = Kernels
    assert train_cli.main(argv) == rc


def _worker(rank, world, port, argv):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank), LOCAL_RANK=str(rank),
                      WORLD_SIZE=str(world))
    _run_cli(argv)
    dist.destroy_process_group()


def _read(path):
    with open(path, 'rb') as f:
        return f.read()


def test_cli_pseudo_likelihood_lines_and_file_one_rank_equals_two_ranks(tmp_path, capsys):
    from predict_cases import write_case
    base = write_case(tmp_path, synth.make_model(48, 12, seed=5), N_SENT, seed=3)
    plain, one, two = tmp_path / 'plain', tmp_path / 'one', tmp_path / 'two'
    for d in (plain, one, two):
        d.mkdir()
    _run_cli(base + ['--save_predictions', str(plain / 'out.pred')])
    out_plain = capsys.readouterr().out
    _run_cli(base + ['--pseudo_likelihood', '--save_predictions', str(one / 'out.pred')])
    out_pl = capsys.readouterr().out
    assert out_pl.startswith(out_plain)
    tail = out_pl[len(out_plain):].strip().splitlines()
    assert [l.split(':')[0] for l in tail] == ['prediction pseudo log-likelihood', 'prediction pseudo Prec at 0']
    mp.spawn(_worker, args=(2, 31700 + 2 * (os.getpid() % 1000), base + ['--pseudo_likelihood', '--save_predictions',
                                                                       str(two / 'out.pred')]), nprocs=2, join=True)
    for name in ('out.pred', 'out.pred.dist'):
        assert _read(plain / name) == _read(one / name) == _read(two / name), name
    assert _read(one / 'out.pred.pl') == _read(two / 'out.pred.pl')
    assert sorted(os.listdir(two)) == ['out.pred', 'out.pred.dist', 'out.pred.pl']
    lines = _read(one / 'out.pred.pl').decode().splitlines()
    assert len(lines) == N_SENT
    tot, n_tok = 0.0, 0
    for i, l in enumerate(lines):
        sid, plv, blv = l.split('\t')
        assert int(sid) == i
        plv, blv = ([float(x) for x in c.split(' ')] for c in (plv, blv))
        assert len(plv) == len(blv) and all(x <= 0 for x in plv)
        tot, n_tok = tot + sum(plv), n_tok + len(plv)
    assert float(tail[0].split()[-1]) == pytest.approx(tot / N_SENT, rel=1e-12)
    assert tail[1].split()[-2:] == ['total:', str(n_tok)]


def test_cli_objective_pl_trains_and_writes_params(tmp_path, capsys):
    from predict_cases import write_case
    from macaronicusermodeling_b200.train_compat import read_params
    base = write_case(tmp_path, synth.make_model(40, 10, seed=6), 24, seed=4)
    args = [a for a in base]
    i = args.index('--load_params')
    del args[i:i + 2]
    ti = args[args.index('--ti') + 1]
    train = args + ['--tune', ti, '--epochs', '2', '--minibatch', '8', '--pseudo_likelihood']
    _run_cli(train + ['--objective', 'pl', '--save_params', str(tmp_path / 'pl.params')])
    out = capsys.readouterr().out
    assert out.count('train pseudo log-likelihood:') == 2 and 'train prediction probs:' not in out
    assert out.count('tune prediction probs:') == 2 and out.count('tune prediction pseudo log-likelihood:') == 2
    te = read_params(str(tmp_path / 'pl.params'))[1]
    assert np.abs(te).sum() > 0
    _run_cli(train + ['--save_params', str(tmp_path / 'lbp.params')])
    out = capsys.readouterr().out
    assert out.count('train prediction probs:') == 2 and 'train pseudo log-likelihood:' not in out


def test_cli_refuses_pl_training_with_adaptation_or_approximations(tmp_path):
    from predict_cases import write_case
    base = write_case(tmp_path, synth.make_model(32, 8, seed=5), 4, seed=3)
    for extra in (['--user_adapt'], ['--experience_adapt'], ['--use_approx_inference'], ['--use_approx_beliefs']):
        _run_cli(base + ['--objective', 'pl', '--save_params', str(tmp_path / 'x.params')] + extra, rc=1)


def _predict_results(out_dir, pseudo):
    """train_cli.predict writing .pred / .dist (and .pl with `pseudo`) on this process's rank: (number of results, results)"""
    import random
    from macaronicusermodeling_b200 import train_cli
    import test_predict_shard_host as sh

    class Kernels(PLKernels, sh.FormatKernels):
        pass

    model = synth.make_model(40, 9, seed=4, dtype=np.float32)
    raw = [synth.make_sentence(model, l, seed=70 + i, sent_id=i) for i, l in enumerate(['pgp', 'ppp', 'gpp', 'pp', 'pgpp', 'p'])]
    sents = [synth.sentence_to_arrays(r) for r in raw]
    eng = Engine(model, kernels=Kernels())
    eng.set_theta(FLAT[0], FLAT[1], with_grad=True)
    opts = train_cli.parse(['--ti', 'x'])
    res = train_cli.predict(eng, train_cli.prediction_units(len(sents), batch=2), sents, raw,
                            [synth.en_word(i) for i in range(model['V'])], opts, random.Random(5), False,
                            out_path=os.path.join(out_dir, 'out.pred'), pseudo=pseudo)
    return len(res), [res[0], list(res[1])] + ([list(res[2])] if len(res) > 2 else [])


def _predict_worker(rank, world, port, out_dir, pseudo, out):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    out[rank] = _predict_results(out_dir, pseudo)
    dist.destroy_process_group()


@pytest.mark.parametrize('pseudo', [False, True], ids=['plain', 'pseudo'])
def test_predict_results_with_output_files_on_one_and_two_ranks(tmp_path, pseudo):
    """predict() returns (logp, counts) -- plus the pseudo-likelihood pair only when asked -- on every rank, files or not"""
    one, two = tmp_path / 'one', tmp_path / 'two'
    one.mkdir()
    two.mkdir()
    n, want = _predict_results(str(one), pseudo)
    assert n == (3 if pseudo else 2)
    out = mp.Manager().dict()
    mp.spawn(_predict_worker, args=(2, 30600 + os.getpid() % 1000 + (7 if pseudo else 0), str(two), pseudo, out), nprocs=2,
             join=True)
    for r in (0, 1):
        assert out[r][0] == n, r
        np.testing.assert_allclose(out[r][1][0], want[0], rtol=1e-12)
        assert out[r][1][1:] == want[1:], r
    for name in ['out.pred', 'out.pred.dist'] + (['out.pred.pl'] if pseudo else []):
        assert _read(one / name) == _read(two / name), name
