"""CPU tier of the Gibbs sampler (K12, Engine.sample, train_cli --gibbs): Philox4x32-10 against Random123's known answers, the
NumPy reference sampler (tests/gibbs_oracle.py) against brute-force marginals on trees and loopy sentences -- and the same check
failing when a pairwise factor is dropped --, one-variable sentences against the normalised unary row, and the engine + command
line on the emulated kernels (tests/fake_gibbs_kernels.py): determinism, batch / order / micro-batch invariance, isolation from
sum-product runs, the refusals, the printed lines and the .gibbs file, two gloo ranks writing the same .gibbs as one, and
.pred / .dist / .joint / .map bytes that --gibbs leaves alone."""
import os
import sys

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))

import gibbs_oracle as go  # noqa: E402
from fake_gibbs_kernels import GibbsKernels  # noqa: E402
from fake_joint_kernels import JointKernels  # noqa: E402
from fake_map_kernels import MapKernels  # noqa: E402
from macaronicusermodeling_b200 import build, synth  # noqa: E402
from macaronicusermodeling_b200._lib import MlbpError  # noqa: E402
from macaronicusermodeling_b200.engine import Corpus, Engine  # noqa: E402

FLAT = ([0.3, -0.2, 0.1], [0.8, -0.5, 0.6, 0.4, 0.3, -0.2])
PEAKED = ([2.0, 1.2, -0.3], [2.0, -1.0, 0.6, 0.4, 0.3, -0.2])
U24 = 2.0 ** -24


@pytest.fixture(scope='module', autouse=True)
def _built():
    build.build()


def test_philox_known_answers():
    cases = [((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
             ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
             ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
              (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1))]
    for ctr, key, want in cases:
        assert [int(w) for w in go.philox4x32_10(np.array(ctr), np.array(key))] == list(want)


def _setup(V, layouts, theta, seed):
    model = synth.make_model(V, 5, seed=seed, dtype=np.float32)
    sents = [synth.sentence_to_arrays(synth.make_sentence(model, l, seed=seed * 10 + i, n_history=2)) for i, l in enumerate(layouts)]
    eng = Engine(model, kernels=GibbsKernels())
    eng.set_theta(theta[0], theta[1], with_grad=True)
    return model, sents, eng


def _reference(eng, corpus, chains, burn_in, n_keep, drop=None):
    """the reference sampler on the engine's U rows and planes; drop = (sentence, pair index) leaves one factor out"""
    U = eng.unary_rows(corpus)[0].numpy()
    V = eng.V
    planes = [eng.planes[p].numpy() for p in range(8)]
    keep = np.ones(corpus.n_pairs, dtype=bool)
    po = corpus.pair_off.copy()
    if drop is not None:
        keep[int(corpus.pair_off[drop[0]]) + drop[1]] = False
        po[drop[0] + 1:] -= 1
    acc, _, _ = go.sample(corpus.var_off, po, corpus.pair_v0[keep], corpus.pair_v1[keep], corpus.pair_gap1[keep],
                          np.arange(corpus.n_sent), U, planes, eng.colsums.numpy(), eng.scale_exp, 11, chains, burn_in, n_keep,
                          False)
    return acc[:, :, :V].astype(np.float64) / n_keep                     # per-chain Rao-Blackwell marginals


def _z_scores(p_chain, exact):
    """|p_hat - p| / (SE + 1e-6 / 5) for every word of every variable"""
    p_hat = p_chain.mean(axis=0)
    se = p_chain.std(axis=0, ddof=1) / np.sqrt(p_chain.shape[0])
    return np.abs(p_hat - exact) / (se + 1e-6 / 5.0)


@pytest.mark.parametrize('layouts, V', [(['pp', 'pgp'], 9), (['ppp', 'pgpp'], 7), (['pppp'], 6)])
@pytest.mark.parametrize('theta', [FLAT, PEAKED], ids=['flat', 'peaked'])
def test_reference_sampler_against_brute_force(layouts, V, theta):
    model, sents, eng = _setup(V, layouts, theta, seed=V)
    corpus = Corpus(sents)
    p = _reference(eng, corpus, 16, 50, 1000)
    exact = [go.exact_marginals(model, s, theta[0], theta[1]) for s in sents]
    ex = np.concatenate(exact)
    z = _z_scores(p, ex)
    assert z.max() <= 5.0, z.max()
    # 3-sweep loopy BP on the same sentences, for scale (exact on the trees)
    roots = corpus.roots_from_positions(synth.draw_roots(sents, 3, seed=1))
    b = eng.run(corpus, roots, 3, want_grad=False, want_beliefs=True).beliefs.numpy()[:, :V].astype(np.float64)
    print('k = %s: BP max |b - p| %.3e, Gibbs max |p_hat - p| %.3e, max z %.2f' % (
        [len(x) for x in exact], np.abs(b - ex).max(), np.abs(p.mean(axis=0) - ex).max(), z.max()))


def test_the_check_has_power_a_dropped_factor_fails_it():
    theta = PEAKED
    model, sents, eng = _setup(7, ['ppp'], theta, seed=7)
    corpus = Corpus(sents)
    ex = go.exact_marginals(model, sents[0], theta[0], theta[1])
    assert _z_scores(_reference(eng, corpus, 16, 50, 1000), ex).max() <= 5.0
    assert _z_scores(_reference(eng, corpus, 16, 50, 1000, drop=(0, 1)), ex).max() > 5.0


def test_one_variable_marginals_are_the_normalised_unary_row():
    model, sents, eng = _setup(37, ['gpg', 'p', 'ggp'], FLAT, seed=3)
    corpus = Corpus(sents)
    n_keep = 50
    r = eng.sample(corpus, chains=3, burn_in=2, n_keep=n_keep, want_beliefs=True)
    U = eng.unary_rows(corpus)[0].numpy()[:, :37].astype(np.float64)
    want = U / U.sum(axis=1, keepdims=True)
    got = r.beliefs.numpy()[:, :37].astype(np.float64)
    assert (np.abs(got - want) <= (n_keep + 1) * U24 * want).all()


def _eng(model, **kw):
    eng = Engine(model, kernels=GibbsKernels(), **kw)
    eng.set_theta(FLAT[0], FLAT[1], with_grad=False)
    return eng


def _outs(r):
    return [r.logp.numpy(), r.logp_var.numpy(), r.top1.numpy(), r.rank.numpy(), r.beliefs.numpy(), r.label_prob.numpy(),
            r.samples.numpy()]


def test_emulated_kernels_are_deterministic_and_batch_invariant():
    model = synth.make_model(40, 6, seed=2, dtype=np.float32)
    sents = synth.make_corpus(model, 5, k=3, g=1, seed=5) + synth.make_corpus(model, 2, k=1, g=2, seed=6)
    kw = dict(chains=3, burn_in=2, n_keep=3, seed=(1 << 63) + 12345, want_beliefs=True, want_samples=True)
    eng = _eng(model)
    ids = np.arange(100, 100 + len(sents))
    a = _outs(eng.sample(Corpus(sents), sent_ids=ids, **kw))
    for x, y in zip(a, _outs(eng.sample(Corpus(sents), sent_ids=ids, **kw))):
        np.testing.assert_array_equal(x, y)
    off = Corpus(sents).var_off
    # one sentence alone, with its id, is the same slice of every output
    for s in (0, 4, 6):
        one = _outs(eng.sample(Corpus([sents[s]]), sent_ids=ids[s:s + 1], **kw))
        lo, hi = off[s], off[s + 1]
        for j, (x, y) in enumerate(zip(a, one)):
            want = x[s:s + 1] if j == 0 else (x[:, :, lo:hi] if j == 6 else x[lo:hi])
            np.testing.assert_array_equal(want, y, err_msg='output %d of sentence %d' % (j, s))
    # reordered
    order = [3, 0, 6, 2, 5, 1, 4]
    ro = _outs(eng.sample(Corpus([sents[i] for i in order]), sent_ids=ids[order], **kw))
    roff = Corpus([sents[i] for i in order]).var_off
    for pos, s in enumerate(order):
        np.testing.assert_array_equal(ro[1][roff[pos]:roff[pos + 1]], a[1][off[s]:off[s + 1]])
        np.testing.assert_array_equal(ro[6][:, :, roff[pos]:roff[pos + 1]], a[6][:, :, off[s]:off[s + 1]])
    # micro-batched under a small workspace
    small = _eng(model, workspace_bytes=3 * 3 * 64 * 4 * 5)
    rb = small.sample(Corpus(sents), sent_ids=ids, **kw)
    assert rb.stats['micro_batches'] > 2
    for x, y in zip(a, _outs(rb)):
        np.testing.assert_array_equal(x, y)
    # another seed gives other draws
    assert not np.array_equal(a[6], _outs(eng.sample(Corpus(sents), sent_ids=ids, **dict(kw, seed=1)))[6])


def test_sum_product_outputs_are_bit_identical_around_a_sample_call():
    model = synth.make_model(64, 9, seed=9, dtype=np.float32)
    sents = synth.make_corpus(model, 4, k=4, g=1, seed=3)
    corpus = Corpus(sents)
    roots = corpus.roots_from_positions(synth.draw_roots(sents, 3, seed=4))
    eng = Engine(model, kernels=GibbsKernels())
    eng.set_theta(FLAT[0], FLAT[1], with_grad=True)
    kw = dict(want_grad=True, want_marg=True, want_beliefs=True)
    a = eng.run(corpus, roots, 3, **kw)
    g = eng.sample(corpus, chains=2, burn_in=1, n_keep=2)
    b = eng.run(corpus, roots, 3, **kw)
    for name in ('grad', 'logp', 'logp_var', 'top1', 'rank', 'beliefs'):
        np.testing.assert_array_equal(getattr(a, name).numpy(), getattr(b, name).numpy(), err_msg=name)
    assert g.grad is None and a.label_prob is None
    # logp is the per-sentence sum of logp_var (mlbp_gradient_reduce), as for BP
    np.testing.assert_allclose(g.logp.numpy(), [g.logp_var.numpy()[corpus.var_off[s]:corpus.var_off[s + 1]].sum()
                                                for s in range(corpus.n_sent)], rtol=1e-12)


def test_refusals():
    model = synth.make_model(32, 6, seed=2, dtype=np.float32)
    corpus = Corpus(synth.make_corpus(model, 2, k=2, g=1, seed=5))
    eng = _eng(model)
    for kw in (dict(chains=0), dict(n_keep=0), dict(burn_in=-1)):
        with pytest.raises(MlbpError):
            eng.sample(corpus, **kw)
    assert eng.k.calls.count('mlbp_gibbs_reduce') == 0


# ---------------------------------------------------------------------------------------------------- command line
N_SENT = 60


class _CliKernels(GibbsKernels, MapKernels, JointKernels):
    pass


def _run_cli(argv):
    from macaronicusermodeling_b200 import engine, train_cli
    import test_predict_shard_host as sh

    class Kernels(_CliKernels, sh.FormatKernels):
        pass

    engine.Kernels = Kernels
    assert train_cli.main(argv) == 0


def _worker(rank, world, port, argv):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank), LOCAL_RANK=str(rank),
                      WORLD_SIZE=str(world))
    _run_cli(argv)
    dist.destroy_process_group()


def _read(path):
    with open(path, 'rb') as f:
        return f.read()


def test_cli_gibbs_lines_and_file_one_rank_equals_two_ranks_and_other_outputs_do_not_move(tmp_path, capsys):
    from predict_cases import write_case
    model = synth.make_model(48, 12, seed=5)
    base = write_case(tmp_path, model, N_SENT, seed=3) + ['--joint_likelihood', '--map_decode']
    plain, one, two = tmp_path / 'plain', tmp_path / 'one', tmp_path / 'two'
    for d in (plain, one, two):
        d.mkdir()
    _run_cli(base + ['--save_predictions', str(plain / 'out.pred')])
    out_plain = capsys.readouterr().out
    _run_cli(base + ['--gibbs', '3', '--save_predictions', str(one / 'out.pred')])
    out_g = capsys.readouterr().out
    assert out_g.startswith(out_plain)
    tail = out_g[len(out_plain):].strip().splitlines()
    assert [l.split(':')[0] for l in tail] == ['prediction Gibbs probs', 'prediction Gibbs Prec at 0',
                                               'prediction Gibbs max standard error']
    port = 31900 + 2 * (os.getpid() % 1000)
    mp.spawn(_worker, args=(2, port, base + ['--gibbs', '3', '--save_predictions', str(two / 'out.pred')]), nprocs=2, join=True)
    for name in ('out.pred', 'out.pred.dist', 'out.pred.joint', 'out.pred.map'):
        assert _read(plain / name) == _read(one / name) == _read(two / name), name
    assert _read(one / 'out.pred.gibbs') == _read(two / 'out.pred.gibbs')
    assert sorted(os.listdir(two)) == ['out.pred', 'out.pred.dist', 'out.pred.gibbs', 'out.pred.joint', 'out.pred.map']
    lines = _read(one / 'out.pred.gibbs').decode().splitlines()
    assert len(lines) == N_SENT
    # the numbers behind the printed lines: the Gibbs log-probabilities, their standard errors, BP's logp_var
    import json
    raw = [json.loads(l) for l in open(base[1])]
    en2id = dict((w.strip(), i) for i, w in enumerate(open(base[3])))
    tot_lp, max_se, n_tok = 0.0, 0.0, 0
    for i, l in enumerate(lines):
        sid, glp, se, blp = l.split('\t')
        assert int(sid) == i
        k = len(synth.sentence_to_arrays(raw[i], en2id).predicted)
        glp, se, blp = ([float(x) for x in c.split(' ')] for c in (glp, se, blp))
        assert len(glp) == len(se) == len(blp) == k
        assert all(x <= 0 for x in glp + blp) and all(x >= 0 for x in se)
        tot_lp, max_se, n_tok = tot_lp + sum(glp), max(max_se, max(se)), n_tok + k
    assert float(tail[0].split()[-1]) == pytest.approx(tot_lp / N_SENT, rel=1e-12)
    assert tail[1].split()[-2:] == ['total:', str(n_tok)]
    assert float(tail[2].split()[-1]) == max_se


def test_cli_refuses_gibbs_0(tmp_path):
    from macaronicusermodeling_b200 import train_cli
    from predict_cases import write_case
    base = write_case(tmp_path, synth.make_model(32, 8, seed=5), 4, seed=3)
    for n in ('0', '-2'):
        assert train_cli.main(base + ['--gibbs', n, '--save_predictions', str(tmp_path / 'x.pred')]) == 1
