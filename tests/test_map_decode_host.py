"""CPU tier of max-product decoding: the float64 reference against brute-force enumeration (exact MAP on trees, a score no
better than the optimum on small loopy sentences), the engine's refusals and isolation from sum-product runs, and the engine +
command line path on the emulated K10 / K11 (tests/fake_map_kernels.py), including two gloo ranks writing the same .map as
one and .pred / .dist / .joint bytes that --map_decode leaves alone."""
import os
import sys

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))

import map_checks as mc  # noqa: E402
import maxprod_oracle as mo  # noqa: E402
from fake_joint_kernels import JointKernels  # noqa: E402
from fake_map_kernels import MapKernels  # noqa: E402
from macaronicusermodeling_b200 import build, synth  # noqa: E402
from macaronicusermodeling_b200.engine import Corpus, Engine  # noqa: E402
from oracle import lbp_oracle as orc  # noqa: E402


@pytest.fixture(scope='module', autouse=True)
def _built():
    build.build()


def _model(V, seed):
    return synth.make_model(V, 12, seed=seed, dtype=np.float32)


@pytest.mark.parametrize('V', [60, 67])
def test_oracle_decoding_is_the_exact_map_on_trees(V):
    model = _model(V, 4)
    tb = orc.Tables(model, mc.THETA_EE, mc.THETA_ED)
    for sent in [synth.sentence_to_arrays(synth.make_sentence(model, l, seed=11 + i, n_history=2))
                 for i, l in enumerate(mc.TREE_LAYOUTS)]:
        g = orc.Graph(sent)
        assert len(g.var_ids) == 2 and not g.has_loops(g.var_ids[0])
        roots = [g.var_ids[0], g.var_ids[1], g.var_ids[0], g.var_ids[1]]
        mm, dec = mo.decode(tb, sent, roots)
        best, best_score, label_score = mc.brute_force(model, sent, mc.THETA_EE, mc.THETA_ED)
        np.testing.assert_array_equal(dec, best)
        c = Corpus([sent])
        assert mo.assignment_scores(model, mc.THETA_EE, mc.THETA_ED, c, dec)[0] == pytest.approx(best_score, abs=1e-6)
        assert mo.assignment_scores(model, mc.THETA_EE, mc.THETA_ED, c, c.var_label)[0] == pytest.approx(label_score, abs=1e-6)
        # on a tree the max-marginal of the decoded word is the largest joint potential: all max-marginals share one scale
        assert (mm.argmax(axis=1) == dec).all()


@pytest.mark.parametrize('V', [41, 67])
def test_oracle_decoding_scores_no_better_than_brute_force_on_loopy_triples(V):
    model = _model(V, 5)
    sents = synth.make_corpus(model, 4, k=3, g=1, seed=12)
    roots = synth.draw_roots(sents, 3, seed=2)
    tb = orc.Tables(model, mc.THETA_EE, mc.THETA_ED)
    hits = 0
    for i, sent in enumerate(sents):
        _, dec = mo.decode(tb, sent, roots[i])
        best, best_score, label_score = mc.brute_force(model, sent, mc.THETA_EE, mc.THETA_ED)
        c = Corpus([sent])
        got = mo.assignment_scores(model, mc.THETA_EE, mc.THETA_ED, c, dec)[0]
        assert got <= best_score + 1e-6
        assert mo.assignment_scores(model, mc.THETA_EE, mc.THETA_ED, c, c.var_label)[0] == pytest.approx(label_score, abs=1e-6)
        hits += int((dec == best).all())
    assert hits >= 1                                              # max-product BP usually finds the optimum of a triangle


def _engine(model):
    return Engine(model, kernels=MapKernels())


def test_engine_refuses_what_max_product_does_not_define():
    model = _model(64, 2)
    sents = synth.make_corpus(model, 3, k=4, g=1, seed=3)
    corpus = Corpus(sents)
    roots = corpus.roots_from_positions(synth.draw_roots(sents, 3, seed=4))
    eng = _engine(model)
    eng.set_theta(mc.THETA_EE, mc.THETA_ED)
    for kw in (dict(want_grad=True), dict(want_joint=True), dict(approx_inference=True), dict(approx_beliefs=True),
               dict(want_marg=False)):
        args = dict(want_grad=False, max_product=True)
        args.update(kw)
        with pytest.raises(ValueError):
            eng.run(corpus, roots, 3, **args)
    assert eng.k.calls.count('mlbp_factor_to_var_maxprod') == 0


def test_engine_decode_matches_the_oracle_and_scores_match_numpy():
    model = _model(67, 7)
    sents = synth.make_corpus(model, 5, k=5, g=1, seed=21) + synth.make_corpus(model, 3, k=3, g=0, seed=22) + \
        [synth.sentence_to_arrays(synth.make_sentence(model, l, seed=30 + i, n_history=2)) for i, l in enumerate(mc.TREE_LAYOUTS)]
    roots = synth.draw_roots(sents, 3, seed=8)
    r, corpus = mc.engine_decode(_engine(model), sents, roots, mc.THETA_EE, mc.THETA_ED)
    want = mc.oracle_decode(model, sents, roots, mc.THETA_EE, mc.THETA_ED)
    excluded = mc.check_decode(r, corpus, model, want, mc.THETA_EE, mc.THETA_ED)
    assert excluded <= 2
    assert (r.map_score.numpy() >= r.label_score.numpy() - 1e-9).sum() >= len(sents) - 2
    # the log-marginal outputs are K5's, on the max-marginals
    B = r.beliefs.numpy()[:, :67].astype(np.float64)
    lab = corpus.var_label
    np.testing.assert_allclose(r.logp_var.numpy(), np.log(B[np.arange(len(lab)), lab]), rtol=1e-6)
    assert (r.rank.numpy() == (B > B[np.arange(len(lab)), lab][:, None]).sum(axis=1)).all()


def test_sum_product_outputs_are_bit_identical_around_a_max_product_run():
    model = _model(64, 9)
    sents = synth.make_corpus(model, 6, k=5, g=1, seed=3)
    corpus = Corpus(sents)
    roots = corpus.roots_from_positions(synth.draw_roots(sents, 3, seed=4))
    eng = _engine(model)
    eng.set_theta(mc.THETA_EE, mc.THETA_ED, with_grad=True)
    kw = dict(want_grad=True, want_marg=True, want_beliefs=True)
    a = eng.run(corpus, roots, 3, **kw)
    m = eng.run(corpus, roots, 3, want_grad=False, want_beliefs=True, max_product=True)
    b = eng.run(corpus, roots, 3, **kw)
    for name in ('grad', 'logp', 'logp_var', 'top1', 'rank', 'beliefs'):
        np.testing.assert_array_equal(getattr(a, name).numpy(), getattr(b, name).numpy(), err_msg=name)
    assert not np.array_equal(a.beliefs.numpy(), m.beliefs.numpy())
    assert a.map_score is None and m.map_score is not None
    # the max-product constant rows are rebuilt after set_theta, and the sum-product ones are not touched by them
    const = eng.const_rows.clone()
    eng.run(corpus, roots, 3, want_grad=False, max_product=True)
    np.testing.assert_array_equal(eng.const_rows.numpy(), const.numpy())
    eng.set_theta([0.2, 0.1, -0.3], mc.THETA_ED)
    assert not eng.map_const_ok
    m2 = eng.run(corpus, roots, 3, want_grad=False, max_product=True)
    assert not np.array_equal(m2.map_score.numpy(), m.map_score.numpy())


# ---------------------------------------------------------------------------------------------------- command line
N_SENT = 140


class _CliKernels(MapKernels, JointKernels):
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


def test_cli_map_file_one_rank_equals_two_ranks_and_other_outputs_do_not_move(tmp_path, capsys):
    from predict_cases import write_case
    model = synth.make_model(64, 16, seed=5)
    base = write_case(tmp_path, model, N_SENT, seed=3) + ['--joint_likelihood']
    plain, one, two = tmp_path / 'plain', tmp_path / 'one', tmp_path / 'two'
    for d in (plain, one, two):
        d.mkdir()
    _run_cli(base + ['--save_predictions', str(plain / 'out.pred')])
    out_plain = capsys.readouterr().out
    _run_cli(base + ['--map_decode', '--save_predictions', str(one / 'out.pred')])
    out_map = capsys.readouterr().out
    assert out_map.startswith(out_plain)
    tail = out_map[len(out_plain):].strip().splitlines()
    assert [l.split(':')[0] for l in tail] == ['prediction MAP token accuracy', 'prediction MAP sentence accuracy']
    port = 30900 + 2 * (os.getpid() % 1000)
    mp.spawn(_worker, args=(2, port, base + ['--map_decode', '--save_predictions', str(two / 'out.pred')]), nprocs=2, join=True)
    for name in ('out.pred', 'out.pred.dist', 'out.pred.joint'):
        assert _read(plain / name) == _read(one / name) == _read(two / name), name
    assert _read(one / 'out.pred.map') == _read(two / 'out.pred.map')
    assert sorted(os.listdir(two)) == ['out.pred', 'out.pred.dist', 'out.pred.joint', 'out.pred.map']
    lines = _read(one / 'out.pred.map').decode().splitlines()
    assert len(lines) == N_SENT
    # the decoded words, per sentence in position order, and the statistics printed from them
    import json
    raw = [json.loads(l) for l in open(base[1])]
    en = [l.strip() for l in open(base[3])]
    en2id = dict((w, i) for i, w in enumerate(en))
    tok_ok = sent_ok = n_tok = 0
    for i, l in enumerate(lines):
        sid, words, ms, ls = l.split('\t')
        assert int(sid) == i
        sent = synth.sentence_to_arrays(raw[i], en2id)
        dec = [en2id[w] for w in words.split(' ')]
        lab = [int(sent.label[p]) for p in sent.predicted]
        assert len(dec) == len(lab)
        if len(lab) <= 2:                                         # a tree: max-product finds the exact optimum
            assert float(ms) >= float(ls) - 1e-9
        ok = np.array(dec) == np.array(lab)
        tok_ok, sent_ok, n_tok = tok_ok + int(ok.sum()), sent_ok + int(ok.all()), n_tok + len(lab)
    assert tail[0].split()[4:] == ['%0.2f' % (100.0 * tok_ok / n_tok), 'total:', str(n_tok)]
    assert tail[1].split()[4:] == ['%0.2f' % (100.0 * sent_ok / N_SENT), 'total:', str(N_SENT)]


def test_cli_refuses_map_decode_with_the_approximate_modes(tmp_path):
    from macaronicusermodeling_b200 import train_cli
    from predict_cases import write_case
    base = write_case(tmp_path, synth.make_model(32, 8, seed=5), 4, seed=3)
    for flag in ('--use_approx_inference', '--use_approx_beliefs'):
        assert train_cli.main(base + ['--map_decode', flag, '--save_predictions', str(tmp_path / 'x.pred')]) == 1
