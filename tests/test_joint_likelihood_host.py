"""CPU tier of the joint log-likelihood (Bethe estimate at the final messages): the float64 reference against brute-force
enumeration and its invariance to message scales, the schedule compiler's joint section (flag bit 4), and the engine + command
line path on the emulated K9 (tests/fake_joint_kernels.py), including two gloo ranks writing the same .joint as one."""
import ctypes
import os
import sys

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))

import bethe_oracle as bo  # noqa: E402
import joint_checks as jc  # noqa: E402
from fake_joint_kernels import JointKernels  # noqa: E402
from macaronicusermodeling_b200 import _lib, build, synth  # noqa: E402
from macaronicusermodeling_b200.engine import (H_PAIR_M0, H_PAIR_M1, H_WORDS, PLAN_BLOB_WORDS, Corpus,  # noqa: E402
                                               Engine)
from oracle import lbp_oracle as orc  # noqa: E402


@pytest.fixture(scope='module', autouse=True)
def _built():
    build.build()


@pytest.mark.parametrize('V', [60, 67])
def test_oracle_equals_brute_force_on_trees(V):
    model = synth.make_model(V, 12, seed=4)
    tb = orc.Tables(model, jc.THETA_EE, jc.THETA_ED)
    for sent in jc.tree_sentences(model):
        g = orc.Graph(sent)
        assert len(g.var_ids) == 2 and not g.has_loops(g.var_ids[0])
        roots = [g.var_ids[0], g.var_ids[1], g.var_ids[0], g.var_ids[1]]
        want = jc.brute_force_joint(model, sent, jc.THETA_EE, jc.THETA_ED)
        assert abs(bo.bethe_joint_logp(tb, sent, roots) - want) < 1e-10 * max(1.0, abs(want))
    # one predicted token: the joint is its log-marginal
    one = synth.sentence_to_arrays(synth.make_sentence(model, 'gpg', seed=3, n_history=2))
    p = int(one.predicted[0])
    r = orc.run_fast(tb, one, [p] * 4)
    assert bo.bethe_joint_logp(tb, one, [p] * 4) == pytest.approx(r['logp'], abs=1e-12)


def test_oracle_is_invariant_to_rescaling_any_one_message():
    model = synth.make_model(40, 10, seed=6)
    sent = synth.make_corpus(model, 1, k=5, g=1, seed=9)[0]
    roots = synth.draw_roots([sent], 3, seed=2)[0]
    tb = orc.Tables(model, jc.THETA_EE, jc.THETA_ED)
    msgs = bo.final_messages(tb, sent, roots)
    base = bo.bethe_joint_logp(tb, sent, roots, messages=msgs)
    assert base == bo.bethe_joint_logp(tb, sent, roots)
    # the final messages are run_fast's: the marginals they give are the oracle's
    g = msgs['graph']
    ref = orc.run_fast(tb, sent, roots)['marginals']
    for i, v in enumerate(g.var_ids):
        m = msgs['uprod'][v] * np.prod([msgs['f2v'][f, v] for f in g.facset[v] if g.factors[f].arity == 2], axis=0)
        np.testing.assert_allclose(m / m.sum(), ref[i], rtol=1e-12, atol=1e-15)
    for part in ('uprod', 'v2f', 'f2v'):
        for key in list(msgs[part])[:6]:
            m = dict(msgs)
            m[part] = dict(msgs[part])
            m[part][key] = msgs[part][key] * 37.5
            assert bo.bethe_joint_logp(tb, sent, roots, messages=m) == pytest.approx(base, rel=1e-12, abs=1e-12), (part, key)


def test_oracle_reports_minus_inf_for_a_label_of_belief_zero():
    model = synth.make_model(40, 10, seed=6)
    sent = synth.make_corpus(model, 1, k=4, g=0, seed=9)[0]
    roots = synth.draw_roots([sent], 3, seed=2)[0]
    tb = orc.Tables(model, jc.THETA_EE, jc.THETA_ED)
    msgs = bo.final_messages(tb, sent, roots)
    g = msgs['graph']
    v = g.var_ids[1]
    m = dict(msgs)
    m['uprod'] = dict(msgs['uprod'])
    m['uprod'][v] = msgs['uprod'][v].copy()
    m['uprod'][v][g.label[v]] = 0.0
    assert bo.bethe_joint_logp(tb, sent, roots, messages=m) == -np.inf


def _blob(eng, corpus, roots, want_grad, want_marg, want_joint, reuse_z=True):
    handle, sizes = eng.compile(corpus, roots, 3, want_grad, want_marg, reuse_z=reuse_z, want_joint=want_joint)
    try:
        b = np.empty(int(sizes[PLAN_BLOB_WORDS]), dtype=np.int32)
        _lib.check(_lib.load().mlbp_plan_export(handle, ctypes.c_void_p(b.ctypes.data)))
    finally:
        _lib.load().mlbp_plan_destroy(handle)
    return b


@pytest.mark.parametrize('reuse_z', [True, False])
def test_plan_joint_section_templated_equals_literal_and_leaves_the_rest(reuse_z, monkeypatch):
    model = synth.make_model(64, 16, seed=1)
    eng = Engine(model, kernels=JointKernels())
    layouts = ['pppp', 'gpgpp', 'ppgpgp', 'pp', 'pgppg', 'gpg', 'ppppppp', 'prpgp', 'p']
    sents = [synth.sentence_to_arrays(synth.make_sentence(model, layouts[(i * 7) % len(layouts)], seed=50 + i, n_history=3))
             for i in range(40)] + synth.make_corpus(model, 12, k=9, g=2, seed=5)
    corpus = Corpus(sents)
    roots = corpus.roots_from_positions(synth.draw_roots(sents, 3, seed=3))
    blobs = {}
    for mode in ('0', '1', '1'):                                 # literal, templated cold, templated warm
        monkeypatch.setenv('MLBP_PLAN_TEMPLATES', mode)
        blobs.setdefault(mode, []).append((_blob(eng, corpus, roots, True, True, False, reuse_z),
                                           _blob(eng, corpus, roots, True, True, True, reuse_z)))
    plain, joint = blobs['0'][0]
    for p, j in blobs['1']:
        np.testing.assert_array_equal(p, plain)
        np.testing.assert_array_equal(j, joint)
    # without the flag nothing is emitted; with it the blob is the plain one plus the two per-factor sections
    assert plain[H_PAIR_M0] == 0 and plain[H_PAIR_M1] == 0
    n_pair = corpus.n_pairs
    assert len(joint) == len(plain) + 2 * n_pair
    hdr = np.arange(H_WORDS)
    keep = (hdr != H_PAIR_M0) & (hdr != H_PAIR_M1)
    np.testing.assert_array_equal(joint[:H_WORDS][keep], plain[:H_WORDS][keep])
    np.testing.assert_array_equal(joint[H_WORDS:len(plain)], plain[H_WORDS:])
    # the mu rows are the rows the marginal stage reads for the factor's two variables
    from macaronicusermodeling_b200.engine import H_MARG_IN, H_MARG_OFF
    m0 = joint[joint[H_PAIR_M0]:joint[H_PAIR_M0] + n_pair]
    m1 = joint[joint[H_PAIR_M1]:joint[H_PAIR_M1] + n_pair]
    moff = joint[joint[H_MARG_OFF]:joint[H_MARG_OFF] + corpus.n_vars + 1]
    min_ = joint[joint[H_MARG_IN]:]
    f = 0
    for s in range(corpus.n_sent):
        v0 = int(corpus.var_off[s])
        slot = {}
        for q in range(int(corpus.pair_off[s]), int(corpus.pair_off[s + 1])):
            a, b = v0 + int(corpus.pair_v0[q]), v0 + int(corpus.pair_v1[q])
            for v, got in ((a, m0[f]), (b, m1[f])):
                k = slot.get(v, 0)
                assert got == min_[moff[v] + k]
                slot[v] = k + 1
            f += 1


def _engine(model):
    return Engine(model, kernels=JointKernels())


def test_engine_joint_matches_brute_force_on_trees_and_logp_on_single_tokens():
    model = synth.make_model(60, 12, seed=4)
    sents = jc.tree_sentences(model) + [synth.sentence_to_arrays(synth.make_sentence(model, 'gpg', seed=3, n_history=2))]
    roots = synth.draw_roots(sents, 3, seed=5)
    r, _ = jc.engine_joint(_engine(model), sents, roots, jc.THETA_EE, jc.THETA_ED)
    lj = r.logp_joint.numpy()
    for i, s in enumerate(sents[:4]):
        want = jc.brute_force_joint(model, s, jc.THETA_EE, jc.THETA_ED)
        assert abs(lj[i] - want) < jc.joint_tol(1, 60), (i, lj[i], want)
    assert lj[4] == r.logp.numpy()[4]


def test_engine_joint_matches_oracle_on_loopy_sentences():
    model = synth.make_model(67, 12, seed=7)
    sents = synth.make_corpus(model, 6, k=5, g=1, seed=21) + synth.make_corpus(model, 3, k=3, g=0, seed=22)
    roots = synth.draw_roots(sents, 3, seed=8)
    r, _ = jc.engine_joint(_engine(model), sents, roots, jc.THETA_EE, jc.THETA_ED)
    want = jc.oracle_joints(model, sents, roots, jc.THETA_EE, jc.THETA_ED)
    tol = jc.joint_tol(np.diff(Corpus(sents).pair_off), 67)
    assert (np.abs(r.logp_joint.numpy() - want) < tol).all(), (r.logp_joint.numpy() - want, tol)


@pytest.mark.parametrize('want_grad', [False, True])
def test_nothing_else_moves(want_grad):
    model = synth.make_model(64, 16, seed=2)
    sents = synth.make_corpus(model, 8, k=5, g=1, seed=3)
    corpus = Corpus(sents)
    roots = corpus.roots_from_positions(synth.draw_roots(sents, 3, seed=4))
    out = []
    for joint in (False, True):
        eng = _engine(model)
        eng.set_theta(jc.THETA_EE, jc.THETA_ED, with_grad=True)
        r = eng.run(corpus, roots, 3, want_grad=want_grad, want_marg=True, want_beliefs=True, want_joint=joint)
        out.append(r)
        assert (r.logp_joint is not None) == joint
    for name in ('grad', 'logp', 'logp_var', 'top1', 'rank', 'beliefs'):
        np.testing.assert_array_equal(getattr(out[0], name).numpy(), getattr(out[1], name).numpy(), err_msg=name)


def test_run_many_passes_want_joint_through_and_refuses_approximate_modes():
    model = synth.make_model(64, 16, seed=4)
    sents = synth.make_corpus(model, 12, k=4, g=1, seed=2)
    corpus = Corpus(sents)
    roots = corpus.roots_from_positions(synth.draw_roots(sents, 3, seed=1))
    eng = _engine(model)
    eng.set_theta(jc.THETA_EE, jc.THETA_ED)
    whole = eng.run(corpus, roots, 3, want_grad=False, want_joint=True)
    eng.rows_budget = lambda: 120
    assert len(eng.microbatches(corpus, 3, True)) > 2
    res = eng.run_many(corpus, roots, 3, want_grad=False, want_joint=True)
    assert len(res) == 5
    np.testing.assert_allclose(res[4].numpy(), whole.logp_joint.numpy(), rtol=1e-12)
    parts = eng.prepare(corpus, 3, want_grad=True)
    np.testing.assert_allclose(eng.run_prepared(parts, roots, 3, want_grad=False, want_joint=True)[4].numpy(),
                               whole.logp_joint.numpy(), rtol=1e-12)
    assert len(eng.run_many(corpus, roots, 3, want_grad=False)) == 4
    for kw in (dict(approx_inference=True), dict(approx_beliefs=True), dict(want_marg=False)):
        with pytest.raises(ValueError):
            eng.run(corpus, roots, 3, want_grad=False, want_joint=True, **kw)


# ---------------------------------------------------------------------------------------------------- command line
N_SENT = 140


def _run_cli(argv):
    from macaronicusermodeling_b200 import engine, train_cli
    import test_predict_shard_host as sh

    class Kernels(JointKernels, sh.FormatKernels):
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


def test_cli_joint_file_one_rank_equals_two_ranks_and_pred_dist_do_not_move(tmp_path, capsys):
    from predict_cases import write_case
    base = write_case(tmp_path, synth.make_model(64, 16, seed=5), N_SENT, seed=3)
    plain, one, two = tmp_path / 'plain', tmp_path / 'one', tmp_path / 'two'
    for d in (plain, one, two):
        d.mkdir()
    _run_cli(base + ['--save_predictions', str(plain / 'out.pred')])
    out_plain = capsys.readouterr().out
    _run_cli(base + ['--joint_likelihood', '--save_predictions', str(one / 'out.pred')])
    out_joint = capsys.readouterr().out
    assert out_joint.startswith(out_plain)
    tail = out_joint[len(out_plain):].strip().split()
    assert tail[:3] == ['prediction', 'joint', 'log-likelihood:']
    port = 30700 + 2 * (os.getpid() % 1000)
    mp.spawn(_worker, args=(2, port, base + ['--joint_likelihood', '--save_predictions', str(two / 'out.pred')]), nprocs=2,
             join=True)
    for name in ('out.pred', 'out.pred.dist'):
        assert _read(plain / name) == _read(one / name) == _read(two / name), name
    assert _read(one / 'out.pred.joint') == _read(two / 'out.pred.joint')
    assert sorted(os.listdir(two)) == ['out.pred', 'out.pred.dist', 'out.pred.joint']
    lines = _read(one / 'out.pred.joint').decode().splitlines()
    assert len(lines) == N_SENT
    ids, joint, marg = zip(*(l.split('\t') for l in lines))
    assert [int(x) for x in ids] == list(range(N_SENT))
    joint, marg = np.array(joint, dtype=float), np.array(marg, dtype=float)
    assert float(tail[3]) == pytest.approx(joint.mean(), rel=1e-12)
    assert np.isfinite(joint).all() and (joint <= 0).all() and not np.array_equal(joint, marg)
