"""GPU tier of max-product decoding (K10 mlbp_factor_to_var_maxprod, K11 mlbp_assignment_score, Engine.run max_product,
train_cli --map_decode):
* K10 through the C ABI against NumPy float64 max-times: all four tables, flat / peaked / zero rows, misaligned row bases,
  garbage in the padding of A and of the feature planes, sentinel-filled D, the output bound, bit-identity across row slicings,
  refused calls that leave their sentinels;
* K11 through the C ABI against NumPy on labels and random assignments, and its refusal of an index outside [0, V);
* the engine's decoding against the float64 reference (tests/maxprod_oracle.py) up to V = 10 000, trees against brute force,
  sum-product outputs bit-identical around a max-product run, and a --map_decode run whose words are the reference's."""
import ctypes
import os
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)

import map_checks as mc  # noqa: E402
import maxprod_oracle as mo  # noqa: E402
from macaronicusermodeling_b200 import _lib, build, synth, train_cli  # noqa: E402
from macaronicusermodeling_b200.engine import Corpus, Engine  # noqa: E402

pytestmark = pytest.mark.gpu

SENTINEL = 12345.5
U32 = 2.0 ** -24


@pytest.fixture(scope='module', autouse=True)
def _built():
    build.build()
    torch.cuda.set_device(0)


def _p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


# ------------------------------------------------------------------------------------------------------------ K10
def _k10_case(V, n_rows, seed):
    """A rows (flat, peaked, zero) as fp16 hi / lo with garbage in the padding, feature planes with garbage in the padding"""
    rng = np.random.default_rng(seed)
    ldv, ldf = (V + 63) // 64 * 64 + 64, (V + 3) // 4 * 4 + 4
    msg = rng.random((n_rows, V)) + 0.05                                    # flat
    for r in range(1, n_rows, 3):                                           # peaked: a few words carry most of the mass
        msg[r] = msg[r] ** 8
        msg[r, rng.integers(0, V, size=3)] = 50.0 * V
    msg[2] = 0.0                                                            # a zero row
    msg[min(4, n_rows - 1), : V // 2] = 0.0
    msg *= 2.0 ** 14 / np.maximum(msg.sum(axis=1, keepdims=True), 1e-300)
    hi = msg.astype(np.float16)
    lo = (msg - hi.astype(np.float64)).astype(np.float16)
    A_hi = np.full((n_rows + 3, ldv), 60000.0, np.float16)                  # the padding is not initialised
    A_lo = np.full((n_rows + 3, ldv), 1000.0, np.float16)
    A_hi[1:1 + n_rows, :V], A_lo[1:1 + n_rows, :V] = hi, lo
    pmi = np.full((V, ldf), 40.0, np.float32)
    w1 = np.full((V, ldf), -40.0, np.float32)
    pmi[:, :V] = rng.random((V, V), dtype=np.float32)
    w1[:, :V] = rng.random((V, V), dtype=np.float32)
    pmi[:, :V][rng.random((V, V)) < 0.3] = 0.0                              # sparse planes: many exactly equal entries
    return dict(V=V, ldv=ldv, ldf=ldf, n_rows=n_rows, a=hi.astype(np.float64) + lo.astype(np.float64), A_hi=A_hi, A_lo=A_lo,
                pmi=pmi, w1=w1, theta=np.array([0.9, -0.6, 0.3]), centre=1)


def _table(c, t):
    """T'[n, k] of message table t in float64"""
    V, th = c['V'], c['theta']
    P, W = c['pmi'][:, :V].astype(np.float64), c['w1'][:, :V].astype(np.float64)
    z = th[0] * P + th[2] - c['centre'] * np.log(2.0) + (th[1] * W if t in (2, 3) else 0.0)
    T = np.exp(z)
    return T.T if t in (1, 3) else T


def _k10(c, t, rows=None, D=None, d_shift=3, ldd=None, **over):
    """launch K10 on A rows [1 + r0, 1 + r1) into D rows d_shift + r0 .. (sentinel-filled D unless given)"""
    dev = torch.device('cuda')
    r0, r1 = rows or (0, c['n_rows'])
    ldd = ldd or c['ldv'] + 8
    if D is None:
        D = torch.full((c['n_rows'] + d_shift + 2, ldd), SENTINEL, dtype=torch.float32, device=dev)
    A_hi, A_lo = torch.from_numpy(c['A_hi']).to(dev), torch.from_numpy(c['A_lo']).to(dev)
    pmi, w1 = torch.from_numpy(c['pmi']).to(dev), torch.from_numpy(c['w1']).to(dev)
    th = np.ascontiguousarray(over.pop('theta', c['theta']), dtype=np.float64)
    args = dict(A_hi=_p(A_hi), A_lo=_p(A_lo), a_rows_total=c['n_rows'] + 3, a_row0=1 + r0, n_rows=r1 - r0, table=t, pmi=_p(pmi),
                pmi_w1=_p(w1), V=c['V'], ldv=c['ldv'], ldf=c['ldf'], theta=th.ctypes.data_as(ctypes.c_void_p),
                centre=c['centre'], D=_p(D), d_row0=d_shift + r0, ldd=ldd)
    args.update(over)
    _lib.call('mlbp_factor_to_var_maxprod', *args.values(), _stream())
    torch.cuda.synchronize()
    return D


@pytest.mark.parametrize('V', [67, 203, 1001, 10000])
def test_k10_against_numpy_float64(V):
    n_rows = 6 if V == 10000 else 37
    c = _k10_case(V, n_rows, seed=V)
    a = c['a']
    amax = a.max(axis=1)
    for t in range(4):
        B = _table(c, t)
        want = mo.max_times(a / np.where(amax > 0, amax, 1.0)[:, None], B.T)
        D = _k10(c, t).cpu().numpy()
        got = D[3:3 + n_rows, :V].astype(np.float64)
        assert (D[:3] == SENTINEL).all() and (D[3 + n_rows:] == SENTINEL).all() and (D[:, V:] == SENTINEL).all(), t
        assert (got[2] == 0).all(), 'a zero row gives a zero D row'
        # expf (<= 2 ulp) and the (1 + lo) factor of exp_f2, the product and the division: <= 8 half-ulps, doubled
        np.testing.assert_allclose(got, want, rtol=16 * U32, atol=0, err_msg='table %d' % t)
        live = amax > 0
        assert (got[live] >= B.min() * (1 - 16 * U32)).all() and (got[live] <= B.max() * (1 + 16 * U32)).all(), t
        print('V = %d table %d: worst relative error %.2e' % (V, t, float((np.abs(got - want) / np.maximum(want, 1e-300)).max())))


def test_k10_is_bit_identical_across_row_slicings():
    c = _k10_case(1001, 300, seed=3)
    for t in range(4):
        whole = _k10(c, t)
        D = torch.full_like(whole, SENTINEL)
        for rows in ((0, 129), (129, 131), (131, 300)):                    # slices that cut through 128-row tiles
            _k10(c, t, rows=rows, D=D)
        assert torch.equal(whole, D), t
        D2 = torch.full_like(whole, SENTINEL)
        for rows in ((200, 300), (0, 1), (1, 200)):                       # another slicing, another launch order
            _k10(c, t, rows=rows, D=D2)
        assert torch.equal(whole, D2), t


def test_k10_refuses_bad_arguments_and_launches_nothing():
    c = _k10_case(203, 8, seed=5)
    D = torch.full((16, c['ldv'] + 8), SENTINEL, dtype=torch.float32, device='cuda')
    bad = [dict(A_hi=None), dict(pmi=None), dict(pmi_w1=None), dict(table=4), dict(table=-1), dict(V=0), dict(ldv=c['V'] - 1),
           dict(ldf=c['V'] - 1), dict(a_rows_total=8), dict(a_row0=5), dict(ldv=c['ldv'] - 4), dict(theta=[np.nan, 0, 0])]
    for over in bad:
        with pytest.raises(_lib.MlbpError):
            _k10(c, 0, D=D, **over)
        assert (D.cpu().numpy() == SENTINEL).all(), over
    _k10(c, 0, rows=(3, 3), D=D)                                            # n_rows == 0: a no-op
    assert (D.cpu().numpy() == SENTINEL).all()


# ------------------------------------------------------------------------------------------------------------ K11
def _k11(eng, corpus, x):
    dev = torch.device('cuda')
    m = eng.model
    c = lambda name: _p(corpus.dev(name, dev))
    xs = torch.from_numpy(np.ascontiguousarray(x, dtype=np.int32)).to(dev)
    out = torch.full((corpus.n_sent,), SENTINEL, dtype=torch.float64, device=dev)
    te, td = np.ascontiguousarray(eng.theta_ee), np.ascontiguousarray(eng.theta_ed)
    _lib.call('mlbp_assignment_score', corpus.n_sent, corpus.n_vars, len(corpus.giv_label), c('var_off'), _p(xs), c('var_de'),
              c('sp_off'), c('sp_en'), c('sp_feat'), c('sp_val'), c('giv_off'), c('giv_label'), c('giv_gap1'), c('pair_off'),
              c('pair_v0'), c('pair_v1'), c('pair_gap1'), _p(m.pmi), _p(m.w1), _p(m.edT), _p(m.pedT), eng.V, eng.ld,
              te.ctypes.data_as(ctypes.c_void_p), td.ctypes.data_as(ctypes.c_void_p), _p(out), _stream())
    return out.cpu().numpy()


def test_k11_against_numpy_and_refuses_out_of_range_indices():
    model = synth.make_model(1001, 40, seed=2, dtype=np.float32)
    sents = synth.make_corpus(model, 30, k=9, g=3, seed=4) + synth.make_corpus(model, 5, k=1, g=2, seed=5)
    corpus = Corpus(sents)
    eng = Engine(model)
    eng.set_theta(mc.THETA_EE, mc.THETA_ED)
    rng = np.random.default_rng(1)
    for x in (corpus.var_label, rng.integers(0, 1001, size=corpus.n_vars)):
        want = mo.assignment_scores(model, mc.THETA_EE, mc.THETA_ED, corpus, x)
        np.testing.assert_allclose(_k11(eng, corpus, x), want, rtol=1e-12, atol=1e-12)
    for bad in (-1, 1001):
        x = corpus.var_label.copy()
        x[7] = bad
        with pytest.raises(_lib.MlbpError):
            _k11(eng, corpus, x)


# ------------------------------------------------------------------------------------------------------------ engine
def _decode(model, sents, roots, te, td):
    r, corpus = mc.engine_decode(Engine(model), sents, roots, te, td)
    want = mc.oracle_decode(model, sents, roots, te, td)
    return mc.check_decode(r, corpus, model, want, te, td), r, corpus, want


def test_trees_against_brute_force():
    model = synth.make_model(203, 12, seed=4, dtype=np.float32)
    sents = [synth.sentence_to_arrays(synth.make_sentence(model, l, seed=11 + i, n_history=2)) for i, l in enumerate(mc.TREE_LAYOUTS)]
    r, corpus = mc.engine_decode(Engine(model), sents, synth.draw_roots(sents, 3, seed=5), mc.THETA_EE, mc.THETA_ED)
    top1, ms = r.top1.cpu().numpy(), r.map_score.cpu().numpy()
    for i, s in enumerate(sents):
        best, best_score, label_score = mc.brute_force(model, s, mc.THETA_EE, mc.THETA_ED)
        np.testing.assert_array_equal(top1[corpus.var_off[i]:corpus.var_off[i + 1]], best)
        assert ms[i] == pytest.approx(best_score, abs=1e-6)
        assert r.label_score.cpu().numpy()[i] == pytest.approx(label_score, abs=1e-6)


@pytest.mark.parametrize('V', [67, 203, 1001])
def test_loopy_against_oracle(V):
    model = synth.make_model(V, 24, seed=V, dtype=np.float32)
    sents = [synth.make_corpus(model, 1, k=k, g=k % 3, seed=100 + k)[0] for k in range(3, 21)]
    roots = synth.draw_roots(sents, 3, seed=7)
    excluded, r, corpus, _ = _decode(model, sents, roots, mc.THETA_EE, mc.THETA_ED)
    print('V = %d, k = 3..20: %d of %d variables excluded as near-ties' % (V, excluded, corpus.n_vars))


@pytest.mark.parametrize('regime', ['flat', 'trained'])
def test_v10000_against_oracle(regime):
    model = synth.make_model(10000, 2000, seed=1234, dtype=np.float32)
    sents = synth.make_corpus(model, 1, k=8, g=0, seed=4242) + synth.make_corpus(model, 1, k=5, g=1, seed=4243)
    roots = synth.draw_roots(sents, 3, seed=11)
    te, td = (([0.8, 0.5, -0.3], [1.0, -0.6, 0.5, 0.3, 0.4, -0.2]) if regime == 'flat' else
              ([-0.003, 0.049, -0.3], [0.101, -0.047, 7.534, 0.3, 0.4, -0.2]))
    excluded, r, corpus, _ = _decode(model, sents, roots, te, td)
    print('V = 10 000 %s: %d of %d variables excluded as near-ties' % (regime, excluded, corpus.n_vars))


@pytest.mark.parametrize('V', [1001, 10000])
def test_sum_product_outputs_are_bit_identical_around_a_max_product_run(V):
    model = synth.make_model(V, 64, seed=3)
    sents = synth.make_corpus(model, 24, k=10, g=2, seed=5)
    corpus = Corpus(sents)
    roots = corpus.roots_from_positions(synth.draw_roots(sents, 3, seed=6))
    eng = Engine(model)
    eng.set_theta(mc.THETA_EE, mc.THETA_ED, with_grad=True)
    runs = []
    for want_grad in (True, False):
        kw = dict(want_grad=want_grad, want_marg=True, want_beliefs=True)
        a = eng.run(corpus, roots, 3, **kw)
        flags = eng.pass_stats()
        m = eng.run(corpus, roots, 3, want_grad=False, want_beliefs=True, max_product=True)
        assert eng.pass_stats() == flags                                 # no flag word or counter moves
        b = eng.run(corpus, roots, 3, **kw)
        for name in ('grad', 'logp', 'logp_var', 'top1', 'rank'):
            assert torch.equal(getattr(a, name), getattr(b, name)), name
        assert torch.equal(a.beliefs[:, :V], b.beliefs[:, :V])
        runs.append(m)
    assert torch.equal(runs[0].top1, runs[1].top1) and torch.equal(runs[0].map_score, runs[1].map_score)


# ------------------------------------------------------------------------------------------------------------ command line
def test_cli_map_words_are_the_oracle_decoding(tmp_path, capsys):
    import json
    from predict_cases import THETA_ED, THETA_EE, write_case
    model = synth.make_model(203, 24, seed=5)
    base = write_case(tmp_path, model, 40, seed=3)
    assert train_cli.main(base + ['--map_decode', '--save_predictions', str(tmp_path / 'out.pred')]) == 0
    out = capsys.readouterr().out
    assert 'prediction MAP token accuracy:' in out and 'prediction MAP sentence accuracy:' in out
    lines = open(tmp_path / 'out.pred.map').read().splitlines()
    assert len(lines) == 40
    # the command line draws each unit's roots from random.Random(seed + 1) in unit order (train_cli.predict)
    import random
    rng = random.Random(1234 + 1)
    raw = [json.loads(l) for l in open(base[1])]
    en = [l.strip() for l in open(base[3])]
    de = [l.strip() for l in open(base[5])]
    en2id, de2id = dict((w, i) for i, w in enumerate(en)), dict((w, i) for i, w in enumerate(de))
    sents = [synth.sentence_to_arrays(r, en2id, de2id, history=True, session_history=True) for r in raw]
    m32 = {k: (np.asarray(v, dtype=np.float32) if hasattr(v, 'dtype') else v) for k, v in model.items()}
    excluded = 0
    for _, idx in train_cli.prediction_units(len(sents)):
        c = Corpus([sents[i] for i in idx])
        roots = train_cli.draw_roots(c, 3, rng)
        roots_pos = [[int(c.var_pos[c.var_off[s] + j]) for j in roots[s]] for s in range(c.n_sent)]
        want = mc.oracle_decode(m32, [sents[i] for i in idx], roots_pos, THETA_EE, THETA_ED)
        for s, i in enumerate(idx):
            words = lines[i].split('\t')[1].split(' ')
            mm, dec = want[s]
            srt = np.sort(mm, axis=1)
            tie = srt[:, -2] >= srt[:, -1] * (1 - 4 * mc.marg_tol(len(dec)))
            excluded += int(tie.sum())
            assert [w for w, t in zip(words, tie) if not t] == [en[e] for e, t in zip(dec, tie) if not t], i
    print('--map_decode at V = 203: %d near-ties excluded' % excluded)
