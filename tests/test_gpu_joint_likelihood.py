"""GPU tier of the joint log-likelihood (K9 mlbp_joint_logp, Engine.run want_joint, train_cli --joint_likelihood):
* K9 through the C ABI on hand-built rows against NumPy float64 (odd V, misaligned row bases, zeros, sentences without pairs,
  refused calls that leave their buffers untouched);
* trees against brute-force enumeration, one-token sentences against logp_sent;
* loopy sentences against the float64 reference (tests/bethe_oracle.py), up to V = 10 000 in the flat and trained regimes;
* grad / logp / beliefs / top1 / rank bit-identical with want_joint on and off, the CLI's .pred / .dist bytes unchanged by
  --joint_likelihood, and two torchrun ranks writing the .joint of one (when the box has two GPUs)."""
import ctypes
import os
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)

import joint_checks as jc  # noqa: E402
from macaronicusermodeling_b200 import _lib, build, synth, train_cli  # noqa: E402
from macaronicusermodeling_b200.engine import Corpus, Engine  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module', autouse=True)
def _built():
    build.build()
    torch.cuda.set_device(0)


# ------------------------------------------------------------------------------------------------------------ kernel level
SENTINEL = 12345.5


def _p(t, byte_off=0):
    return ctypes.c_void_p(t.data_ptr() + byte_off) if t is not None else None


def _case(V, ld, n_sent, seed):
    """hand-built rows: positive messages of mixed magnitude with zeros, pairs per sentence 0..4"""
    rng = np.random.default_rng(seed)
    pairs_per = rng.integers(0, 5, size=n_sent)
    pairs_per[0] = 0
    vars_per = rng.integers(1, 5, size=n_sent)
    var_off = np.concatenate([[0], np.cumsum(vars_per)]).astype(np.int32)
    fac_off = np.concatenate([[0], np.cumsum(pairs_per)]).astype(np.int32)
    nv, npair = int(var_off[-1]), int(fac_off[-1])
    labels = rng.integers(0, V, size=nv).astype(np.int32)
    s_of = np.repeat(np.arange(n_sent), pairs_per)
    v0 = np.array([var_off[s] + rng.integers(0, vars_per[s]) for s in s_of], dtype=np.int32)
    v1 = np.array([var_off[s] + rng.integers(0, vars_per[s]) for s in s_of], dtype=np.int32)
    n_a, n_d = 2 * npair + 3, 2 * npair + 4
    msg = rng.random((n_a, V)) * np.exp(rng.normal(0, 2, size=(n_a, V)))
    msg[:, rng.integers(0, V, size=3)] = 0.0                                       # zero entries (a label slot among them)
    msg[0, labels[v0[0]] if npair else 0] = 0.0
    hi = msg.astype(np.float16)
    lo = (msg - hi.astype(np.float64)).astype(np.float16)
    A_hi, A_lo = np.zeros((n_a, ld), np.float16), np.zeros((n_a, ld), np.float16)
    A_hi[:, :V], A_lo[:, :V] = hi, lo
    A_hi[:, V:] = np.float16(np.nan)                                               # the padding must never be read
    Dm = np.full((n_d, ld), np.nan, np.float32)
    Dm[:, :V] = (rng.random((n_d, V)) * np.exp(rng.normal(0, 2, size=(n_d, V))) + 1e-3).astype(np.float32)
    Dm[0, :V] = 1.0
    c_row = rng.permutation(n_a)[:npair].astype(np.int32)
    r_row = rng.permutation(n_a)[:npair].astype(np.int32)
    m0 = rng.integers(-1, n_d, size=npair).astype(np.int32)
    m1 = rng.integers(-1, n_d, size=npair).astype(np.int32)
    gap1 = rng.integers(0, 2, size=npair).astype(np.int32)
    stats = np.zeros((max(npair, 1), 3))
    stats[:npair, 0] = rng.random(npair) * 10.0 ** rng.integers(-3, 4, size=npair) + 1e-3
    pmi = rng.normal(0, 1, size=(V, ld)).astype(np.float32)
    w1 = rng.normal(0, 1, size=(V, ld)).astype(np.float32)
    logp_var = np.log(rng.random(nv) * 0.9 + 0.05)
    if n_sent > 2:
        logp_var[var_off[2]] = -99.99                                              # a label of belief 0: -inf
    return dict(var_off=var_off, fac_off=fac_off, labels=labels, v0=v0, v1=v1, A_hi=A_hi, A_lo=A_lo, D=Dm, c_row=c_row,
                r_row=r_row, m0=m0, m1=m1, gap1=gap1, stats=stats, pmi=pmi, w1=w1, logp_var=logp_var, V=V, ld=ld,
                theta=np.array([0.7, -0.4, 0.2]), zlog2=-17)


def _numpy_joint(c):
    V = c['V']
    H = c['A_hi'][:, :V].astype(np.float32)
    L = c['A_lo'][:, :V].astype(np.float32)
    Dm = c['D'][:, :V]
    th = c['theta']
    npair = int(c['fac_off'][-1])
    term = np.zeros(npair)
    with np.errstate(divide='ignore', invalid='ignore'):
        for f in range(npair):
            y0, y1 = c['labels'][c['v0'][f]], c['labels'][c['v1'][f]]
            mu0, mu1 = Dm[max(c['m0'][f], 0)].astype(np.float64), Dm[max(c['m1'][f], 0)].astype(np.float64)
            o0 = ((H[c['c_row'][f]] + L[c['c_row'][f]]).astype(np.float64) * mu0).sum()
            o1 = ((H[c['r_row'][f]] + L[c['r_row'][f]]).astype(np.float64) * mu1).sum()
            log_t = th[0] * float(c['pmi'][y0, y1]) + th[2] + (th[1] * float(c['w1'][y0, y1]) if c['gap1'][f] else 0.0)
            log_z = np.log(c['stats'][f, 0]) - c['zlog2'] * np.log(2.0)
            term[f] = log_t - log_z + np.log(o0) + np.log(o1) - np.log(mu0[y0]) - np.log(mu1[y1])
    out = []
    for s in range(len(c['var_off']) - 1):
        lv = c['logp_var'][c['var_off'][s]:c['var_off'][s + 1]]
        out.append(-np.inf if (lv == -99.99).any() else lv.sum() + term[c['fac_off'][s]:c['fac_off'][s + 1]].sum())
    return np.array(out), term


def _call(c, shift=0, **over):
    """mlbp_joint_logp on device copies of case c; shift > 0 offsets every row base by `shift` elements (misaligned)"""
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    V, ld = c['V'], c['ld']
    g = {k: dev(c[k]) for k in ('var_off', 'fac_off', 'labels', 'v0', 'v1', 'c_row', 'r_row', 'm0', 'm1', 'gap1', 'stats', 'pmi',
                                 'w1', 'logp_var')}
    pad = lambda a, dt: torch.cat([torch.zeros(shift, dtype=dt), torch.from_numpy(a.reshape(-1))]).cuda()
    A_hi, A_lo, D = pad(c['A_hi'], torch.float16), pad(c['A_lo'], torch.float16), pad(c['D'], torch.float32)
    n_sent, npair = len(c['var_off']) - 1, int(c['fac_off'][-1])
    out = torch.full((max(n_sent, 1),), SENTINEL, dtype=torch.float64, device='cuda')
    ws = torch.full((max(npair, 1),), SENTINEL, dtype=torch.float64, device='cuda')
    th = np.ascontiguousarray(over.pop('theta', c['theta']), dtype=np.float64)
    args = dict(n_sent=n_sent, n_pairs=npair, V=V, ldv=ld, ldf=ld, zlog2=c['zlog2'], A_hi=_p(A_hi, 2 * shift),
                A_lo=_p(A_lo, 2 * shift), D=_p(D, 4 * shift), c_row=_p(g['c_row']))
    args.update(over)
    rc = _lib.load().mlbp_joint_logp(args['n_sent'], args['n_pairs'], _p(g['var_off']), _p(g['fac_off']), _p(g['logp_var']),
                                     args['c_row'], _p(g['r_row']), _p(g['m0']), _p(g['m1']), _p(g['v0']), _p(g['v1']),
                                     _p(g['labels']), _p(g['gap1']), _p(g['stats']), args['A_hi'], args['A_lo'], args['D'],
                                     args['ldv'], args['V'], _p(g['pmi']), _p(g['w1']), args['ldf'],
                                     th.ctypes.data_as(ctypes.c_void_p), args['zlog2'], _p(ws), _p(out),
                                     ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return rc, out.cpu().numpy()[:n_sent], ws.cpu().numpy()[:npair]


# Tolerance per factor: each O dot sums fp32 products (each rounded once, 2^-24 relative; hi + lo of a hand-built pair can round
# once more, 2^-24) of non-negative terms in float64, so log O is within ~2^-23 relative of exact; two dots per factor, and the
# float64 logs and sums are ~1e-15.  4 x 2^-23 per factor, with room.
PAIR_TOL = 4 * 2.0 ** -23


@pytest.mark.parametrize('V,ld,shift', [(203, 256, 0), (10000, 10048, 0), (67, 67, 0), (1001, 1024, 3), (9, 64, 1)])
def test_k9_against_numpy_float64(V, ld, shift):
    c = _case(V, ld, 40, seed=V + shift)
    rc, got, term = _call(c, shift)
    assert rc == 0, _lib.load().mlbp_last_error()
    want, want_term = _numpy_joint(c)
    npp = np.diff(c['fac_off'])
    fin = np.isfinite(want)
    assert (~fin).any() and (got[~fin] == want[~fin]).all()                    # the -99.99 sentence
    # (+ 1e-14: the sentence's logp_var are summed in another order than NumPy's)
    assert (np.abs(got[fin] - want[fin]) <= (npp[fin] * PAIR_TOL + 1e-14) * np.maximum(1.0, np.abs(want[fin]))).all()
    ok = np.isfinite(want_term)
    assert np.allclose(term[ok], want_term[ok], rtol=PAIR_TOL, atol=PAIR_TOL)
    assert npp[0] == 0 and got[0] == pytest.approx(c['logp_var'][c['var_off'][0]:c['var_off'][1]].sum(), rel=1e-15)
    # deterministic
    rc2, got2, _ = _call(c, shift)
    assert rc2 == 0 and np.array_equal(got, got2, equal_nan=True)


def test_k9_refuses_bad_arguments_and_launches_nothing():
    c = _case(67, 128, 12, seed=5)
    lib = _lib.load()
    for over in (dict(V=0), dict(ldv=60), dict(ldf=60), dict(n_pairs=-1), dict(n_sent=-1), dict(zlog2=5000),
                 dict(c_row=None), dict(A_hi=None), dict(theta=[np.inf, 0.0, 0.0]), dict(theta=[0.0, np.nan, 0.0])):
        rc, out, ws = _call(c, **over)
        assert rc == 1, over
        assert b'joint_logp' in lib.mlbp_last_error()
        assert (out == SENTINEL).all() and (ws == SENTINEL).all(), over
    rc, out, _ = _call(c, n_sent=0, n_pairs=0)
    assert rc == 0


# ------------------------------------------------------------------------------------------------------------ engine level
@pytest.mark.parametrize('V', [60, 67])
def test_trees_against_brute_force(V):
    model = synth.make_model(V, 12, seed=4)
    sents = jc.tree_sentences(model) + [synth.sentence_to_arrays(synth.make_sentence(model, 'gpg', seed=3, n_history=2))]
    roots = synth.draw_roots(sents, 3, seed=5)
    r, _ = jc.engine_joint(Engine(model), sents, roots, jc.THETA_EE, jc.THETA_ED)
    lj = r.logp_joint.cpu().numpy()
    for i, s in enumerate(sents[:4]):
        want = jc.brute_force_joint(model, s, jc.THETA_EE, jc.THETA_ED)
        assert abs(lj[i] - want) < jc.joint_tol(1, V), (i, lj[i], want)
    assert lj[4] == r.logp.cpu().numpy()[4]                                        # one predicted token: logp_sent exactly


def _loopy(model, sents, roots, te, td, **eng_kw):
    r, corpus = jc.engine_joint(Engine(model, **eng_kw), sents, roots, te, td)
    want = jc.oracle_joints(model, sents, roots, te, td)
    err = np.abs(r.logp_joint.cpu().numpy() - want)
    tol = jc.joint_tol(np.diff(corpus.pair_off), model['V'])
    assert (err < tol).all(), (err, tol)
    return float(err.max()), float((err / np.diff(corpus.pair_off)).max())


@pytest.mark.parametrize('V', [67, 203, 1001])
def test_loopy_against_oracle(V):
    model = synth.make_model(V, 24, seed=V)
    sents = [synth.make_corpus(model, 1, k=k, g=k % 3, seed=100 + k)[0] for k in range(3, 21)]
    roots = synth.draw_roots(sents, 3, seed=7)
    worst, per_pair = _loopy(model, sents, roots, jc.THETA_EE, jc.THETA_ED)
    print('V = %d, k = 3..20: worst |joint - oracle| %.2e (%.2e per factor)' % (V, worst, per_pair))


def _m64(model):
    return {k: (np.asarray(v, dtype=np.float64) if hasattr(v, 'dtype') else v) for k, v in model.items()}


@pytest.mark.parametrize('regime', ['flat', 'trained'])
def test_v10000_against_oracle(regime):
    """C3 size with the default one-pass rows, in the flat regime and the regime bench.py's SGD reaches (test_gpu_gates.py)"""
    model = synth.make_model(10000, 2000, seed=1234, dtype=np.float32)
    sents = synth.make_corpus(model, 3, k=20, g=0, seed=4242)
    roots = synth.draw_roots(sents, 3, seed=11)
    te, td = (([0.8, 0.5, -0.3], [1.0, -0.6, 0.5, 0.3, 0.4, -0.2]) if regime == 'flat' else
              ([-0.003, 0.049, -0.3], [0.101, -0.047, 7.534, 0.3, 0.4, -0.2]))
    worst, per_pair = _loopy(_m64(model), sents, roots, te, td)
    print('V = 10 000 %s: worst |joint - oracle| %.2e (%.2e per factor)' % (regime, worst, per_pair))


def test_three_pass_message_rows_against_oracle():
    model = synth.make_model(1001, 24, seed=9)
    sents = synth.make_corpus(model, 6, k=8, g=1, seed=31)
    roots = synth.draw_roots(sents, 3, seed=2)
    worst, _ = _loopy(model, sents, roots, jc.THETA_EE, jc.THETA_ED, msg_passes=3)
    print('msg_passes = 3: worst %.2e' % worst)


@pytest.mark.parametrize('V,want_grad', [(1001, True), (1001, False), (10000, True), (10000, False)])
def test_nothing_else_moves(V, want_grad):
    model = synth.make_model(V, 64, seed=3)
    sents = synth.make_corpus(model, 24, k=10, g=2, seed=5)
    corpus = Corpus(sents)
    roots = corpus.roots_from_positions(synth.draw_roots(sents, 3, seed=6))
    out = []
    for joint in (False, True):
        eng = Engine(model)
        eng.set_theta(jc.THETA_EE, jc.THETA_ED, with_grad=True)
        out.append(eng.run(corpus, roots, 3, want_grad=want_grad, want_marg=True, want_beliefs=True, want_joint=joint))
    for name in ('grad', 'logp', 'logp_var', 'top1', 'rank'):
        assert torch.equal(getattr(out[0], name), getattr(out[1], name)), name
    assert torch.equal(out[0].beliefs[:, :V], out[1].beliefs[:, :V])         # (the row padding is never written)
    assert torch.isfinite(out[1].logp_joint).all()


def test_approximate_modes_are_refused():
    model = synth.make_model(203, 24, seed=1)
    sents = synth.make_corpus(model, 2, k=4, g=1, seed=2)
    with pytest.raises(ValueError):
        jc.engine_joint(Engine(model), sents, synth.draw_roots(sents, 3, seed=1), jc.THETA_EE, jc.THETA_ED,
                        approx_inference=True)


# ------------------------------------------------------------------------------------------------------------ command line
def _cli(argv, capsys):
    assert train_cli.main(argv) == 0
    return capsys.readouterr().out


def _read(p):
    with open(p, 'rb') as f:
        return f.read()


def test_cli_pred_and_dist_do_not_move_and_joint_file(tmp_path, capsys):
    from predict_cases import write_case
    base = write_case(tmp_path, synth.make_model(2304, 48, seed=5), 80, seed=3)
    (tmp_path / 'a').mkdir(); (tmp_path / 'b').mkdir()
    out_a = _cli(base + ['--save_predictions', str(tmp_path / 'a' / 'out.pred')], capsys)
    out_b = _cli(base + ['--joint_likelihood', '--save_predictions', str(tmp_path / 'b' / 'out.pred')], capsys)
    for name in ('out.pred', 'out.pred.dist'):
        assert _read(tmp_path / 'a' / name) == _read(tmp_path / 'b' / name), name
    assert out_b.startswith(out_a) and 'prediction joint log-likelihood:' in out_b[len(out_a):]
    lines = _read(tmp_path / 'b' / 'out.pred.joint').decode().splitlines()
    assert len(lines) == 80 and all(len(l.split('\t')) == 3 for l in lines)


def test_two_rank_torchrun_joint_equals_one_rank(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs for a 2-rank torchrun prediction; this box has %d' % torch.cuda.device_count())
    import subprocess
    from predict_cases import write_case
    base = write_case(tmp_path, synth.make_model(2304, 48, seed=5), 150, seed=4)
    (tmp_path / 'one').mkdir(); (tmp_path / 'two').mkdir()
    assert train_cli.main(base + ['--joint_likelihood', '--save_predictions', str(tmp_path / 'one' / 'out.pred')]) == 0
    env = dict(os.environ, PYTHONPATH=os.path.dirname(HERE))
    subprocess.check_call([sys.executable, '-m', 'torch.distributed.run', '--standalone', '--nproc_per_node', '2', '-m',
                           'macaronicusermodeling_b200.train_cli'] + base +
                          ['--joint_likelihood', '--save_predictions', str(tmp_path / 'two' / 'out.pred')], env=env)
    for name in ('out.pred', 'out.pred.dist', 'out.pred.joint'):
        assert _read(tmp_path / 'one' / name) == _read(tmp_path / 'two' / name), name
