"""GPU tier of the pseudo-likelihood (K13 mlbp_pseudo_likelihood, Engine.pseudo_likelihood, Trainer(objective='pl')):
* K13 through the C ABI against the plane-level reference (tests/pl_oracle.py) fed the same U rows and planes -- top1 and rank
  equal, logp_var within a few ulp, gradients within 1e-6 of their terms' scale -- and against the float64 model-level
  reference -- logp_var within the error budget of include/mlbp.h, gradients within 1e-4 relative (2e-6 absolute floor) -- at
  V = 67, 1 001 and 10 000, k = 1, 2, 3, 20 and 49, with and without given tokens, on the fp32 and the fp64 product paths, with
  garbage in the padding and sentinels in everything the kernel must not write;
* k = 1: logp_var equals BP's (both exact); a sentence with a label outside [0, V) gets NaN outputs, its neighbours do not;
* refused calls leave their sentinels; determinism, batch and micro-batch invariance; sum-product bit-identical around a call;
* one objective='pl' SGD step against the model-level reference."""
import ctypes
import os
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)

import pl_oracle  # noqa: E402
from macaronicusermodeling_b200 import _lib, build, synth  # noqa: E402
from macaronicusermodeling_b200.engine import Corpus, Engine  # noqa: E402

pytestmark = pytest.mark.gpu

SENTINEL = 12345.5
INT_MAX = 2 ** 31 - 1
THETA = ([0.6, -0.4, 0.1], [0.9, -0.5, 0.4, 0.3, 0.3, -0.1])


@pytest.fixture(scope='module', autouse=True)
def _built():
    build.build()
    torch.cuda.set_device(0)


def _p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _i32(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).cuda()


def _engine(V, seed=1):
    model = synth.make_model(V, 64, seed=seed, dtype=np.float32)
    eng = Engine(model)
    eng.set_theta(THETA[0], THETA[1], with_grad=True)
    return model, eng


def _corpus(model, ks, seed, given=(0, 1, 2)):
    sents = []
    for i, k in enumerate(ks):
        sents += synth.make_corpus(model, 1, k=k, g=given[i % len(given)], seed=seed + i)
    return sents, Corpus(sents)


class _DevRows(object):
    """plane p of a device tensor, read row by row for the reference (a host copy of 20 planes at V = 10 000 is 4 GB)"""

    def __init__(self, t):
        self.t = t

    def __getitem__(self, idx):
        return self.t[idx[0]][idx[1]].cpu().numpy()


class Case(object):
    """a batch through the C ABI: K1's rows and the engine's planes and features, copied with garbage in a padding of our own
    (V < 10 000; at 10 000 the engine's own buffers), sentinel-filled outputs"""

    def __init__(self, eng, model, corpus, own_padding=True):
        self.eng, self.model, self.c, self.V = eng, model, corpus, eng.V
        V = self.V
        self.ld = eng.ld + 16 if own_padding else eng.ld
        ld = self.ld
        rng = np.random.default_rng(V + corpus.n_vars)
        U = eng.unary_rows(corpus)[0][:, :V].cpu().numpy()
        self.U_host = U

        def pad(a, dtype, fill):
            out = np.full((a.shape[0], ld), fill, dtype=dtype)
            out[:, V:] = rng.choice(np.array([np.inf, -1e30, 7.0, np.nan]).astype(dtype), size=(a.shape[0], ld - V))
            out[:, :V] = a[:, :V]
            return torch.from_numpy(out).cuda()

        self.U = pad(U, np.float32, np.nan)
        m = eng.model
        if own_padding:
            P = np.full((20, V, ld), np.float16(np.nan), dtype=np.float16)
            P[:, :, :V] = eng.planes[:20, :, :V].cpu().numpy()
            self.planes_host = [P[p] for p in range(20)]
            self.planes = torch.from_numpy(P).cuda()
            self.feat = [pad(t.cpu().numpy(), np.float32, np.nan) for t in (m.pmi, m.w1, m.edT, m.pedT)]
        else:
            self.planes, self.feat = eng.planes, [m.pmi, m.w1, m.edT, m.pedT]
            self.planes_host = [_DevRows(eng.planes[p]) for p in range(20)]
        self.fhost = [np.asarray(model['pmi']), np.asarray(model['pmi_w1']), np.asarray(model['ed']).T, np.asarray(model['ped']).T]
        self.dev = dict((n, _i32(getattr(corpus, n) if len(getattr(corpus, n)) else [0])) for n in Corpus.FIELDS if n != 'sp_val')
        self.dev['sp_val'] = torch.from_numpy(np.ascontiguousarray(corpus.sp_val if len(corpus.sp_val) else [0.0],
                                                                   dtype=np.float32)).cuda()

    def run(self, range_log2, want_grad=True, labels=None, **over):
        nv, ld = self.c.n_vars, self.ld
        out = dict(lp=torch.full((nv + 1,), SENTINEL, dtype=torch.float64, device='cuda'),
                   t1=torch.full((nv + 1,), -7, dtype=torch.int32, device='cuda'),
                   rk=torch.full((nv + 1,), -7, dtype=torch.int32, device='cuda'),
                   g=torch.full((nv + 1, 9), SENTINEL, dtype=torch.float64, device='cuda'),
                   b=torch.full((nv + 1, ld), SENTINEL, dtype=torch.float32, device='cuda'))
        d = self.dev
        lab = d['var_label'] if labels is None else _i32(labels)
        args = dict(n_sent=self.c.n_sent, max_k=int(np.diff(self.c.var_off).max()), n_vars=nv, var_off=_p(d['var_off']),
                    pair_off=_p(d['pair_off']), v0=_p(d['pair_v0']), v1=_p(d['pair_v1']), gap1=_p(d['pair_gap1']),
                    var_label=_p(lab), var_de=_p(d['var_de']), sp_off=_p(d['sp_off']), sp_en=_p(d['sp_en']),
                    sp_feat=_p(d['sp_feat']), sp_val=_p(d['sp_val']), giv_off=_p(d['giv_off']), giv_label=_p(d['giv_label']),
                    giv_gap1=_p(d['giv_gap1']), U=_p(self.U), planes=_p(self.planes), ps=self.V * ld, ldv=ld, V=self.V,
                    scale_exp=self.eng.scale_exp, colsums=_p(self.eng.colsums), pmi=_p(self.feat[0]), w1=_p(self.feat[1]),
                    edT=_p(self.feat[2]), pedT=_p(self.feat[3]), ldf=ld, range_log2=range_log2, logp_var=_p(out['lp']),
                    top1=_p(out['t1']), rank=_p(out['rk']), grad=_p(out['g']) if want_grad else None, beliefs=_p(out['b']))
        args.update(over)
        rc = _lib.load().mlbp_pseudo_likelihood(*args.values(), _stream())
        torch.cuda.synchronize()
        return rc, dict((k, v.cpu().numpy()) for k, v in out.items())

    def check(self, f64):
        rc, o = self.run(200.0 if f64 else 0.0)
        assert rc == 0, _lib.load().mlbp_last_error()
        V, nv = self.V, self.c.n_vars
        assert o['lp'][-1] == SENTINEL and o['t1'][-1] == -7 and o['rk'][-1] == -7 and (o['g'][-1] == SENTINEL).all()
        assert (o['b'][-1] == SENTINEL).all() and (o['b'][:, V:] == SENTINEL).all()
        lp, t1, rk, g, rows, scale = pl_oracle.planes_reference(self.c, self.U_host, self.planes_host, self.eng.colsums.cpu().numpy(),
                                                                self.eng.scale_exp, *self.fhost, f64)
        np.testing.assert_array_equal(o['t1'][:-1], t1)
        np.testing.assert_array_equal(o['rk'][:-1], rk)
        np.testing.assert_allclose(o['lp'][:-1], lp, rtol=4e-15, atol=4e-16)
        np.testing.assert_array_equal(o['b'][:-1, :V], rows)
        assert (np.abs(o['g'][:-1] - g) <= 1e-6 * scale + 1e-12).all(), np.abs(o['g'][:-1] - g).max()
        assert (o['g'][:-1][:, [2, 8]] == 0).all()
        # the float64 model.  Each factor of q carries at most ~2^-22 relative error (the 22-bit hi + lo planes, K2's ~1 ulp
        # entries, the fp32 products), K1's row about two factors' worth, so log q(y) / Z is off by at most 2 max_x |delta(x)|:
        # 4 (deg + g + 2) 2^-22.  The gradient is held to the project's contract.
        m_lp, m_g, _ = pl_oracle.model_reference(self.c, self.model, *THETA)
        deg = np.repeat(np.diff(self.c.var_off) - 1, np.diff(self.c.var_off))
        budget = (deg + np.diff(self.c.giv_off) + 2) * 2.0 ** -22
        err = np.abs(o['lp'][:-1] - m_lp)
        worst = float((err / budget).max())
        gworst = float((np.abs(o['g'][:-1] - m_g) / (1e-4 * np.abs(m_g) + 2e-6)).max())
        print('V = %d %s: logp_var error <= %.2f x (deg + g + 2) 2^-22 (max %.2e); gradient error <= %.3f of the contract' % (
            V, 'fp64' if f64 else 'fp32', worst, float(err.max()), gworst))
        assert worst <= 4.0, worst
        np.testing.assert_allclose(o['g'][:-1], m_g, rtol=1e-4, atol=2e-6)
        return o


@pytest.mark.parametrize('V', [67, 1001, 10000])
@pytest.mark.parametrize('f64', [False, True], ids=['fp32', 'fp64'])
def test_k13_against_the_references(V, f64):
    model, eng = _engine(V)
    ks = [1, 2, 3, 20, 49, 3, 2] if V < 10000 else [1, 2, 3, 20, 49]
    sents, c = _corpus(model, ks, seed=V)
    assert (np.diff(c.giv_off) == 0).any() and (np.diff(c.giv_off) > 0).any()
    Case(eng, model, c, own_padding=V < 10000).check(f64)


def test_k1_sentences_equal_bp():
    model, eng = _engine(1001, seed=3)
    sents, c = _corpus(model, [1] * 8, seed=5)
    r = eng.pseudo_likelihood(c)
    b = eng.run(c, c.roots_from_positions(synth.draw_roots(sents, 3, seed=1)), 3, want_grad=False)
    np.testing.assert_allclose(r.logp_var.cpu().numpy(), b.logp_var.cpu().numpy(), rtol=0, atol=1e-6)


def test_bad_label_gives_nan_outputs_and_refusals_leave_their_sentinels():
    model, eng = _engine(67, seed=2)
    sents, c = _corpus(model, [3, 4, 2], seed=8)
    case = Case(eng, model, c)
    lab = c.var_label.copy()
    lab[4] = 67                                                           # a label of sentence 1 outside [0, V)
    rc, o = case.run(0.0, labels=lab)
    assert rc == 0
    bad = slice(int(c.var_off[1]), int(c.var_off[2]))
    assert np.isnan(o['lp'][bad]).all() and (o['t1'][bad] == -1).all() and (o['rk'][bad] == INT_MAX).all()
    assert np.isnan(o['g'][bad]).all() and np.isnan(o['b'][bad, :67]).all()
    rc, ok = case.run(0.0)
    good = np.r_[0:int(c.var_off[1]), int(c.var_off[2]):c.n_vars]
    np.testing.assert_array_equal(o['lp'][good], ok['lp'][good])
    np.testing.assert_array_equal(o['g'][good], ok['g'][good])
    refused = [(1, dict(U=None)), (1, dict(planes=None)), (1, dict(logp_var=None)), (1, dict(V=0)), (1, dict(ldv=case.V - 1)),
               (1, dict(ldv=case.ld - 4)), (1, dict(ldf=case.ld - 4)), (1, dict(U=ctypes.c_void_p(case.U.data_ptr() + 4))),
               (1, dict(pmi=None)), (3, dict(max_k=50))]
    for code, over in refused:
        rc, o = case.run(0.0, **over)
        assert rc == code, over
        assert (o['lp'] == SENTINEL).all() and (o['t1'] == -7).all() and (o['g'] == SENTINEL).all() and \
            (o['b'] == SENTINEL).all(), over
    rc, o = case.run(0.0, want_grad=False, pmi=None, w1=None, edT=None, pedT=None, var_de=None)   # no gradient: no features
    assert rc == 0 and (o['g'] == SENTINEL).all() and (o['lp'][:-1] == ok['lp'][:-1]).all()
    rc, o = case.run(0.0, n_sent=0)
    assert rc == 0 and (o['lp'] == SENTINEL).all()


def _outs(r):
    return [x.cpu().numpy() for x in (r.grad, r.logp, r.logp_var, r.top1, r.rank, r.beliefs)]


def test_device_determinism_and_batch_order_microbatch_invariance():
    model, eng = _engine(1001, seed=5)
    sents = synth.make_corpus(model, 6, k=4, g=1, seed=9) + synth.make_corpus(model, 3, k=7, g=2, seed=10)
    a = _outs(eng.pseudo_likelihood(Corpus(sents), want_beliefs=True))
    for x, y in zip(a, _outs(eng.pseudo_likelihood(Corpus(sents), want_beliefs=True))):
        np.testing.assert_array_equal(x, y)
    off = Corpus(sents).var_off
    order = list(np.random.default_rng(2).permutation(len(sents)))
    co = Corpus([sents[i] for i in order])
    ro = _outs(eng.pseudo_likelihood(co, want_beliefs=True))
    for pos, s in enumerate(order):
        np.testing.assert_array_equal(ro[0][pos], a[0][s])
        for j in (2, 3, 4, 5):
            np.testing.assert_array_equal(ro[j][co.var_off[pos]:co.var_off[pos + 1]], a[j][off[s]:off[s + 1]])
    small = Engine(model, workspace_bytes=8 * eng.ld * 4 * 2)             # 8 variables per micro-batch
    small.set_theta(THETA[0], THETA[1], with_grad=True)
    rb = small.pseudo_likelihood(Corpus(sents), want_beliefs=True)
    assert rb.stats['micro_batches'] > 2
    for x, y in zip(a, _outs(rb)):
        np.testing.assert_array_equal(x, y)


def test_sum_product_bit_identical_around_pseudo_likelihood():
    model, eng = _engine(2304, seed=6)
    sents = synth.make_corpus(model, 6, k=5, g=1, seed=3)
    c = Corpus(sents)
    roots = c.roots_from_positions(synth.draw_roots(sents, 3, seed=4))
    kw = dict(want_grad=True, want_marg=True, want_beliefs=True)
    a = eng.run(c, roots, 3, **kw)
    eng.pseudo_likelihood(c, want_beliefs=True, want_topk=5)
    b = eng.run(c, roots, 3, **kw)
    for name in ('grad', 'logp', 'logp_var', 'top1', 'rank', 'beliefs'):
        np.testing.assert_array_equal(getattr(a, name).cpu().numpy(), getattr(b, name).cpu().numpy(), err_msg=name)


def test_trainer_pl_step_against_the_model_reference():
    from macaronicusermodeling_b200.trainer import Trainer
    model, eng = _engine(1001, seed=7)
    sents = synth.make_corpus(model, 16, k=6, g=1, seed=11)
    tr = Trainer(eng, reg_param=0.2, N=100, objective='pl')
    tr.theta_ee, tr.theta_ed = np.array(THETA[0]), np.array(THETA[1])
    h = tr.apply(tr.step(Corpus(sents), None, 0.01), 0.01)
    lp, g, _ = pl_oracle.model_reference(Corpus(sents), model, *THETA)
    np.testing.assert_allclose(h[:9], g.sum(axis=0), rtol=1e-4, atol=2e-6 * len(sents))
    assert h[9] == pytest.approx(lp.sum(), rel=1e-5) and h[14] == 16
    np.testing.assert_allclose(tr.theta_ed, np.array(THETA[1]) + 0.01 * (h[3:9] - 16 * 0.2 / 100 * np.array(THETA[1])),
                               rtol=1e-15)
