"""Shared checks of max-product decoding (Engine.run max_product, K10 / K11) for the CPU tier (emulated kernels) and the GPU
tier: brute-force enumeration of small sentences, the float64 reference (tests/maxprod_oracle.py) and the tolerance of a
device max-marginal against it."""
import numpy as np

from macaronicusermodeling_b200.engine import Corpus
import maxprod_oracle
from joint_checks import THETA_ED, THETA_EE, TREE_LAYOUTS  # noqa: F401  (shared cases)
from oracle import lbp_oracle as orc

U32 = 2.0 ** -24              # unit roundoff of fp32


def log_potentials(model, sent, te, td):
    """(var_ids, unary log-potentials {v: [V]}, pairwise {(a, b): [V, V]}) of a sentence, from the oracle's dense features"""
    g = orc.Graph(sent)
    V = model['pmi'].shape[0]
    phi_ee, phi_ee_w1 = orc.dense_phi_en_en(model)
    phi_ed = orc.dense_phi_en_de(model, sent)
    te, td = np.asarray(te, dtype=np.float64), np.asarray(td, dtype=np.float64)
    unary = {v: np.zeros(V) for v in g.var_ids}
    pair = {}
    for f in g.factors:
        if f.arity == 1:
            phi = phi_ed if f.ftype == orc.T_EN_DE else (phi_ee if f.gap > 1 else phi_ee_w1)
            unary[f.vars[0]] = unary[f.vars[0]] + phi[:, f.obs, :].dot(td if f.ftype == orc.T_EN_DE else te)
        else:
            pair[tuple(f.vars)] = (phi_ee if f.gap > 1 else phi_ee_w1).dot(te)
    return g.var_ids, unary, pair


def brute_force(model, sent, te, td):
    """(best assignment in predicted-position order, its log-potential, the labels' log-potential) by enumerating V^k"""
    var_ids, unary, pair = log_potentials(model, sent, te, td)
    k = len(var_ids)
    V = model['pmi'].shape[0]
    L = np.zeros((V,) * k)
    for i, v in enumerate(var_ids):
        L = L + unary[v].reshape([V if j == i else 1 for j in range(k)])
    for (a, b), P in pair.items():
        ia, ib = var_ids.index(a), var_ids.index(b)
        P = P if ia < ib else P.T                                 # axes in ascending variable order
        L = L + P.reshape([V if j in (ia, ib) else 1 for j in range(k)])
    best = np.unravel_index(int(np.argmax(L)), L.shape)
    labels = tuple(int(sent.label[v]) for v in var_ids)
    return np.array(best), float(L[best]), float(L[labels])


def marg_tol(k, sweeps=3, max_in=None):
    """Relative tolerance of a device max-marginal entry against float64.  Local roundings per update:
      K10  2^-22 (hi + lo of the stored message), ~2 ulp (exp_f2 of a compensated argument), one fp32 product, the 1/amax division;
      K3   one fp32 product per input (max_in + 1) and the renormalisation, ~2 ulp;
      K5   max_in + 1 fp32 products and the normalisation.
    A max passes the relative error of its arguments through without growth (it is 1-Lipschitz in the largest relative error),
    and a product adds its inputs' errors, so to first order a belief's error is the sum of the local roundings of the
    updates it depends on -- at most every update of the schedule, sweeps * k (k - 1) of each kind."""
    max_in = k - 1 if max_in is None else max_in
    k10 = 2.0 ** -22 + 4 * U32
    k3 = (max_in + 3) * U32
    k5 = (max_in + 2) * U32
    return sweeps * k * (k - 1) * (k10 + k3) + k5 + 2 * U32


def engine_decode(engine, sents, roots_pos, te, td, sweeps=3, **kw):
    """(Result, corpus) of one max-product run"""
    engine.set_theta(te, td, with_grad=True)
    corpus = Corpus(sents)
    return engine.run(corpus, corpus.roots_from_positions(roots_pos), sweeps, want_grad=False, want_marg=True,
                      want_beliefs=True, max_product=True, **kw), corpus


def oracle_decode(model, sents, roots_pos, te, td, sweeps=3):
    """[(max-marginals, decoding)] per sentence"""
    tb = orc.Tables(model, te, td)
    return [maxprod_oracle.decode(tb, s, roots_pos[i], sweeps) for i, s in enumerate(sents)]


def check_decode(result, corpus, model, want, te, td, sweeps=3):
    """device max-marginals within marg_tol of the oracle's, the decoding equal wherever the oracle's runner-up is outside the
    band, scores equal to NumPy's on the device's decoding and the labels; returns the number of near-ties excluded"""
    V = model['pmi'].shape[0]
    B = result.beliefs.cpu().numpy()[:, :V].astype(np.float64)
    top1 = result.top1.cpu().numpy()
    excluded = 0
    for s, (mm, dec) in enumerate(want):
        lo, hi = int(corpus.var_off[s]), int(corpus.var_off[s + 1])
        tol = marg_tol(hi - lo, sweeps)
        err = np.abs(B[lo:hi] - mm)
        assert (err <= 2 * tol * mm + 2.0 ** -126).all(), (s, float((err / np.maximum(mm, 1e-300)).max()), tol)
        srt = np.sort(mm, axis=1)
        tie = srt[:, -2] >= srt[:, -1] * (1 - 4 * tol)
        excluded += int(tie.sum())
        assert (top1[lo:hi][~tie] == dec[~tie]).all(), (s, top1[lo:hi], dec)
    np.testing.assert_allclose(result.map_score.cpu().numpy(), maxprod_oracle.assignment_scores(model, te, td, corpus, top1),
                               rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(result.label_score.cpu().numpy(),
                               maxprod_oracle.assignment_scores(model, te, td, corpus, corpus.var_label), rtol=1e-12, atol=1e-12)
    return excluded
