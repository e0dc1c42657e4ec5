"""Shared checks of the joint log-likelihood (Engine.run want_joint, K9 mlbp_joint_logp) for the CPU tier (emulated kernels)
and the GPU tier: brute-force enumeration on trees, the float64 reference (tests/bethe_oracle.py) on loopy sentences."""
import numpy as np

from macaronicusermodeling_b200 import synth
from macaronicusermodeling_b200.engine import Corpus
import bethe_oracle
from oracle import lbp_oracle as orc

TREE_LAYOUTS = ['pp', 'pgp', 'gpgpg', 'prp']
THETA_EE, THETA_ED = [0.7, -0.4, 0.2], [1.1, -0.6, 0.4, 0.3, -0.5, 0.1]


def brute_force_joint(model, sent, te, td):
    """log p(y) of the labels by enumerating the two-variable joint  u_a(x_a) u_b(x_b) T[x_a, x_b]"""
    g = orc.Graph(sent)
    V = model['pmi'].shape[0]
    phi_ee, phi_ee_w1 = orc.dense_phi_en_en(model)
    phi_ed = orc.dense_phi_en_de(model, sent)
    te, td = np.asarray(te, dtype=np.float64), np.asarray(td, dtype=np.float64)
    unary = {v: np.ones(V) for v in g.var_ids}
    pair = None
    for f in g.factors:
        if f.arity == 1:
            phi = phi_ed if f.ftype == orc.T_EN_DE else (phi_ee if f.gap > 1 else phi_ee_w1)
            unary[f.vars[0]] = unary[f.vars[0]] * np.exp(phi[:, f.obs, :].dot(td if f.ftype == orc.T_EN_DE else te))
        else:
            pair = f
    a, b = pair.vars
    joint = unary[a][:, None] * unary[b][None, :] * np.exp((phi_ee if pair.gap > 1 else phi_ee_w1).dot(te))
    return float(np.log(joint[g.label[a], g.label[b]] / joint.sum()))


def joint_tol(n_pairs, V):
    """Absolute tolerance of a sentence's device joint against float64.  Each factor's Z comes from gradient-stage rows that
    multiply only the fp16 hi half of the message r (A_HI_ONLY, and one pass on top at V >= 4096), while O_1 reads hi + lo:
    log Z is off by the relative share of the dropped lo halves, each at most 2^-11 of its element and of random sign, so
    ~2^-11 / sqrt(V) per factor (8 sigma here); one-pass rows add their accumulation bias, -4.4e-6 relative per Z row
    (DESIGN.md section 4).  The O dots (fp32 products, float64 sums) and the 2^-22 hi/lo split are far below both."""
    return n_pairs * (8.0 * 2.0 ** -11 / np.sqrt(V) + 5e-6) + 1e-6


def tree_sentences(model, seed=11):
    return [synth.sentence_to_arrays(synth.make_sentence(model, l, seed=seed + i, n_history=2)) for i, l in enumerate(TREE_LAYOUTS)]


def engine_joint(engine, sents, roots_pos, te, td, sweeps=3, want_grad=False, **kw):
    """(Result, corpus) of one want_joint run"""
    engine.set_theta(te, td, with_grad=True)
    corpus = Corpus(sents)
    return engine.run(corpus, corpus.roots_from_positions(roots_pos), sweeps, want_grad=want_grad, want_marg=True,
                      want_joint=True, **kw), corpus


def oracle_joints(model, sents, roots_pos, te, td, sweeps=3):
    tb = orc.Tables(model, te, td)
    return np.array([bethe_oracle.bethe_joint_logp(tb, s, roots_pos[i], sweeps) for i, s in enumerate(sents)])
