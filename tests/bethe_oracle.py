"""Float64 reference of the joint log-likelihood (Engine.run want_joint, K9 mlbp_joint_logp) -- TEST INFRASTRUCTURE.

`final_messages` runs the message loop of oracle/lbp_oracle.run_fast (same graph, schedule, unary products, batched
factor->variable GEMVs, renormalisation) and keeps the final messages, which run_fast discards.  `bethe_joint_logp` evaluates
the Bethe estimate of log p(y) at those messages:
    log p_B(y) = sum_i log b_i(y_i)
               + sum_F [ log T_F(y) - log Z_F + sum_{k in F} ( log O_{F,k} - log mu_{F->k}(y_k) ) ]
    Z_F = nu_{i->F}' T_F nu_{j->F},   O_{F,k} = nu_{k->F} . mu_{F->k}
Every message enters once with + and once with -, so the value does not depend on any one message's scale.  Exact on trees.
-inf when some label has belief 0 (where the marginal sum counts -99.99, LBP.py:247-259)."""
import numpy as np

from oracle import lbp_oracle as orc


def final_messages(tables, sent, roots, sweeps=3):
    """{'graph', 'uprod', 'v2f', 'f2v'} after the reference's sweeps, float64, as run_fast computes them"""
    model = tables.model
    td = tables.td
    g = orc.Graph(sent)
    V = model['pmi'].shape[0]
    unary = {}
    for f in g.factors:
        if f.arity != 1:
            continue
        if f.ftype == orc.T_EN_DE:
            z = td[0] * tables.edT[f.obs] + td[1] * tables.pedT[f.obs] + td[5]
            for e, d, k, val in sent.sparse:
                if int(d) == f.obs:
                    z[int(e)] += td[int(k)] * val
            unary[f.id] = np.exp(z)
        else:
            unary[f.id] = (tables.T1t if f.gap == 1 else tables.Tt)[f.obs]
    uprod = {}
    for v in g.var_ids:
        m = np.full(V, 1.0 / V)
        for fid in g.facset[v]:
            if g.factors[fid].arity == 1:
                m = m * (unary[fid] / unary[fid].sum())
        uprod[v] = m
    uni = np.full(V, 1.0 / V)
    v2f, f2v = {}, {}
    for f in g.factors:
        if f.arity == 2:
            for v in f.vars:
                v2f[v, f.id] = uni
                f2v[f.id, v] = uni
    _, seq = g.update_sequence(roots, sweeps)
    i = 0
    while i < len(seq):
        frm, to = seq[i]
        if frm[0] == 'X':
            v, fid = frm[1], to[1]
            m = uprod[v]
            for of in g.facset[v]:
                if of != fid and g.factors[of].arity == 2:
                    m = m * f2v[of, v]
            s = m.sum()
            v2f[v, fid] = m / s if s > 0 else uni
            i += 1
            continue
        run = []
        while i < len(seq) and seq[i][0][0] == 'F':
            fid, v = seq[i][0][1], seq[i][1][1]
            if g.factors[fid].arity == 2:
                run.append((fid, v))
            i += 1
        groups = {}
        for fid, v in run:
            f = g.factors[fid]
            to_dim0 = (f.vars[0] == v)
            o = f.vars[1] if to_dim0 else f.vars[0]
            groups.setdefault((f.gap == 1, to_dim0), []).append((fid, v, v2f[o, fid]))
        for (w1, to_dim0), items in groups.items():
            B = (tables.T1t if w1 else tables.Tt) if to_dim0 else (tables.T1 if w1 else tables.T)
            D = np.stack([it[2] for it in items]).dot(B)
            for (fid, v, _), row in zip(items, D):
                s = row.sum()
                f2v[fid, v] = row / s if s > 0 else uni
    return {'graph': g, 'uprod': uprod, 'v2f': v2f, 'f2v': f2v}


def bethe_joint_logp(tables, sent, roots, sweeps=3, messages=None):
    """the Bethe estimate of the labels' joint log-likelihood at `messages` (default: final_messages(...))"""
    if messages is None:
        messages = final_messages(tables, sent, roots, sweeps)
    g, uprod, v2f, f2v = messages['graph'], messages['uprod'], messages['v2f'], messages['f2v']
    te = tables.te
    pmi, w1 = tables.model['pmi'], tables.model['pmi_w1']
    total = 0.0
    for v in g.var_ids:
        m = uprod[v]
        for fid in g.facset[v]:
            if g.factors[fid].arity == 2:
                m = m * f2v[fid, v]
        s = m.sum()
        b = m[g.label[v]] / s if s > 0 else 1.0 / len(m)
        if not b > 0:
            return -np.inf
        total += np.log(b)
    for f in g.factors:
        if f.arity != 2:
            continue
        a, b = f.vars
        ya, yb = g.label[a], g.label[b]
        gap1 = f.gap == 1
        log_t = te[0] * float(pmi[ya, yb]) + te[2] + (te[1] * float(w1[ya, yb]) if gap1 else 0.0)
        z = v2f[a, f.id].dot((tables.T1 if gap1 else tables.T).dot(v2f[b, f.id]))
        total += log_t - np.log(z)
        for k, y in ((a, ya), (b, yb)):
            mu = f2v[f.id, k]
            total += np.log(v2f[k, f.id].dot(mu)) - np.log(mu[y])
    return float(total)
