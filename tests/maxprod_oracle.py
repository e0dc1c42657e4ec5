"""Float64 reference of max-product decoding (Engine.run max_product, K10 / K11) -- TEST INFRASTRUCTURE.

`final_messages` is bethe_oracle.final_messages' message loop (the schedule, unary products and renormalisation of
oracle/lbp_oracle.run_fast) with the pairwise update replaced by the max-product one,
    mu_{F->v}(x) = max_y T_F(x, y) nu_{u->F}(y),
computed in column blocks so that V = 10 000 stays feasible for short sentences.  `decode` gives the normalised max-marginals
and their arg-max (np.argmax: first index on ties).  `assignment_scores` is the log of the unnormalised joint potential of any
assignment, K11's formula on the Corpus arrays."""
import numpy as np

from oracle import lbp_oracle as orc

BLOCK_ELEMS = 1 << 22          # float64 elements of one (rows x V x columns) product block


def max_times(M, B):
    """out[i, n] = max_k M[i, k] * B[k, n] (M, B >= 0), in column blocks"""
    M = np.asarray(M, dtype=np.float64)
    out = np.empty((M.shape[0], B.shape[1]))
    step = max(1, BLOCK_ELEMS // max(1, M.shape[0] * M.shape[1]))
    for n0 in range(0, B.shape[1], step):
        out[:, n0:n0 + step] = (M[:, :, None] * B[None, :, n0:n0 + step]).max(axis=1)
    return out


def final_messages(tables, sent, roots, sweeps=3):
    """{'graph', 'uprod', 'v2f', 'f2v'} after max-product sweeps, float64"""
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
            D = max_times(np.stack([it[2] for it in items]), B)
            for (fid, v, _), row in zip(items, D):
                s = row.sum()
                f2v[fid, v] = row / s if s > 0 else uni
    return {'graph': g, 'uprod': uprod, 'v2f': v2f, 'f2v': f2v}


def decode(tables, sent, roots, sweeps=3):
    """(max-marginals [k, V] normalised to sum 1, decoding [k]) in the order of the sentence's predicted positions"""
    msgs = final_messages(tables, sent, roots, sweeps)
    g = msgs['graph']
    rows = []
    for v in g.var_ids:
        m = msgs['uprod'][v]
        for fid in g.facset[v]:
            if g.factors[fid].arity == 2:
                m = m * msgs['f2v'][fid, v]
        rows.append(m / m.sum())
    mm = np.array(rows)
    return mm, np.argmax(mm, axis=1)


def assignment_scores(model, theta_ee, theta_ed, corpus, x):
    """[n_sent] float64: K11's log-potential of the assignment x (one entry per Corpus variable) from the model's feature
    arrays (pmi, pmi_w1 [V, V], ed, ped [V, Vd]) and the Corpus arrays"""
    te, td = np.asarray(theta_ee, dtype=np.float64).reshape(3), np.asarray(theta_ed, dtype=np.float64).reshape(6)
    P, W = np.asarray(model['pmi'], dtype=np.float64), np.asarray(model['pmi_w1'], dtype=np.float64)
    E, Pd = np.asarray(model['ed'], dtype=np.float64), np.asarray(model['ped'], dtype=np.float64)
    x = np.asarray(x).astype(np.int64)
    c = corpus
    ell = lambda a, b, g: te[0] * P[a, b] + te[2] + (te[1] * W[a, b] if g else 0.0)
    out = np.zeros(c.n_sent)
    for s in range(c.n_sent):
        v0 = int(c.var_off[s])
        total = 0.0
        for v in range(v0, int(c.var_off[s + 1])):
            xi, d = int(x[v]), int(c.var_de[v])
            if d >= 0:
                total += td[0] * E[xi, d] + td[1] * Pd[xi, d] + td[5]
                for q in range(int(c.sp_off[v]), int(c.sp_off[v + 1])):
                    if int(c.sp_en[q]) == xi:
                        total += td[int(c.sp_feat[q])] * float(c.sp_val[q])
            for j in range(int(c.giv_off[v]), int(c.giv_off[v + 1])):
                total += ell(xi, int(c.giv_label[j]), int(c.giv_gap1[j]))
        for f in range(int(c.pair_off[s]), int(c.pair_off[s + 1])):
            total += ell(int(x[v0 + int(c.pair_v0[f])]), int(x[v0 + int(c.pair_v1[f])]), int(c.pair_gap1[f]))
        out[s] = total
    return out
