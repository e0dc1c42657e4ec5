"""References of the pseudo-likelihood kernel K13 (mlbp_pseudo_likelihood, csrc/pseudo.cu).

* plane level (`planes_reference`): K13's conditional q from the same fp16 planes and K1 rows, formed as tests/gibbs_oracle.py
  forms a Gibbs conditional with the labels as the state, Z in the kernel's block order, and the gradient from the gradient
  planes in float64 -- logp_var, top1 and rank reproduce the device's exactly up to the last bits of the log;
* model level (`model_reference`): float64 from the fp32 feature matrices, only the label rows and columns (O(V) per factor):
  the quantity K13 approximates, with its exact gradient."""
import numpy as np

import gibbs_oracle

N_GRAD = 9


def block_total(q):
    """Z = sum of q [V] in K13's (= K12's) block order: C(V - 1) of include/mlbp.h"""
    V = q.shape[0]
    E = gibbs_oracle.columns_per_thread(V)
    T = gibbs_oracle.THREADS
    Q = np.zeros(T * E)
    Q[:V] = q
    s = np.cumsum(Q.reshape(T, E), axis=1)
    W = s[:, -1].reshape(T // 32, 32).copy()
    for d in (1, 2, 4, 8, 16):
        W[:, d:] = W[:, d:] + W[:, :-d]
    ex = np.zeros_like(W)
    ex[:, 1:] = W[:, :-1]
    O = np.zeros(T // 32)
    for w in range(1, T // 32):
        O[w] = O[w - 1] + W[w - 1, -1]
    base = (O[:, None] + ex).reshape(T)
    t = (V - 1) // E
    return float(base[t] + s[t, -1])


def _sentences(c):
    for s in range(c.n_sent):
        v0, v1, p0, p1 = int(c.var_off[s]), int(c.var_off[s + 1]), int(c.pair_off[s]), int(c.pair_off[s + 1])
        pairs = list(zip(c.pair_v0[p0:p1].tolist(), c.pair_v1[p0:p1].tolist(), c.pair_gap1[p0:p1].tolist()))
        yield v0, v1, gibbs_oracle.neighbours(v1 - v0, pairs)


def _giv(c, i):
    return [(int(c.giv_label[j]), int(c.giv_gap1[j])) for j in range(int(c.giv_off[i]), int(c.giv_off[i + 1]))]


def _sparse(c, i):
    return [(int(c.sp_en[j]), int(c.sp_feat[j]), float(c.sp_val[j])) for j in range(int(c.sp_off[i]), int(c.sp_off[i + 1]))]


def planes_reference(c, U, planes, colsums, scale_exp, pmi, w1, edT, pedT, f64, want_grad=True):
    """K13 from the kernel's inputs: U [n_vars, >= V] fp32 (K1's rows), planes: 20 fp16 arrays [V, >= V], colsums [7, V],
    pmi / w1 [V, >= V] and edT / pedT [Vd, >= V] fp32.  Returns (logp_var, top1, rank, grad [n_vars, 9], beliefs [n_vars, V] fp32,
    grad_scale [n_vars, 9]: the sum of the absolute values of the terms of each gradient component, the scale of its rounding)."""
    V = colsums.shape[1]
    nv = c.n_vars
    unscale = 2.0 ** -scale_exp
    logp, top1, rank = np.zeros(nv), np.zeros(nv, dtype=np.int32), np.zeros(nv, dtype=np.int32)
    grad, scale = np.zeros((nv, N_GRAD)), np.zeros((nv, N_GRAD))
    rows = np.zeros((nv, V), dtype=np.float32)
    tab = lambda p, y: planes[p][y, :V].astype(np.float32) + planes[p + 1][y, :V].astype(np.float32)
    for v0, v1, nb in _sentences(c):
        lab = c.var_label[v0:v1]
        for li in range(v1 - v0):
            i = v0 + li
            yi = int(lab[li])
            q = U[i, :V].astype(np.float64 if f64 else np.float32)
            terms = []                                                 # (T row, G row plane, W row plane or None, row, obs cell)
            for j, dim1, g in nb[li]:
                y = int(lab[j])
                plane = (4 if g else 0) if dim1 else (6 if g else 2)
                t = tab(plane, y)
                f = np.float32(unscale * V / colsums[(6 if g else 5) if dim1 else (1 if g else 0)][y])
                q = q * (t.astype(np.float64) * np.float64(f)) if f64 else q * (t * f)
                terms.append((t, (10 if g else 8) if dim1 else (16 if g else 14), (12 if dim1 else 18) if g else None, y,
                              (y, yi) if dim1 else (yi, y)))
            for o, g in _giv(c, i):
                terms.append((tab(6 if g else 2, o), 16 if g else 14, 18 if g else None, o, (yi, o)))
            Z = block_total(q.astype(np.float64))
            logp[i] = np.log(float(q[yi]) / Z) if q[yi] > 0 else -99.99
            top1[i] = int(np.argmax(q))
            rank[i] = int((q > q[yi]).sum())
            rows[i] = (q.astype(np.float64) / Z).astype(np.float32)
            if not want_grad:
                continue
            p = (q.astype(np.float64) * (1.0 / Z)).astype(np.float32).astype(np.float64)
            live = p > 0
            for t, gp, wp, y, cell in terms:
                for comp, plane, M in ((0, gp, pmi), (1, wp, w1)):
                    if plane is None:
                        continue
                    feat = np.where(live, tab(plane, y).astype(np.float64) / np.where(live, t, 1.0), 0.0)
                    grad[i, comp] += float(M[cell]) - (p * feat).sum()
                    scale[i, comp] += abs(float(M[cell])) + (p * np.abs(feat)).sum()
            d = int(c.var_de[i])
            if d >= 0:
                for comp, M in ((3, edT), (4, pedT)):
                    grad[i, comp] = float(M[d, yi]) - (p * M[d, :V]).sum()
                    scale[i, comp] = abs(float(M[d, yi])) + (p * np.abs(M[d, :V])).sum()
                for e, f, val in _sparse(c, i):
                    pe = p[e] if 0 <= e < V else 0.0
                    grad[i, 3 + f] += val * ((1.0 if e == yi else 0.0) - pe)
                    scale[i, 3 + f] += abs(val)
    return logp, top1, rank, grad, rows, scale


class _Rows(object):
    """float64 rows / columns of a matrix, converted one at a time (V = 50 000 stays O(V) per read)"""

    def __init__(self, a):
        self.a = a

    def __getitem__(self, idx):
        return np.asarray(self.a[idx], dtype=np.float64)


def model_reference(c, model, te, td):
    """float64 conditionals of the model's labels from the feature matrices (model dict: pmi, pmi_w1 [V, V], ed, ped [V, Vd]):
    (logp_var, grad [n_vars, 9], p [n_vars, V]).  log q_i(x) = the en_de log-potential (with the sparse features) + one pmi /
    pmi_w1 log-potential per given token and per pairwise factor at the neighbours' labels."""
    P, W, ed, ped = (_Rows(model[k]) for k in ('pmi', 'pmi_w1', 'ed', 'ped'))
    te, td = np.asarray(te, dtype=np.float64), np.asarray(td, dtype=np.float64)
    V = P.a.shape[0]
    nv = c.n_vars
    logp, grad, probs = np.zeros(nv), np.zeros((nv, N_GRAD)), np.zeros((nv, V))
    for v0, v1, nb in _sentences(c):
        lab = c.var_label[v0:v1]
        for li in range(v1 - v0):
            i = v0 + li
            yi = int(lab[li])
            feats = []                                                 # (component, feature [V] over x)
            L = np.zeros(V)
            d = int(c.var_de[i])
            if d >= 0:
                L += td[0] * ed[:, d] + td[1] * ped[:, d] + td[5]
                feats += [(3, ed[:, d]), (4, ped[:, d])]
                for e, f, val in _sparse(c, i):
                    one = np.zeros(V)
                    one[e] = val
                    L += td[f] * one
                    feats.append((3 + f, one))
            cols = [(W[:, o] if g else None, P[:, o]) for o, g in _giv(c, i)]
            for j, dim1, g in nb[li]:
                y = int(lab[j])
                cols.append(((W[y, :] if dim1 else W[:, y]) if g else None, P[y, :] if dim1 else P[:, y]))
            for w, pm in cols:
                L += te[0] * pm + te[2] + (te[1] * w if w is not None else 0.0)
                feats.append((0, pm))
                if w is not None:
                    feats.append((1, w))
            p = np.exp(L - L.max())
            p /= p.sum()
            probs[i] = p
            logp[i] = np.log(p[yi])
            for comp, phi in feats:
                grad[i, comp] += phi[yi] - p.dot(phi)
    return logp, grad, probs
