"""NumPy reference of the Gibbs sampler K12 and its reduce (mlbp_gibbs_sample / mlbp_gibbs_reduce, csrc/gibbs.cu), vectorised over
chains: the conditional's products, the float64 running sums, the block-scan order of the draw, Philox4x32-10 and the
Rao-Blackwell rows in exactly the order include/mlbp.h states, so that the device's samples, accumulators and marginals can be
compared bit for bit.  Also the exact marginals of a small sentence by enumeration, the yardstick of the sampler's statistics."""
import numpy as np

THREADS = 256                        # MLBP_GIBBS_THREADS
MASK = np.uint64(0xffffffff)
_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)


def philox4x32_10(ctr, key):
    """Philox4x32-10 (Random123): ctr [..., 4] and key [..., 2] of 32-bit words -> [..., 4] uint64 holding 32-bit words"""
    ctr, key = np.asarray(ctr, dtype=np.uint64), np.asarray(key, dtype=np.uint64)
    c = [ctr[..., j] & MASK for j in range(4)]
    k0, k1 = key[..., 0] & MASK, key[..., 1] & MASK
    for _ in range(10):
        p0, p1 = c[0] * _M0, c[2] * _M1                          # < 2^64: exact in uint64
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & MASK, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & MASK]
        k0, k1 = (k0 + _W0) & MASK, (k1 + _W1) & MASK
    return np.stack(c, axis=-1)


def uniforms(seed, sent_id, chains, sweep, i):
    """the 53-bit uniform of update (sweep, i) of every chain of sentence sent_id"""
    seed = int(seed) & 0xffffffffffffffff
    n = len(chains)
    ctr = np.stack([np.full(n, int(sent_id) & 0xffffffff), np.asarray(chains), np.full(n, sweep), np.full(n, i)], axis=-1)
    w = philox4x32_10(ctr.astype(np.uint64), np.array([seed & 0xffffffff, seed >> 32], dtype=np.uint64))
    return ((w[:, 0] >> np.uint64(5)).astype(np.float64) * 2.0 ** 26 + (w[:, 1] >> np.uint64(6)).astype(np.float64)) * 2.0 ** -53


def columns_per_thread(V):
    return (V + 8 * THREADS - 1) // (8 * THREADS) * 8


def draw(q, u):
    """(x [C], Rao-Blackwell row [C, V] fp32, relative margin [C]) of the conditionals q [C, V] (fp32 or fp64) and uniforms u [C]:
    C(e) = (O_w + E_t) + s_t(e) of include/mlbp.h, x = the smallest x with C(x) > u C(V - 1).  The margin is the distance of
    u C(V - 1) from the two running sums around the draw, over C(V - 1): a draw the device could take differently only if it
    is tiny."""
    C, V = q.shape
    E = columns_per_thread(V)
    Q = np.zeros((C, THREADS * E))
    Q[:, :V] = q
    s = np.cumsum(Q.reshape(C, THREADS, E), axis=2)               # sequential float64 sums (np.add.accumulate)
    W = s[:, :, -1].reshape(C, THREADS // 32, 32).copy()
    for d in (1, 2, 4, 8, 16):                                    # Kogge-Stone inside each warp
        W[:, :, d:] = W[:, :, d:] + W[:, :, :-d]
    ex = np.zeros_like(W)
    ex[:, :, 1:] = W[:, :, :-1]
    O = np.zeros((C, THREADS // 32))
    for w in range(1, THREADS // 32):
        O[:, w] = O[:, w - 1] + W[:, w - 1, -1]
    base = (O[:, :, None] + ex).reshape(C, THREADS)
    Cx = (base[:, :, None] + s).reshape(C, -1)[:, :V]
    tot = Cx[:, V - 1]
    ok = (tot > 0) & np.isfinite(tot)
    with np.errstate(invalid='ignore', over='ignore', divide='ignore'):
        target = u * tot
        hit = Cx > target[:, None]
        last = V - 1 - np.argmax((q > 0)[:, ::-1], axis=1)
        x = np.where(hit.any(axis=1), np.argmax(hit, axis=1), last)
        x = np.where(ok, x, np.minimum((u * V).astype(np.int64), V - 1))
        term = np.where(ok[:, None], (q.astype(np.float64) / tot[:, None]).astype(np.float32), np.float32(1.0 / V))
        rows = np.arange(C)
        above = np.abs(Cx[rows, x] - target)
        below = np.where(x > 0, np.abs(target - Cx[rows, np.maximum(x - 1, 0)]), np.inf)
        margin = np.where(ok, np.minimum(above, below) / tot, np.inf)
    return x, term.astype(np.float32), margin


def neighbours(k, pairs):
    """per variable, (other variable, 1 if the variable is dim 1, gap1) of every factor touching it, in pair-list order"""
    nb = [[] for _ in range(k)]
    for a, b, g in pairs:
        nb[a].append((b, 0, int(bool(g))))
        nb[b].append((a, 1, int(bool(g))))
    return nb


def sample_sentence(U, planes, colsums, scale_exp, pairs, sent_id, seed, chains, burn_in, n_keep, f64):
    """One sentence, every chain at once.  U [k, >= V] fp32 (K1's rows); planes: fp16 [>= 8, V, >= V] (T.hi T.lo Tt.hi Tt.lo T1.hi
    T1.lo T1t.hi T1t.lo); colsums [7, V] float64; pairs [(v0, v1, gap1)] local.  Returns (acc [chains, k, V] fp32, samples
    [chains, n_keep, k] int32, min_margin [chains, n_sweeps, k])."""
    V = colsums.shape[1]
    k = U.shape[0]
    nb = neighbours(k, pairs)
    unscale = 2.0 ** -scale_exp
    ch = np.arange(chains)
    x = np.zeros((chains, k), dtype=np.int64)
    acc = np.zeros((chains, k, V), dtype=np.float32)
    samples = np.zeros((chains, n_keep, k), dtype=np.int32)
    margins = np.zeros((chains, 1 + burn_in + n_keep, k))
    for sw in range(1 + burn_in + n_keep):
        for i in range(k):
            q = np.broadcast_to(U[i, :V].astype(np.float64 if f64 else np.float32), (chains, V)).copy()
            for j, dim1, g in (nb[i] if sw > 0 else ()):
                y = x[:, j]
                plane = (4 if g else 0) if dim1 else (6 if g else 2)
                t = planes[plane][y, :V].astype(np.float32) + planes[plane + 1][y, :V].astype(np.float32)
                f = (unscale * V / colsums[(6 if g else 5) if dim1 else (1 if g else 0)][y]).astype(np.float32)
                if f64:
                    q = q * (t.astype(np.float64) * f.astype(np.float64)[:, None])
                else:
                    q = q * (t * f[:, None])
            xi, term, margins[:, sw, i] = draw(q, uniforms(seed, sent_id, ch, sw, i))
            x[:, i] = xi
            if sw > burn_in:
                acc[:, i] = term if sw == burn_in + 1 else acc[:, i] + term
        if sw > burn_in:
            samples[:, sw - burn_in - 1] = x
    return acc, samples, margins


def sample(var_off, pair_off, pair_v0, pair_v1, pair_gap1, sent_ids, U, planes, colsums, scale_exp, seed, chains, burn_in, n_keep,
           f64):
    """Every sentence of a batch: (acc [chains, n_vars, V], samples [chains, n_keep, n_vars], margins [chains, sweeps, n_vars])"""
    V = colsums.shape[1]
    nv = int(var_off[-1])
    acc = np.zeros((chains, nv, V), dtype=np.float32)
    smp = np.zeros((chains, n_keep, nv), dtype=np.int32)
    mg = np.zeros((chains, 1 + burn_in + n_keep, nv))
    for s in range(len(var_off) - 1):
        v0, v1, p0, p1 = int(var_off[s]), int(var_off[s + 1]), int(pair_off[s]), int(pair_off[s + 1])
        pairs = list(zip(pair_v0[p0:p1].tolist(), pair_v1[p0:p1].tolist(), pair_gap1[p0:p1].tolist()))
        acc[:, v0:v1], smp[:, :, v0:v1], mg[:, :, v0:v1] = sample_sentence(U[v0:v1], planes, colsums, scale_exp, pairs,
                                                                           int(sent_ids[s]), seed, chains, burn_in, n_keep, f64)
    return acc, smp, mg


def reduce(acc, labels, n_keep):
    """mlbp_gibbs_reduce: (marginals fp32 [n, V], label_prob [n, chains], logp_var, top1, rank)"""
    chains, n, V = acc.shape
    s = np.zeros((n, V))
    for c in range(chains):
        s = s + acc[c].astype(np.float64)
    m = s / (float(chains) * float(n_keep))
    rows = np.arange(n)
    ml = m[rows, labels]
    with np.errstate(divide='ignore'):
        logp = np.where(ml > 0, np.log(np.where(ml > 0, ml, 1.0)), -99.99)
    label_prob = acc[:, rows, labels].T.astype(np.float64) / n_keep
    return m.astype(np.float32), label_prob, logp, np.argmax(m, axis=1).astype(np.int32), (m > ml[:, None]).sum(axis=1)


def exact_marginals(model, sent, te, td, drop=()):
    """per-variable marginals [k, V] of the model's joint by enumerating V^k (pairwise factors listed in `drop` left out, to
    show that a check has power)"""
    from map_checks import log_potentials
    var_ids, unary, pair = log_potentials(model, sent, te, td)
    k, V = len(var_ids), model['pmi'].shape[0]
    L = np.zeros((V,) * k)
    for i, v in enumerate(var_ids):
        L = L + unary[v].reshape([V if j == i else 1 for j in range(k)])
    for (a, b), P in pair.items():
        ia, ib = var_ids.index(a), var_ids.index(b)
        if (ia, ib) in drop:
            continue
        P = P if ia < ib else P.T
        L = L + P.reshape([V if j in (ia, ib) else 1 for j in range(k)])
    p = np.exp(L - L.max())
    p /= p.sum()
    return np.array([p.sum(axis=tuple(j for j in range(k) if j != i)) for i in range(k)])
