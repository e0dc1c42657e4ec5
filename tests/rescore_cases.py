"""Near-tie cases for K5 (mlbp_marginals with near-tie flags) and K5b (mlbp_rescore_candidates, csrc/rescore.cu), laid out as
the engine lays them out, with their float64 reference and an exact host model of K5's flags.  Host only: NumPy.

Layout (include/mlbp.h):
  U        [n_u, ld] fp32, ld = roundup(V, 64), one row per variable;
  A_hi/lo  [n_a, ld] fp16 message rows;
  D        [MLBP_D_CONST_ROWS + n_a, ld] fp32: row 0 the constant-one row, rows 1..4 constant-folded rows (K5b uses them as
           stored), row MLBP_D_CONST_ROWS + a the stored message row of A row a;
  planes   MLBP_N_PLANES fp16 planes [V, ld]: plane pair p (tables 0..3 are the message tables) has row e = row rowmap[p, e] of
           one pool of hi / lo rows.  Each pair has its own row map, so the ten pairs hold distinct content (a wrong plane
           index reads valid memory and gives wrong numbers) while the host keeps one table's worth of float64 values.
  Every row's padding (columns V .. ld) is NaN: the last 16-byte chunk of a row must be masked wherever V % 8 != 0.
  msg_blocks {table, a0, d0, rows}: ascending, contiguous, several blocks per table.

Stored message rows are  D[5 + a] = fp32(alpha_a * Dhat_a * (1 + eps_a)),  Dhat_a = (A_hi + A_lo)[a] . (B_hi + B_lo)[table]^T in
float64 and alpha_a a power of two (stored rows near 1).  eps_a stands in for the rounding of reduced-pass GEMM rows: per
variable the perturbations of its rows add up to at most eps = tau / 8 at every element.

Reference: the log belief  log U[e] + sum_j log Dhat_j[e]  (constant rows: the stored value; uniform inputs skipped); its
arg-max (first index on ties) and the label's rank #{e : b[e] > b[label]}.  Log space keeps the variables whose products
leave the fp32 range exact.

Engineered variables (kind):
  argmax      the two largest beliefs at a relative gap in [1e-6, tau/2]; about half are reversed in the stored rows by eps
  argmax_tie  an exact float64 tie of the two largest (duplicated table rows, equal U), a third candidate just below it
  rank        the label below R < 46 certainly-larger beliefs, with band neighbours within +-tau_label/2, some reversed by eps
  bit1_50 / bit1_51   exactly 50 / 51 beliefs certainly above the label plus one reversed band neighbour
  edge_best   no pairwise inputs (two uniform ones): the runner-up exactly at best * (1 - tau) in fp32
  edge_lab    no inputs at all: neighbours exactly at plab * (1 + tau_label) and plab * (1 - tau_label) in fp32
  mass        70 candidates inside the arg-max band (K5b skips it: counters[1])
  degenerate  a zero A row under a positive stored D row (K5b skips it: counters[2])
  zero_label  U[label] = 0 and a reversed arg-max near-tie
  deep        64 inputs (message, constant and uniform); deep_underflow: its product underflows fp32 (fp64 variants only)
  random      no engineering (1..8 inputs of all three sorts)
"""
import numpy as np

D_CONST_ROWS = 5                  # MLBP_D_CONST_ROWS
N_PLANE_PAIRS = 10                # MLBP_N_PLANES / 2
MAX_IN = 64                       # inputs a variable may have (K5, K5b)
MAX_CAND = 64                     # RS_MAX_CAND in csrc/rescore.cu
RANK_LIMIT = 50                   # K5 flags the label's rank while at most this many beliefs are certainly above it
# K5b's own error on a ratio of two beliefs: fp32 products of the 22-bit operands, per-thread fp32 chains of V / 256 terms,
# float64 block sums -- ~1e-8 per hop.  Float64 decisions between beliefs closer than this are not promised.
GAP = 1e-7
BANDS = {'two_pass': (2e-4, 1e-4), 'one_pass': (4e-4, 2e-4)}     # engine.py's (tau, tau_label) for reduced-pass rows
KEEPS_K5 = ('mass', 'degenerate')                               # K5b skips these and keeps K5's answers

PROFILES = {      # variables per kind
    'many': dict(argmax=800, rank=750, argmax_tie=40, zero_label=4, edge_best=2, edge_lab=2, bit1_50=2, bit1_51=2, mass=2,
                 degenerate=2, deep=1, deep_underflow=1, random=300),
    'few': dict(argmax=30, rank=30, argmax_tie=6, zero_label=2, edge_best=1, edge_lab=1, bit1_50=1, bit1_51=1, mass=1,
                degenerate=1, deep=1, deep_underflow=1, random=15),
    'small': dict(argmax=6, rank=6, argmax_tie=3, random=6),
}


def roundup(x, m):
    return (x + m - 1) // m * m


def split16(x32):
    """fp32 -> (hi, lo) fp16 as K3 / K2 split them: hi = rn(x), lo = rn(x - hi); hi + lo is exact in fp32"""
    hi = x32.astype(np.float16)
    lo = (x32 - hi.astype(np.float32)).astype(np.float16)
    return hi, lo


def _pad(x, ld, dtype):
    out = np.full((x.shape[0], ld), np.nan, dtype=dtype)
    out[:, :x.shape[1]] = x
    return out


def build_case(V, seed=0, bands='two_pass', profile='many', chunk=1024):
    rng = np.random.default_rng(seed)
    tau, tau_label = BANDS[bands]
    eps = tau / 8
    ld = roundup(V, 64)
    # ---- pairs of elements with identical table rows in every plane pair, equal constant rows and equal stored eps
    ends = rng.choice(np.arange(1, V - 1), size=6, replace=False)
    dups = [tuple(sorted(p)) for p in ends.reshape(3, 2)] + [(int(rng.integers(0, V - 8)), V - 1)]
    dup_elems = {e for p in dups for e in p}
    free_pool = np.array([e for e in range(V) if e not in dup_elems])

    # ---- variables: composition and engineering
    groups = []
    n_a = 0

    def new_group(kind, m, c, u, fp64_only=False):
        nonlocal n_a
        g = dict(kind=kind, m=m, a0=n_a, consts=list(rng.integers(1, D_CONST_ROWS, size=c)), n_uniform=u, levels={},
                 delta={}, ulink=[], uset={}, pairs=[], ties=[], eng=set(), use_stored=False, fp64_only=fp64_only,
                 alpha_shift=0, zero_rows=[])
        n_a += m
        groups.append(g)
        return g

    def small_mix(kind):
        return new_group(kind, int(rng.integers(1, 5)), int(rng.integers(0, 2)), int(rng.integers(0, 2)))

    def pick(g, k):
        cand = np.setdiff1d(free_pool, np.fromiter(g['eng'], dtype=np.int64, count=len(g['eng'])))
        e = [int(x) for x in rng.choice(cand, size=k, replace=False)]
        g['eng'].update(e)
        return e

    def margin(g):          # fp32 product and storage roundings of a pair of elements stay below this
        return max(1e-6, 4 * (g['m'] + len(g['consts']) + 2) * 2.0 ** -24)

    def loguniform(lo, hi):
        return float(np.exp(rng.uniform(np.log(lo), np.log(hi))))

    def argmax_pair(g, flip, label_is_loser=False):
        a, b = pick(g, 2)
        mg = margin(g)
        gap = loguniform(1e-6, 0.9 * (2 * eps - mg)) if flip else loguniform(1e-6, tau / 2)
        lg = float(np.log1p(gap))
        g['levels'].update({a: lg, b: 0.0})
        if flip:            # the stored rows put b above a by mg
            g['delta'].update({a: -(lg + mg) / 2, b: (lg + mg) / 2})
        else:
            g['delta'].update({a: 0.0, b: 0.0})
        g['pairs'].append((a, b, lg, flip))
        g['label'] = b if label_is_loser else pick(g, 1)[0]

    def rank_setup(g, R, n_band, flips, tie=False):
        if tie:
            pair = dups[int(rng.integers(len(dups)))]
            lab, other = pair if rng.random() < 0.5 else pair[::-1]
            g['eng'].update(pair)
            g['ulink'].append((other, lab))
            g['ties'].append(pair)
            g['delta'][lab] = 0.0
        else:
            lab = pick(g, 1)[0]
            g['delta'][lab] = 0.0
        g['label'] = lab
        g['levels'][lab] = 0.0
        for i, e in enumerate(pick(g, R)):
            g['levels'][e] = float(np.log1p(0.004 * (i + 1)))
        mg = margin(g)
        for k, e in enumerate(pick(g, n_band)):
            flip = k < flips
            sgn = 1.0 if rng.random() < 0.5 else -1.0
            gap = loguniform(1e-6, 0.9 * (eps - mg)) if flip else loguniform(1e-6, tau_label / 2)
            lg = float(np.log1p(sgn * gap))
            g['levels'][e] = lg
            g['delta'][e] = -lg - sgn * mg if flip else 0.0
            g['pairs'].append((e, lab, lg, flip))

    prof = PROFILES[profile]
    for i in range(prof.get('argmax', 0)):
        g = small_mix('argmax')
        argmax_pair(g, flip=i % 2 == 0, label_is_loser=i % 3 == 0)
    for i in range(prof.get('rank', 0)):
        g = small_mix('rank')
        rank_setup(g, R=int(rng.integers(0, min(46, V // 8))), n_band=int(rng.integers(2, 7)), flips=int(rng.integers(1, 3)),
                   tie=i % 5 == 0)
    for i in range(prof.get('argmax_tie', 0)):
        g = small_mix('argmax_tie')
        pair = dups[i % len(dups)]
        g['eng'].update(pair)
        g['levels'][pair[0]] = 0.0
        g['ulink'].append((pair[1], pair[0]))
        g['ties'].append(pair)
        g['delta'][pair[0]] = 0.0
        (c,) = pick(g, 1)
        mg = margin(g)
        gap = loguniform(1e-6, 0.9 * (eps - mg))
        lg = float(np.log1p(-gap))
        g['levels'][c] = lg
        flip = i % 2 == 0
        g['delta'][c] = -lg + mg if flip else 0.0          # flipped: the stored rows put c above the tied pair by mg
        g['pairs'].append((pair[0], c, -lg, flip))
        g['label'] = pair[1] if i % 3 == 0 else pick(g, 1)[0]
    for i in range(prof.get('zero_label', 0)):
        g = small_mix('zero_label')
        argmax_pair(g, flip=True)
        g['uset'][g['label']] = 0.0
    for kind in ('bit1_50', 'bit1_51'):
        for i in range(prof.get(kind, 0)):
            g = small_mix(kind)
            rank_setup(g, R=int(kind[-2:]), n_band=1, flips=1)
            (e, lab, lg, _), = g['pairs']
            if lg < 0:      # the neighbour is above the label in float64 and below it in fp32
                g['levels'][e] = -lg
                g['delta'][e] = lg - margin(g)
                g['pairs'][0] = (e, lab, -lg, True)
    for i in range(prof.get('edge_best', 0)):
        g = new_group('edge_best', 0, 0, 2)
        a, b = pick(g, 2)
        u_best = np.float32(1.6)
        g['uset'].update({a: u_best, b: u_best * (np.float32(1) - np.float32(tau))})
        g['label'] = pick(g, 1)[0]
        g['edge'] = (a, b)
    for i in range(prof.get('edge_lab', 0)):
        g = new_group('edge_lab', 0, 0, 0)
        lab, hi, lo = pick(g, 3)
        x = np.float32(1.2)
        g['uset'].update({lab: x, hi: x * (np.float32(1) + np.float32(tau_label)), lo: x * (np.float32(1) - np.float32(tau_label))})
        for k, e in enumerate(pick(g, 10)):
            g['uset'][e] = np.float32(1.3 + 0.02 * k)
        g['label'] = lab
        g['edge'] = (hi, lo)
    for i in range(prof.get('mass', 0)):
        g = small_mix('mass')
        for e in pick(g, 70):
            g['levels'][e] = float(rng.uniform(0, tau / 4))
        g['label'] = pick(g, 1)[0]
    for i in range(prof.get('degenerate', 0)):
        g = new_group('degenerate', 2, 0, 1)
        g['zero_rows'] = [0]
        g['use_stored'] = True
        a, b = pick(g, 2)
        g['levels'].update({a: float(np.log1p(1e-5)), b: 0.0})
        g['label'] = pick(g, 1)[0]
    for kind in ('deep', 'deep_underflow'):
        for i in range(prof.get(kind, 0)):
            g = new_group(kind, 24, 20, 20, fp64_only=kind == 'deep_underflow')
            if kind == 'deep_underflow':
                g['alpha_shift'] = -7                     # 24 rows near 2^-7: the product is ~2^-168
            argmax_pair(g, flip=True)
    for i in range(prof.get('random', 0)):
        g = new_group('random', int(rng.integers(0, 5)), int(rng.integers(0, 3)), int(rng.integers(0, 2)))
        if g['m'] + len(g['consts']) + g['n_uniform'] == 0:
            g['consts'] = [1 + i % 4]
        g['label'] = int(rng.integers(0, V))

    # ---- in_row: message rows, constant rows and uniform inputs in a random order
    n_g = len(groups)
    grp_off = [0]
    in_row = []
    for g in groups:
        rows = [D_CONST_ROWS + g['a0'] + j for j in range(g['m'])] + [int(c) for c in g['consts']] + [-1] * g['n_uniform']
        rng.shuffle(rows)
        assert len(rows) <= MAX_IN
        g['rows'] = rows
        in_row += rows
        grp_off.append(len(in_row))

    # ---- message blocks: contiguous, ascending, each table in several of them
    lens = []
    while sum(lens) < n_a:
        lens.append(int(rng.integers(1, max(2, n_a // 16) + 1)))
    lens[-1] -= sum(lens) - n_a
    tables = np.resize(np.arange(4), len(lens))
    rng.shuffle(tables)
    blocks, row_table, a = [], np.zeros(n_a, dtype=np.int64), 0
    for t, n in zip(tables, lens):
        blocks.append((int(t), a, D_CONST_ROWS + a, n))
        row_table[a:a + n] = t
        a += n

    # ---- operands: the table pool, the row maps, the A rows
    rowmap = np.stack([rng.permutation(V) for _ in range(N_PLANE_PAIRS)])
    for e1, e2 in dups:
        rowmap[:, e2] = rowmap[:, e1]
    A = (rng.random((n_a, V)) * 2.0 ** 15 / V + 2.0 ** 10 / V).astype(np.float32)
    for g in groups:
        for j in g['zero_rows']:
            A[g['a0'] + j] = 0.0
    A_hi, A_lo = split16(A)
    A_exact = A_hi.astype(np.float64) + A_lo.astype(np.float64)
    pool_hi = np.full((V, ld), np.nan, dtype=np.float16)
    pool_lo = np.full((V, ld), np.nan, dtype=np.float16)
    G = np.empty((n_a, V))                                 # G[a, j] = A row a . pool row j
    for j0 in range(0, V, chunk):
        j1 = min(V, j0 + chunk)
        h, l_ = split16((rng.random((j1 - j0, V), dtype=np.float32) * 48 + 8).astype(np.float32))
        pool_hi[j0:j1, :V], pool_lo[j0:j1, :V] = h, l_
        G[:, j0:j1] = A_exact @ (h.astype(np.float64) + l_.astype(np.float64)).T
    Dhat = np.take_along_axis(G, rowmap[row_table], axis=1) if n_a else G
    del G

    # ---- perturbations and the stored rows
    E = np.zeros((n_a, V))
    for g in groups:
        if g['m'] == 0:
            continue
        r0, r1 = g['a0'], g['a0'] + g['m']
        E[r0:r1] = rng.uniform(-1, 1, (g['m'], V)) * eps / g['m']
        for e, d in g['delta'].items():
            e = _canon(e, dups)
            E[r0:r1, e] = 0.0
            E[r0, e] = d
    for e1, e2 in dups:
        E[:, e2] = E[:, e1]
    const = rng.uniform(0.5, 1.5, (D_CONST_ROWS, V)).astype(np.float32)
    const[0] = 1.0
    for e1, e2 in dups:
        const[:, e2] = const[:, e1]
    D = np.empty((D_CONST_ROWS + n_a, V), dtype=np.float32)
    D[:D_CONST_ROWS] = const
    for g in groups:
        for j in range(g['m']):
            a = g['a0'] + j
            if j in g['zero_rows']:                        # a positive stored row over a zero A row: exact product 0
                D[D_CONST_ROWS + a] = rng.uniform(0.5, 1.5, V).astype(np.float32)
                continue
            alpha = 2.0 ** (-np.round(np.log2(Dhat[a].mean())) + g['alpha_shift'])
            D[D_CONST_ROWS + a] = (alpha * Dhat[a] * (1.0 + E[a])).astype(np.float32)
    with np.errstate(divide='ignore'):
        logd = np.log(np.concatenate([const.astype(np.float64), Dhat]))

    # ---- U: engineered levels on top of random rows
    U = rng.uniform(0.5, 1.5, (n_g, V)).astype(np.float32)
    with np.errstate(divide='ignore'):
        logD = np.log(D.astype(np.float64))
    for gi, g in enumerate(groups):
        if g['kind'] in ('edge_best', 'edge_lab'):
            U[gi] *= np.float32(0.6)                       # every other element far below the engineered ones
        src = logD if g['use_stored'] else logd
        Q = np.zeros(V)
        for r in g['rows']:
            if r >= 0:
                Q += src[r]
        if g['levels']:
            free = np.ones(V, dtype=bool)
            free[list(g['eng'])] = False
            base = (np.log(U[gi].astype(np.float64)) + Q)[free].max() + np.log(1.05)
            for e, lv in g['levels'].items():
                U[gi, e] = np.float32(np.exp(base + lv - Q[e]))
        for dst, s in g['ulink']:
            U[gi, dst] = U[gi, s]
        for e, v in g['uset'].items():
            U[gi, e] = v
    label = np.array([g['label'] for g in groups], dtype=np.int32)
    grp_u = rng.permutation(n_g + 3)[:n_g].astype(np.int32)         # variables read U rows in no particular order
    U_rows = np.full((n_g + 3, ld), np.nan, dtype=np.float32)
    U_rows[:n_g + 3, :V] = rng.uniform(0.5, 1.5, (n_g + 3, V)).astype(np.float32)
    U_rows[grp_u, :V] = U
    return dict(V=V, ld=ld, tau=tau, tau_label=tau_label, eps=eps, groups=groups, dups=dups, n_groups=n_g, n_a=n_a,
                grp_u=grp_u, grp_off=np.array(grp_off, dtype=np.int32),
                in_row=np.array(in_row if in_row else [-1], dtype=np.int32), label=label, U=U_rows,
                D=_pad(D, ld, np.float32), A_hi=_pad(A_hi, ld, np.float16), A_lo=_pad(A_lo, ld, np.float16),
                pool_hi=pool_hi, pool_lo=pool_lo, rowmap=rowmap, blocks=np.array(blocks, dtype=np.int32).reshape(-1, 4),
                row_table=row_table, logd=logd, max_in=max(len(g['rows']) for g in groups))


def _canon(e, dups):
    for e1, e2 in dups:
        if e == e2:
            return e1
    return e


def group_rows(c, g):
    return c['in_row'][c['grp_off'][g]:c['grp_off'][g + 1]][:MAX_IN]


def reference(c, g):
    """float64 log belief of variable g (-inf where a factor is 0)"""
    with np.errstate(divide='ignore'):
        L = np.log(c['U'][c['grp_u'][g], :c['V']].astype(np.float64))
    for r in group_rows(c, g):
        if r >= 0:
            L = L + c['logd'][r]
    return L


def decisions(L, lab):
    """float64 arg-max (first index on ties) and the label's rank"""
    return int(np.argmax(L)), int((L > L[lab]).sum())


def top1_ok(L, got):
    """got is the float64 arg-max, or within K5b's own error of it (never on an exact tie: the first index wins)"""
    best = int(np.argmax(L))
    return got == best or 0 < L[best] - L[got] < GAP


def rank_ok(L, lab, got):
    """got is the float64 rank up to candidates within K5b's own error of the label (exact ties never count); where both
    the reference and got are above RANK_LIMIT the value does not matter"""
    with np.errstate(invalid='ignore'):
        d = L - L[lab]
    d[lab] = 0.0
    lo = int((d >= GAP).sum())
    hi = int((d > 0).sum()) + int(((d > -GAP) & (d < 0)).sum())
    return lo <= got <= hi or (got > RANK_LIMIT and int((d > 0).sum()) > RANK_LIMIT)


def k5_model(c, g, fp64):
    """K5 (marginals_kernel) for variable g, exactly: the products in the kernel's type and order, the arg-max with the first
    index, the runner-up, the counts and the flags; plus the candidate bits K5b derives from them"""
    V = c['V']
    T = np.float64 if fp64 else np.float32
    p = c['U'][c['grp_u'][g], :V].astype(T)
    with np.errstate(under='ignore', over='ignore'):
        for r in group_rows(c, g):
            if r >= 0:
                p = p * c['D'][r, :V].astype(T)
        s = p.astype(np.float64).sum()
    ok = bool(s > 0 and np.isfinite(s))
    lab = int(c['label'][g])
    one = np.float32(1)
    plab = p[lab]
    best = p.max()
    second = np.partition(p, V - 2)[V - 2] if V > 1 else best
    best_lo = best * T(one - np.float32(c['tau']))
    lab_lo, lab_hi = plab * T(one - np.float32(c['tau_label'])), plab * T(one + np.float32(c['tau_label']))
    not_lab = np.arange(V) != lab
    icnt = int((p > plab).sum())
    inh = int(((p > plab) & (p <= lab_hi)).sum())
    inl = int(((p <= plab) & (p >= lab_lo) & not_lab).sum())
    f = 0
    if ok and V > 1 and second >= best_lo:
        f |= 1
    if ok and inh + inl > 0 and icnt - inh <= RANK_LIMIT:
        f |= 2
    b0 = (p >= best_lo) if f & 1 else np.zeros(V, dtype=bool)
    b2 = ((p >= lab_lo) & (p <= lab_hi) & not_lab) if f & 2 else np.zeros(V, dtype=bool)
    return dict(p=p, ok=ok, top1=int(np.argmax(p)) if ok else 0, rank=icnt if ok else 0, flags=f, best=float(best),
                plab=float(plab), icnt=icnt, inh=inh, inl=inl, b0=b0, b2=b2, n_cand=1 + int(((b0 | b2) & not_lab).sum()))


def planes_exact(c, table):
    """float64 (B_hi + B_lo) of plane pair `table`, [V, V] (small V only)"""
    V, rm = c['V'], c['rowmap'][table]
    return c['pool_hi'][rm, :V].astype(np.float64) + c['pool_lo'][rm, :V].astype(np.float64)


def plane_stack(c):
    """the MLBP_N_PLANES planes as one fp16 array [20, V, ld] (small V only; the GPU test gathers them on the device)"""
    return np.stack([pl[c['rowmap'][p]] for p in range(N_PLANE_PAIRS) for pl in (c['pool_hi'], c['pool_lo'])])
