"""GPU tier, kernel level: K3 (var -> factor messages), K5 edges, K6a/b/c, K1 and the small row kernels through the C ABI,
each against a plain NumPy float64 evaluation of the same operation on the same fp32 / fp16 inputs.

Every output buffer starts filled with a sentinel; after a call the values that must be written are compared with the
reference, and rows and padding columns the kernel must not write are checked to still hold the sentinel.

Tolerances are derived from the arithmetic of each kernel, with u = 2^-24 (one fp32 rounding):
  - an fp32 product of k factors carries <= k roundings; a sum of positive fp32 terms accumulated in a chain of m steps
    carries <= m roundings relative to the sum;
  - a value x split into fp16 hi + lo (mlbp.h: 2^14-scaled message rows) keeps |hi + lo - x| <= 2^-22 |x| + 2^-25: hi is
    within half an fp16 ulp (2^-11 |x|) and lo rounds that remainder to 11 bits, except that a subnormal fp16 lo has an
    absolute step of 2^-24 (error <= 2^-25)."""
import ctypes
import math
import re
import types

import numpy as np
import pytest
import torch

from macaronicusermodeling_b200 import _lib, build
from oracle import lbp_oracle as orc

pytestmark = pytest.mark.gpu

U32 = 2.0 ** -24
SPLIT_REL, SPLIT_ABS = 2.0 ** -22, 2.0 ** -25
SCALE = 2.0 ** 14                         # MLBP_A_SCALE_LOG2
SENT16 = -1.5                             # fp16 sentinel of A rows
SENT32 = -7.0                             # fp32 / fp64 sentinel
ERR_INVALID, ERR_UNSUPPORTED = 1, 3


@pytest.fixture(scope='module')
def lib():
    build.build()
    return _lib.require_device()


def P(t, byte_offset=0):
    """device pointer of a tensor; the caller keeps the tensor alive until the kernels that read it have finished"""
    return ctypes.c_void_p(t.data_ptr() + byte_offset) if t is not None else None


def S():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def roundup(x, m):
    return (x + m - 1) // m * m


def split16(x):
    """float -> (hi, lo) fp16 as the kernels split it: hi = rn(x), lo = rn(x - hi), in fp32"""
    x32 = np.asarray(x, dtype=np.float32)
    hi = x32.astype(np.float16)
    lo = (x32 - hi.astype(np.float32)).astype(np.float16)
    return hi, lo


def launched(fn, pattern):
    """names of the CUDA kernels matching `pattern` that ran inside fn() (torch.profiler, CUDA activities)"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sorted({e.name for e in prof.events() if re.search(pattern, e.name)})


# ================================================================================================ K3 mlbp_var_to_factor
K3_SMEM = 100 * 1024
K3_BUCKETS = (4, 8, 12, 16, 20, 24, 32, 48)


def k3_selection(V, max_in, range_log2, aligned=True, forced_stream=False):
    """the kernel mlbp_var_to_factor picks (mirrors the host code): ('resident', NIN, C, S) or ('stream', NMAX, T, OCC)"""
    fp32 = 0.0 <= range_log2 < 100.0
    nin = max(max_in, 1)
    if fp32 and not forced_stream and nin <= 24 and aligned:
        for c in (1, 2, 4, 8):
            s4 = (-(-V // c) + 3) & ~3
            s32 = (s4 + 31) & ~31
            if (nin + 1) * s32 * 4 <= K3_SMEM:
                return ('resident', nin, c, s32)
            if (nin + 1) * s4 * 4 <= K3_SMEM:
                return ('resident', nin, c, s4)
    nmax = next(b for b in K3_BUCKETS if max_in <= b)
    if fp32:
        return ('stream', nmax, 'float', 3 if nmax <= 20 else 1)
    return ('stream', nmax, 'double', 1)


def k3_kernel_pattern(sel):
    if sel[0] == 'resident':
        return r'var_to_factor_resident_kernel<%d>' % sel[1]
    return r'var_to_factor_kernel<%d,\s*%s,\s*%d>' % (sel[1], sel[2], sel[3])


def k3_rel_tol(sel, V):
    """fp32 products: each output <= NIN + 1 roundings (prefix, suffix, their product, the scale), each summed term <= NIN;
    the sum <= ceil(V / 256) + 5 chained fp32 roundings (per-thread chain + warp tree) before the float64 stages; the scale
    and the uniform value 1 rounding each.  fp64 products: only the final fp32 rounding of x (double arithmetic adds
    < (2 NIN + V) 2^-53).  Both then pay the fp16 hi / lo split."""
    nin = sel[1]
    if sel[0] == 'stream' and sel[2] == 'double':
        return U32 + SPLIT_REL + (2 * nin + V + 8) * 2.0 ** -53
    return (2 * nin + math.ceil(V / 256) + 8) * U32 + SPLIT_REL


def k3_case(rng, V, n_groups, max_in, counts=None, n_dest=(1,), p_uniform=0.0, lo=0.5, hi=1.5, u_scale=1.0,
            d_scale=1.0, spare_a_rows=7):
    """n_groups (variable, level) groups; group g has counts[g] inputs (default max_in), each input a distinct D row
    (in_row < 0 with probability p_uniform) with a number of destinations drawn from n_dest, scattered over the A rows."""
    ld = roundup(V, 64)
    counts = np.full(n_groups, max_in) if counts is None else np.asarray(counts)
    assert counts.max() <= max_in
    n_in = int(counts.sum())
    grp_off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    n_d = 1 + n_in + 2
    D = np.full((n_d, ld), np.nan, dtype=np.float32)             # row padding is never read: poisoned
    D[:, :V] = (rng.uniform(lo, hi, (n_d, V)) * d_scale).astype(np.float32)
    D[0] = 1.0                                                     # the constant-one row of the uniform inputs
    in_row = (1 + rng.permutation(n_in + 2)[:n_in]).astype(np.int32)
    in_row[rng.random(n_in) < p_uniform] = -1
    n_u = n_groups + 3
    U = np.full((n_u, ld), np.nan, dtype=np.float32)
    U[:, :V] = (rng.uniform(lo, hi, (n_u, V)) * u_scale).astype(np.float32)
    grp_u = rng.permutation(n_u)[:n_groups].astype(np.int32)
    nd = rng.choice(np.asarray(n_dest), size=n_in).astype(np.int32)
    dest_off = np.concatenate([[0], np.cumsum(nd)]).astype(np.int32)
    n_a = int(nd.sum()) + spare_a_rows
    dest = rng.permutation(n_a)[:int(nd.sum())].astype(np.int32)
    first = np.array([dest[dest_off[i]] if nd[i] > 0 else -1 for i in range(n_in)], dtype=np.int32)
    second = np.array([dest[dest_off[i] + 1] if nd[i] > 1 else -1 for i in range(n_in)], dtype=np.int32)
    return dict(V=V, ld=ld, max_in=max_in, grp_u=grp_u, grp_off=grp_off, in_row=in_row, dest_off=dest_off,
                dest=np.concatenate([dest, [-1]]).astype(np.int32), first=first, second=second, U=U, D=D, n_a=n_a,
                n_groups=n_groups)


def k3_reference(c):
    """A row -> float64 message: x = 2^14 U[u] prod_{j != i} D[in_row[j]] / sum(...), in_row < 0 = a row of ones,
    sum <= 0 or non-finite -> 2^14 / V"""
    V = c['V']
    U64, D64 = c['U'][:, :V].astype(np.float64), c['D'][:, :V].astype(np.float64)
    want = {}
    with np.errstate(invalid='ignore', over='ignore'):
        for g in range(c['n_groups']):
            i0, i1 = c['grp_off'][g], c['grp_off'][g + 1]
            rows = np.stack([D64[r] if r >= 0 else np.ones(V) for r in c['in_row'][i0:i1]]) if i1 > i0 else np.ones((0, V))
            for k, i in enumerate(range(i0, i1)):
                dsts = c['dest'][c['dest_off'][i]:c['dest_off'][i + 1]]
                if len(dsts) == 0:
                    continue
                p = U64[c['grp_u'][g]] * np.prod(np.delete(rows, k, axis=0), axis=0)
                t = p.sum()
                x = SCALE * p / t if (t > 0 and np.isfinite(t)) else np.full(V, SCALE / V)
                for d in dsts:
                    want[int(d)] = x
    return want


def run_k3(lib, c, range_log2, u_off=0, d_off=0, max_in=None):
    """one mlbp_var_to_factor call; u_off / d_off shift the U / D base by that many floats (misaligned bases).
    Returns (rc, hi, lo) as float64 arrays [n_a, ld]."""
    V, ld = c['V'], c['ld']
    Ub = torch.full((u_off + c['U'].size,), float('nan'), dtype=torch.float32, device='cuda')
    Ub[u_off:] = dev(c['U'].ravel())
    Db = torch.full((d_off + c['D'].size,), float('nan'), dtype=torch.float32, device='cuda')
    Db[d_off:] = dev(c['D'].ravel())
    hi = torch.full((c['n_a'], ld), SENT16, dtype=torch.float16, device='cuda')
    lo = torch.full((c['n_a'], ld), SENT16, dtype=torch.float16, device='cuda')
    ints = [dev(c[k]) for k in ('grp_u', 'grp_off', 'in_row', 'dest_off', 'dest', 'first', 'second')]
    rc = lib.mlbp_var_to_factor(c['n_groups'], *[P(t) for t in ints], P(Ub, 4 * u_off), P(Db, 4 * d_off), c.get('ldv', ld), V,
                                P(hi), P(lo), c['max_in'] if max_in is None else max_in, range_log2, S())
    torch.cuda.synchronize()
    return rc, hi.cpu().numpy().astype(np.float64), lo.cpu().numpy().astype(np.float64)


def check_k3(c, hi, lo, rel):
    V = c['V']
    want = k3_reference(c)
    for r in range(c['n_a']):
        if r not in want:
            assert (hi[r] == SENT16).all() and (lo[r] == SENT16).all(), 'A row %d is no destination but was written' % r
            continue
        x = want[r]
        got = hi[r, :V] + lo[r, :V]
        err = np.abs(got - x)
        bound = rel * np.abs(x) + SPLIT_ABS
        assert (err <= bound).all(), 'row %d col %d: got %r want %r (rel tol %.3g)' % (
            r, int(np.argmax(err - bound)), got[np.argmax(err - bound)], x[np.argmax(err - bound)], rel)
        # every emitted row sums to 2^14 (the one-pass residual GEMM's add_const assumes it)
        assert abs(got.sum() - SCALE) <= rel * SCALE + V * SPLIT_ABS, (r, got.sum())
        assert (hi[r, V:] == SENT16).all() and (lo[r, V:] == SENT16).all(), 'row padding of A row %d was written' % r
    return want


def k3_run_checked(lib, c, range_log2, forced_stream=False, **kw):
    sel = k3_selection(c['V'], c['max_in'], range_log2, aligned=not (kw.get('u_off', 0) % 4 or kw.get('d_off', 0) % 4),
                       forced_stream=forced_stream)
    out = {}

    def call():
        out['r'] = run_k3(lib, c, range_log2, **kw)
    names = launched(call, r'var_to_factor')
    assert len(names) == 1 and re.search(k3_kernel_pattern(sel), names[0]), (sel, names)
    rc, hi, lo = out['r']
    assert rc == 0, _lib.load().mlbp_last_error()
    check_k3(c, hi, lo, k3_rel_tol(sel, c['V']))
    return sel, hi, lo


@pytest.mark.parametrize('V,max_in,C,slice_cols', [(1000, 19, 1, 1024), (2000, 19, 2, 1024), (4000, 19, 4, 1024), (10000, 19, 8, 1280),
                                          (3650, 6, 1, 3652), (4001, 19, 4, 1024), (10000, 24, 0, 0)])
def test_k3_resident_cluster_sizes(lib, V, max_in, C, slice_cols):
    """resident kernel at cluster sizes 1 / 2 / 4 / 8, a slice that is not a multiple of 32 (3652), an odd last slice
    (V = 4001: 929 columns), and a shape whose slices do not fit (streams)"""
    sel = k3_selection(V, max_in, 60.0)
    assert sel == (('resident', max_in, C, slice_cols) if C else ('stream', 24, 'float', 1))
    if C:
        last = V - (C - 1) * slice_cols
        assert last > 0 and (V != 4001 or last % 2 == 1)
    rng = np.random.default_rng(V + max_in)
    c = k3_case(rng, V, 6, max_in, counts=[max_in, max_in - 1, max_in, 1, max_in - 3, max_in], n_dest=(0, 1, 1, 2, 3))
    k3_run_checked(lib, c, 60.0)


@pytest.mark.parametrize('nin', list(range(1, 25)))
def test_k3_resident_every_nin(lib, nin):
    rng = np.random.default_rng(100 + nin)
    V = 300 + nin
    counts = [nin, max(nin - 1, 0), nin, 1 if nin > 1 else 0, nin]
    c = k3_case(rng, V, 5, nin, counts=counts, n_dest=(0, 1, 1, 2, 3, 5), p_uniform=0.15)
    sel, _, _ = k3_run_checked(lib, c, 60.0)
    assert sel[:3] == ('resident', nin, 1)


@pytest.mark.parametrize('fp64', [False, True], ids=['fp32', 'fp64'])
@pytest.mark.parametrize('max_in', [3, 8, 11, 16, 17, 24, 29, 48])
def test_k3_streaming_every_bucket(lib, monkeypatch, max_in, fp64):
    """the two-read kernel in every NMAX bucket (4 .. 48), fp32 (MLBP_K3_IMPL=1) and fp64 products (range_log2 < 0)"""
    monkeypatch.setenv('MLBP_K3_IMPL', '1')
    rng = np.random.default_rng(200 + max_in + 50 * fp64)
    V = 1000 + max_in
    counts = [max_in, max_in - 1, 2, max_in, 0, max_in - 2]
    c = k3_case(rng, V, 6, max_in, counts=counts, n_dest=(0, 1, 2, 3, 5), p_uniform=0.1)
    sel, _, _ = k3_run_checked(lib, c, -1.0 if fp64 else 60.0, forced_stream=True)
    assert sel[0] == 'stream' and sel[1] == next(b for b in K3_BUCKETS if max_in <= b)


@pytest.mark.parametrize('which', ['U', 'D'])
def test_k3_misaligned_base_streams(lib, which):
    """a U or D base that is 4 bytes off a 16-byte boundary (ldv % 4 == 0 still holds) takes the streaming kernel with the
    same results"""
    rng = np.random.default_rng(7)
    c = k3_case(rng, 2000, 8, 6, n_dest=(1, 2))
    sel_al, hi_al, lo_al = k3_run_checked(lib, c, 60.0)
    assert sel_al[0] == 'resident'
    sel, hi, lo = k3_run_checked(lib, c, 60.0, **({'u_off': 1} if which == 'U' else {'d_off': 1}))
    assert sel == ('stream', 8, 'float', 3)
    rel = k3_rel_tol(sel, c['V']) + k3_rel_tol(sel_al, c['V'])
    m = hi_al != SENT16
    assert (np.abs((hi + lo)[m] - (hi_al + lo_al)[m]) <= rel * np.abs(hi_al + lo_al)[m] + 2 * SPLIT_ABS).all()


@pytest.mark.parametrize('path', ['resident', 'stream32', 'stream64'])
def test_k3_group_structure(lib, monkeypatch, path):
    """several hundred groups (each persistent resident cluster runs the double-buffered partial-sum exchange many times),
    groups with fewer inputs than max_in (also none), and inputs with 0, 1, 2, 3 and 5 scattered destinations"""
    if path == 'stream32':
        monkeypatch.setenv('MLBP_K3_IMPL', '1')
    rng = np.random.default_rng(11)
    V, max_in, n_groups = 4001, 12, 500
    counts = rng.integers(0, max_in + 1, size=n_groups)
    counts[::7] = max_in
    c = k3_case(rng, V, n_groups, max_in, counts=counts, n_dest=(0, 1, 1, 1, 2, 2, 3, 5), p_uniform=0.1, spare_a_rows=40)
    nd = np.diff(c['dest_off'])
    assert {0, 1, 2, 3, 5} <= set(nd.tolist())
    sel, _, _ = k3_run_checked(lib, c, -1.0 if path == 'stream64' else 60.0, forced_stream=path == 'stream32')
    assert sel[0] == ('resident' if path == 'resident' else 'stream')
    if path == 'resident':
        assert sel[2] == 4


@pytest.mark.parametrize('path', ['resident', 'stream32', 'stream64'])
def test_k3_renormalisation_edges(lib, monkeypatch, path):
    """an all-zero U row (every sum is 0 -> uniform), and one input row holding a NaN and a +inf: only the leave-one-out
    product that excludes that row stays finite, the group's other messages fall back to uniform"""
    if path == 'stream32':
        monkeypatch.setenv('MLBP_K3_IMPL', '1')
    rng = np.random.default_rng(13)
    V = 2001
    c = k3_case(rng, V, 4, 5, n_dest=(1, 2))
    c['U'][c['grp_u'][0], :V] = 0.0
    bad = c['in_row'][c['grp_off'][1] + 2]
    c['D'][bad, 17] = np.nan
    c['D'][bad, 1500] = np.inf
    _, hi, lo = k3_run_checked(lib, c, -1.0 if path == 'stream64' else 60.0, forced_stream=path == 'stream32')
    uni = np.float64(np.float32(SCALE) / np.float32(V))
    for g, finite_k in ((0, None), (1, 2)):
        for k, i in enumerate(range(c['grp_off'][g], c['grp_off'][g + 1])):
            for d in c['dest'][c['dest_off'][i]:c['dest_off'][i + 1]]:
                row = hi[d, :V] + lo[d, :V]
                if k == finite_k:
                    assert np.isfinite(row).all() and np.ptp(row) > 0
                else:
                    assert np.abs(row - uni).max() <= SPLIT_REL * uni + SPLIT_ABS, (g, k)


@pytest.mark.parametrize('range_log2', [200.0, -1.0])
@pytest.mark.parametrize('n_in', [3, 4])
@pytest.mark.parametrize('target', ['above-2^170', 'below-2^-120', 'near-2^150'])
def test_k3_fp64_extreme_magnitudes(lib, target, n_in, range_log2):
    """the fp64 product path with leave-one-out sums t far outside the fp32 range: U and D entries near 2^+-60 (fp32 inputs)
    put t above 2^170, where a float normaliser 2^14 / t is 0, and below 2^-120, where it is +inf; near 2^150 it is a
    subnormal float with ~13 bits.  The fp64 variant is the always-safe fallback for range_log2 >= 100 or unknown, so these
    messages must be as accurate as any other."""
    mag = {'above-2^170': 60, 'below-2^-120': -60, 'near-2^150': 140 // n_in}[target]
    rng = np.random.default_rng(300 + mag + n_in)
    V = 1500
    c = k3_case(rng, V, 3, n_in, n_dest=(1, 2), u_scale=2.0 ** mag, d_scale=2.0 ** mag)
    loo = c['U'][c['grp_u'][0], :V].astype(np.float64) * np.prod(c['D'][c['in_row'][1:n_in], :V].astype(np.float64), axis=0)
    lg = math.log2(loo.sum())
    assert {'above-2^170': lg > 170, 'below-2^-120': lg < -120, 'near-2^150': 141 < lg < 163}[target], lg
    sel, _, _ = k3_run_checked(lib, c, range_log2)
    assert sel == ('stream', 4, 'double', 1)


@pytest.mark.parametrize('path', ['resident', 'stream64'])
def test_k3_deterministic(lib, path):
    rng = np.random.default_rng(17)
    c = k3_case(rng, 10000, 300, 8, counts=rng.integers(1, 9, size=300), n_dest=(1, 2, 3))
    r1 = run_k3(lib, c, 60.0 if path == 'resident' else -1.0)
    r2 = run_k3(lib, c, 60.0 if path == 'resident' else -1.0)
    assert r1[0] == 0 and r2[0] == 0
    assert np.array_equal(r1[1], r2[1]) and np.array_equal(r1[2], r2[2])
    assert (r1[1] != SENT16).any()


def test_k3_refused_calls_leave_buffers(lib):
    rng = np.random.default_rng(19)
    c = k3_case(rng, 1000, 2, 4)
    rc, hi, lo = run_k3(lib, c, 60.0, max_in=49)
    assert rc == ERR_UNSUPPORTED and (hi == SENT16).all() and (lo == SENT16).all()
    c['ldv'] = c['V'] + 2                                          # ldv >= V but not a multiple of 4
    rc, hi, lo = run_k3(lib, c, 60.0)
    assert rc == ERR_INVALID and (hi == SENT16).all() and (lo == SENT16).all()


# ================================================================================================ K5 mlbp_marginals edges
def k5_reference(c, labels):
    V = c['V']
    U64, D64 = c['U'][:, :V].astype(np.float64), c['D'][:, :V].astype(np.float64)
    out = []
    for g in range(c['n_groups']):
        p = U64[c['grp_u'][g]].copy()
        for r in c['in_row'][c['grp_off'][g]:c['grp_off'][g + 1]]:
            if r >= 0:
                p = p * D64[r]
        s = p.sum()
        ok = s > 0 and np.isfinite(s)
        b = p / s if ok else np.full(V, 1.0 / V)
        lab = labels[g]
        out.append(dict(p=p, b=b, ok=ok, logp=np.log(b[lab]) if b[lab] > 0 else -99.99,
                        top1=int(np.argmax(b)) if ok else 0, rank=int((b > b[lab]).sum()) if ok else 0))
    return out


def run_k5(lib, c, labels, range_log2, vec=True, max_in=None):
    V, ld, n = c['V'], c['ld'], c['n_groups']
    ints = [dev(c[k]) for k in ('grp_u', 'grp_off', 'in_row')]
    lab = dev(np.asarray(labels, dtype=np.int32))
    logp = torch.full((n,), SENT32, dtype=torch.float64, device='cuda')
    top1 = torch.full((n,), -5, dtype=torch.int32, device='cuda')
    rank = torch.full((n,), -5, dtype=torch.int32, device='cuda')
    bel = torch.full((n * ld + 4,), SENT32, dtype=torch.float32, device='cuda')
    off = 0 if vec else 4                                          # 4 bytes off 16: the element-wise variant
    tU, tD = dev(c['U']), dev(c['D'])
    rc = lib.mlbp_marginals(n, *[P(t) for t in ints], P(lab), P(tU), P(tD), ld, V, P(logp), P(top1), P(rank),
                            P(bel, off), range_log2, c['max_in'] if max_in is None else max_in, 0.0, 0.0,
                            None, None, None, None, None, S())
    torch.cuda.synchronize()
    B = bel.cpu().numpy()[off // 4:off // 4 + n * ld].reshape(n, ld)
    return rc, logp.cpu().numpy(), top1.cpu().numpy(), rank.cpu().numpy(), B


def k5_case(rng, V, max_in, dyadic):
    c = k3_case(rng, V, 10, max_in, counts=[max_in, max_in, 1, max_in - 1, max_in, max_in, 0, max_in, max_in, max_in],
                p_uniform=0.2)
    if dyadic:                                                     # exact products and sums in fp32: every decision is exact
        c['U'][:, :V] = rng.integers(1, 9, size=(c['U'].shape[0], V)) / 8.0
        c['D'][1:, :V] = rng.integers(2, 7, size=(c['D'].shape[0] - 1, V)) / 4.0
    labels = rng.integers(0, V, size=10)
    g = 1                                                          # an exact tie of the arg-max (two threads / warps)
    for a, b in ((5, 900),):
        c['U'][c['grp_u'][g], [a, b]] = 1024.0
        for r in c['in_row'][c['grp_off'][g]:c['grp_off'][g + 1]]:
            if r >= 0:
                c['D'][r, b] = c['D'][r, a]
    labels[g] = 900
    c['U'][c['grp_u'][4], :V] = 0.0                                # a zero product sum
    c['U'][c['grp_u'][5], labels[5]] = 0.0                         # a zero label belief
    g = 7                                                          # a tie of the arg-max inside one thread's four columns
    c['U'][c['grp_u'][g], [8, 9]] = 1024.0
    for r in c['in_row'][c['grp_off'][g]:c['grp_off'][g + 1]]:
        if r >= 0:
            c['D'][r, 9] = c['D'][r, 8]
    labels[7] = 8
    c['in_row'][c['grp_off'][8]:c['grp_off'][9]] = -1              # every input still uniform
    return c, labels


@pytest.mark.parametrize('fp64', [False, True], ids=['fp32', 'fp64'])
def test_k5_marginals_match_float64(lib, fp64):
    """fp32 and fp64 products against float64, with uniform inputs (dropped), exact arg-max ties (first index), a zero
    product sum (uniform beliefs, logp = log(1/V), top1 = rank = 0) and a zero label belief (logp = -99.99)"""
    rng = np.random.default_rng(23 + fp64)
    V, max_in = 1001, 5
    c, labels = k5_case(rng, V, max_in, dyadic=False)
    rc, logp, top1, rank, B = run_k5(lib, c, labels, -1.0 if fp64 else 50.0)
    assert rc == 0
    # fp32: each product <= max_in + 1 roundings; the sum a per-thread chain of <= 4 ceil(V / 1024) terms plus the block
    # tree (float64 after the warp); the belief one more rounding.  fp64: only the final fp32 rounding of the belief.
    rel_p = 0.0 if fp64 else (max_in + 1) * U32
    rel = rel_p + (U32 if fp64 else (max_in + 1 + 4 * math.ceil(V / 1024) + 8) * U32) + 2.0 ** -50
    ref = k5_reference(c, labels)
    for g, r in enumerate(ref):
        assert abs(logp[g] - r['logp']) <= 2 * rel, (g, logp[g], r['logp'])
        assert np.abs(B[g, :V] - r['b']).max() <= rel * r['b'].max() + 1e-45, g
        assert (B[g, V:] == SENT32).all(), 'belief row padding was written'
        b = r['b']
        band = 2 * rel_p + 2.0 ** -50
        assert r['ok'] or (top1[g] == 0 and rank[g] == 0)
        if r['ok']:
            assert b[top1[g]] >= b.max() * (1 - band), g
            lo_, hi_ = int((b > b[labels[g]] * (1 + band)).sum()), int((b > b[labels[g]] * (1 - band)).sum())
            assert lo_ <= rank[g] <= hi_, (g, rank[g], lo_, hi_)
    assert top1[1] == 5 and rank[1] == 0 and top1[7] == 8 and rank[7] == 0     # exact ties: the first index, not counted
    assert not ref[4]['ok'] and abs(logp[4] - math.log(1.0 / V)) <= 2 * rel and (B[4, :V] == np.float32(1.0) / np.float32(V)).all()
    assert logp[5] == -99.99 and rank[5] == int((ref[5]['b'] > 0).sum())


@pytest.mark.parametrize('fp64', [False, True], ids=['fp32', 'fp64'])
def test_k5_vector_and_scalar_variants_agree(lib, fp64):
    """the 16-byte-load variant and the element-wise one (beliefs 4 bytes off alignment) are bit-identical, and exact on
    inputs whose products and sums fp32 represents exactly (eighths times quarters: every decision, tie and rank is exact)"""
    rng = np.random.default_rng(29)
    V, max_in = 1001, 3
    c, labels = k5_case(rng, V, max_in, dyadic=True)
    rv = run_k5(lib, c, labels, -1.0 if fp64 else 50.0, vec=True)
    rs = run_k5(lib, c, labels, -1.0 if fp64 else 50.0, vec=False)
    assert rv[0] == 0 and rs[0] == 0
    for a, b in zip(rv[1:], rs[1:]):
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
    ref = k5_reference(c, labels)
    _, logp, top1, rank, B = rv
    for g, r in enumerate(ref):
        assert top1[g] == r['top1'] and rank[g] == r['rank'], (g, top1[g], r['top1'], rank[g], r['rank'])
        assert abs(logp[g] - r['logp']) <= 1e-15 * abs(r['logp']) + 1e-15, g   # exact p / s, then one float64 log
        assert np.abs(B[g, :V] - r['b']).max() <= U32 * r['b'].max(), g


def test_k5_max_in_limit(lib):
    """64 incoming messages are accepted (and all of them multiplied), 65 are refused with the outputs untouched"""
    rng = np.random.default_rng(31)
    V = 200
    c = k3_case(rng, V, 2, 64, counts=[64, 30], lo=0.9, hi=1.1)
    labels = [3, 150]
    rc, logp, top1, rank, B = run_k5(lib, c, labels, 50.0)
    assert rc == 0
    rel = (65 + 4 + 8 + 1) * U32
    for g, r in enumerate(k5_reference(c, labels)):
        assert np.abs(B[g, :V] - r['b']).max() <= rel * r['b'].max()
        assert abs(logp[g] - r['logp']) <= 2 * rel
    c['max_in'] = 65
    rc, logp, top1, rank, B = run_k5(lib, c, labels, 50.0)
    assert rc == ERR_UNSUPPORTED
    assert (logp == SENT32).all() and (top1 == -5).all() and (rank == -5).all() and (B == SENT32).all()


# ================================================================================================ K6a mlbp_pair_expectations
def k6a_setup(rng, V):
    ld = roundup(V, 64)
    n_a, n_d = 12, 10
    A = rng.random((n_a, V)) * SCALE / V * 2
    h, l = split16(A)
    Ah = np.full((n_a, ld), np.nan, dtype=np.float16)             # the padding of A rows is never written: poisoned
    Al = np.full((n_a, ld), np.nan, dtype=np.float16)
    Ah[:, :V], Al[:, :V] = h, l
    D = np.zeros((n_d, ld), dtype=np.float32)                      # the GEMM writes D padding as zero
    D[:, :V] = rng.uniform(0.5, 1.5, (n_d, V)).astype(np.float32)
    return ld, Ah, Al, D


def k6a_base(Ah, Al, D, V, fac):
    c = lambda r: Ah[r, :V].astype(np.float64) + Al[r, :V].astype(np.float64)
    Dx = D[:, :V].astype(np.float64)
    out = []
    for cr, zr, u0, u1, u2 in fac:
        out.append([c(zr) @ Dx[u0], c(cr) @ Dx[u1], c(cr) @ Dx[u2] if u2 >= 0 else 0.0])
    return np.array(out)


FACTORS = [  # c_row, z_row, u0, u1, u2, r_row, gap1
    (1, 1, 2, 3, 4, 5, 1),    # z_row == c_row, gap 1
    (2, 6, 5, 6, -1, 6, 0),   # z_row != c_row, no u2
    (3, 3, 7, 8, -1, 9, 0),   # z_row == c_row, gap > 1
    (7, 8, 1, 9, 0, 8, 1),    # z_row != c_row, gap 1
    (10, 10, 0, 2, 3, 11, 0),  # the r row has no spikes
]


def run_k6a(lib, Ah, Al, D, V, ld, fac, spikes=None, alpha=1.0):
    cols = list(zip(*fac))
    ints = [dev(np.asarray(x, dtype=np.int32)) for x in cols]
    stats = torch.full((len(fac), 3), SENT32, dtype=torch.float64, device='cuda')
    tA, tL, tD = dev(Ah), dev(Al), dev(D)
    if spikes is None:
        rc = lib.mlbp_pair_expectations(len(fac), *[P(t) for t in ints[:5]], P(tA), P(tL), P(tD), ld, V, P(stats),
                                        None, None, None, None, None, None, 0, 0.0, S())
    else:
        words, cnt, ent, planes = [dev(x) for x in spikes]
        rc = lib.mlbp_pair_expectations(len(fac), *[P(t) for t in ints[:5]], P(tA), P(tL), P(tD), ld, V, P(stats),
                                        P(ints[5]), P(ints[6]), P(words), P(cnt), P(ent), P(planes), V * ld, alpha, S())
    torch.cuda.synchronize()
    return rc, stats.cpu().numpy()


def k6a_rel(V):
    """c = hi + lo in fp32 (one rounding), fp32 fma chains of 8 ceil(V / 2048) positive terms per thread, float64 after"""
    return (8 * math.ceil(V / 2048) + 4) * U32


@pytest.mark.parametrize('V', [1001, 2048, 4099])
def test_k6a_pair_expectations(lib, V):
    """{z . u0, c . u1, c . u2} from hi + lo for z_row == / != c_row, u2_row < 0, V not a multiple of 8 with NaN A padding"""
    rng = np.random.default_rng(V)
    ld, Ah, Al, D = k6a_setup(rng, V)
    fac = [f[:5] for f in FACTORS]
    rc, st = run_k6a(lib, Ah, Al, D, V, ld, [f + (0, 0) for f in fac])
    assert rc == 0
    want = k6a_base(Ah, Al, D, V, fac)
    assert np.all(np.abs(st - want) <= k6a_rel(V) * np.abs(want))
    assert st[1, 2] == 0.0 and st[2, 2] == 0.0


def test_k6a_spike_cells(lib):
    """one-pass gradient rows: the kernel adds alpha c[a] r_hi[b] B_lo[a, b] for every pair of spikes of the c and r rows, with
    B the T / G / G1w lo planes of the factor's gap class; a set PEAK word (or no spike lists) disables it"""
    rng = np.random.default_rng(41)
    V = 1001
    ld, Ah, Al, D = k6a_setup(rng, V)
    spikes_of = {1: [3, 500], 5: [7, 8, 1000], 2: [999], 6: [0, 64, 65, 66], 3: [11], 9: [12], 7: [4, 900], 8: [4],
                 10: [50]}
    words = np.zeros(5, dtype=np.int32)
    cnt = np.zeros(12, dtype=np.int32)
    ent = np.zeros((12, 4, 2), dtype=np.int32)
    for r, cols in spikes_of.items():
        for i, col in enumerate(cols):
            Ah[r, col], Al[r, col] = split16(SCALE * (0.05 + 0.01 * i))
            ent[r, i, 0] = col
            ent[r, i, 1] = int(np.float32(Al[r, col]).view(np.int32))
        cnt[r] = len(cols)
    planes = np.zeros((20, V, ld), dtype=np.float16)
    for t in (0, 2, 4, 5, 6):                                      # lo planes of T, T1, G, G1, G1w
        planes[2 * t + 1, :, :V] = (2.0 ** -6 + rng.random((V, V)) * 2.0 ** -4).astype(np.float16)
    alpha = 2.0 ** -9
    fac = [f[:5] for f in FACTORS]
    base = k6a_base(Ah, Al, D, V, fac)
    rc, st = run_k6a(lib, Ah, Al, D, V, ld, FACTORS, spikes=(words, cnt, ent, planes), alpha=alpha)
    assert rc == 0
    want = base.copy()
    cx = lambda r, k: float(Ah[r, k]) + float(Al[r, k])
    for f, (cr, zr, u0, u1, u2, rr, g1) in enumerate(FACTORS):
        for a in spikes_of.get(cr, [])[:4]:
            for b in spikes_of.get(rr, [])[:4]:
                w = alpha * cx(cr, a) * float(Ah[rr, b])
                if zr == cr:               # z_row != c_row: Z is NOT corrected (the kernel only restores Z = c . T r)
                    want[f, 0] += w * float(planes[2 * (2 if g1 else 0) + 1, a, b])
                want[f, 1] += w * float(planes[2 * (5 if g1 else 4) + 1, a, b])
                if u2 >= 0:
                    want[f, 2] += w * float(planes[2 * 6 + 1, a, b])
    rel = k6a_rel(V)
    assert np.all(np.abs(st - want) <= rel * np.abs(want) + 1e-300)
    moved = np.abs(want - base) > 100 * rel * np.abs(base)
    assert moved[0].all() and moved[1, 1] and moved[2, :2].all() and moved[3, 1:].all()   # the corrections are visible
    assert not moved[1, 0] and not moved[3, 0] and not moved[4].any()
    words[0] = 1                                                   # PEAK: the gradient rows ran two passes, nothing to restore
    rc, st = run_k6a(lib, Ah, Al, D, V, ld, FACTORS, spikes=(words, cnt, ent, planes), alpha=alpha)
    assert rc == 0 and np.all(np.abs(st - base) <= rel * np.abs(base))


# ================================================================================================ K6b / K6c
def test_k6b_gradient_reduce(lib):
    """sentences with 0 variables / 0 factors / more than 32 of each (lane striding), Z <= 0 (expectations 0, bias +1),
    factors with and without gap1; float64 throughout (1e-12 relative to the sum of magnitudes)"""
    rng = np.random.default_rng(43)
    V, ldf = 300, 320
    nv_s = [3, 0, 40, 5, 70, 1]
    nf_s = [2, 0, 0, 37, 65, 0]
    sv = np.concatenate([[0], np.cumsum(nv_s)]).astype(np.int32)
    sf = np.concatenate([[0], np.cumsum(nf_s)]).astype(np.int32)
    nv, nf = int(sv[-1]), int(sf[-1])
    g_un = rng.normal(size=(nv, 9))
    stats = np.abs(rng.normal(size=(nf, 3))) + 0.1
    stats[::5, 0] = 0.0
    stats[1::7, 0] = -1.0
    label = rng.integers(0, V, size=nv).astype(np.int32)
    v0 = np.zeros(nf, dtype=np.int32)
    v1 = np.zeros(nf, dtype=np.int32)
    for s in range(len(nv_s)):
        if nf_s[s]:
            v0[sf[s]:sf[s + 1]] = rng.integers(sv[s], sv[s + 1], size=nf_s[s])
            v1[sf[s]:sf[s + 1]] = rng.integers(sv[s], sv[s + 1], size=nf_s[s])
    gap1 = (rng.random(nf) < 0.5).astype(np.int32)
    pmi = np.full((V, ldf), np.nan, dtype=np.float32)
    w1 = np.full((V, ldf), np.nan, dtype=np.float32)
    pmi[:, :V] = rng.random((V, V))
    w1[:, :V] = rng.random((V, V))
    logp_v = -rng.random(nv) * 10
    want = np.zeros((len(nv_s), 9))
    mag = np.zeros((len(nv_s), 9))
    want_lp = np.array([logp_v[sv[s]:sv[s + 1]].sum() for s in range(len(nv_s))])
    for s in range(len(nv_s)):
        want[s] = g_un[sv[s]:sv[s + 1]].sum(0)
        mag[s] = np.abs(g_un[sv[s]:sv[s + 1]]).sum(0)
        for f in range(sf[s], sf[s + 1]):
            z = stats[f, 0]
            a, b = label[v0[f]], label[v1[f]]
            e1 = stats[f, 1] / z if z > 0 else 0.0
            want[s, 0] += float(pmi[a, b]) - e1
            mag[s, 0] += abs(float(pmi[a, b])) + abs(e1)
            if gap1[f]:
                e2 = stats[f, 2] / z if z > 0 else 0.0
                want[s, 1] += float(w1[a, b]) - e2
                mag[s, 1] += abs(float(w1[a, b])) + abs(e2)
            want[s, 2] += 0.0 if z > 0 else 1.0
            mag[s, 2] += 1.0
    ns = len(nv_s)
    t = {k: dev(x) for k, x in dict(sv=sv, sf=sf, g=g_un, st=stats, v0=v0, v1=v1, lab=label, gap=gap1, pmi=pmi, w1=w1,
                                    lp=logp_v).items()}
    grad = torch.full((ns, 9), SENT32, dtype=torch.float64, device='cuda')
    lps = torch.full((ns + 1,), SENT32, dtype=torch.float64, device='cuda')
    _lib.check(lib.mlbp_gradient_reduce(ns, P(t['sv']), P(t['sf']), P(t['g']), P(t['st']), P(t['v0']), P(t['v1']), P(t['lab']),
                                        P(t['gap']), P(t['pmi']), P(t['w1']), ldf, P(t['lp']), P(grad), P(lps), S()))
    torch.cuda.synchronize()
    G, L = grad.cpu().numpy(), lps.cpu().numpy()
    assert np.all(np.abs(G - want) <= 1e-12 * mag + 1e-300)
    assert np.all(np.abs(L[:ns] - want_lp) <= 1e-12 * np.abs(logp_v).sum()) and L[ns] == SENT32
    assert (G[1] == 0).all() and L[1] == 0.0
    # sent_fac_off and logp_var NULL: the unary terms only, log-posteriors 0
    grad.fill_(SENT32); lps.fill_(SENT32)
    _lib.check(lib.mlbp_gradient_reduce(ns, P(t['sv']), None, P(t['g']), None, None, None, None, None, P(t['pmi']), P(t['w1']),
                                        ldf, None, P(grad), P(lps), S()))
    torch.cuda.synchronize()
    want_u = np.array([g_un[sv[s]:sv[s + 1]].sum(0) for s in range(ns)])
    mag_u = np.array([np.abs(g_un[sv[s]:sv[s + 1]]).sum(0) for s in range(ns)])
    assert np.all(np.abs(grad.cpu().numpy() - want_u) <= 1e-12 * mag_u + 1e-300)
    assert (lps.cpu().numpy()[:ns] == 0.0).all()


def test_k6c_batch_reduce(lib):
    """more than 1 024 sentences (block striding), ranks at the P@0 / P@25 / P@50 edges, two calls accumulating into out16,
    the maximum of the peak-flag code, and NULL arguments"""
    rng = np.random.default_rng(47)
    ns, nv = 2500, 3001
    grad = rng.normal(size=(ns, 9))
    lps = -rng.random(ns) * 30
    rank = rng.integers(0, 200, size=nv).astype(np.int32)
    rank[:10] = [0, 25, 26, 49, 50, 0, 25, 26, 49, 50]
    out0 = rng.normal(size=16)
    out0[15] = 1.0
    t_g, t_l, t_r = dev(grad), dev(lps), dev(rank)
    out = dev(out0)
    words = dev(np.array([0, 0, 0, 1, 0], dtype=np.int32))        # SPIKE only: code 2
    _lib.check(lib.mlbp_batch_reduce(ns, P(t_g), P(t_l), nv, P(t_r), P(words), P(out), S()))
    words2 = dev(np.array([1, 0, 0, 0, 0], dtype=np.int32))       # PEAK only: code 1 < 2, the maximum stays
    _lib.check(lib.mlbp_batch_reduce(ns, P(t_g), P(t_l), nv, P(t_r), P(words2), P(out), S()))
    torch.cuda.synchronize()
    one = np.concatenate([grad.sum(0), [lps.sum(), (rank == 0).sum(), (rank < 26).sum(), (rank < 50).sum(), nv, ns]])
    mag = np.concatenate([np.abs(grad).sum(0), [np.abs(lps).sum(), nv, nv, nv, nv, ns]])
    got = out.cpu().numpy()
    assert np.all(np.abs(got[:15] - (out0[:15] + 2 * one)) <= 1e-12 * (2 * mag + np.abs(out0[:15])))
    assert got[15] == 2.0
    w3 = dev(np.array([1, 0, 0, 1, 0], dtype=np.int32))           # both: code 3
    _lib.check(lib.mlbp_batch_reduce(ns, P(t_g), P(t_l), nv, P(t_r), P(w3), P(out), S()))
    torch.cuda.synchronize()
    assert out.cpu().numpy()[15] == 3.0
    # NULL grad / logp_sent / rank / peak_flag: only the sentence count moves
    before = out.cpu().numpy()
    _lib.check(lib.mlbp_batch_reduce(ns, None, None, nv, None, None, P(out), S()))
    torch.cuda.synchronize()
    after = out.cpu().numpy()
    assert np.array_equal(after[:14], before[:14]) and after[14] == before[14] + ns and after[15] == before[15]
    assert lib.mlbp_batch_reduce(-1, None, None, 0, None, None, P(out), S()) == ERR_INVALID


# ================================================================================================ K1 and the small kernels
THETA_ED = np.array([0.7, -0.4, 0.3, 0.2, -0.5, 0.1])
THETA_EE = np.array([0.6, -0.3, 0.2])


def unary_model(V, Vd, ldf, seed):
    rng = np.random.default_rng(seed)
    m = {'V': V, 'Vd': Vd}
    for k, shape in (('pmi', (V, V)), ('pmi_w1', (V, V)), ('ed', (V, Vd)), ('ped', (V, Vd))):
        m[k] = rng.random(shape, dtype=np.float32).astype(np.float64)   # fp32-representable: what the device reads
    pad = lambda X: np.concatenate([X, np.zeros((X.shape[0], ldf - X.shape[1]))], axis=1).astype(np.float32)
    planes = dict(pmi=pad(m['pmi']), w1=pad(m['pmi_w1']), edT=pad(m['ed'].T), pedT=pad(m['ped'].T))
    return m, planes


def test_build_unary_tables(lib):
    V, Vd, ldf = 1001, 37, 1004
    m, pl = unary_model(V, Vd, ldf, 51)
    es = torch.full((Vd + 1, 3), SENT32, dtype=torch.float64, device='cuda')
    edT, pedT = dev(pl['edT']), dev(pl['pedT'])
    _lib.check(lib.mlbp_build_unary_tables(P(edT), P(pedT), V, Vd, ldf,
                                           THETA_ED.ctypes.data_as(ctypes.c_void_p), P(es), S()))
    torch.cuda.synchronize()
    got = es.cpu().numpy()
    psi = np.exp(THETA_ED[0] * m['ed'] + THETA_ED[1] * m['ped'] + THETA_ED[5])      # [V, Vd]
    want = np.stack([psi.sum(0), (psi * m['ed']).sum(0), (psi * m['ped']).sum(0)], axis=1)
    assert np.all(np.abs(got[:Vd] - want) <= 1e-12 * np.abs(want))                  # float64 exp, float64 sums
    assert (got[Vd] == SENT32).all()


def unary_batch(V):
    """variables: (var_de, label, sparse [(e, feat, val)], given [(label, gap1)])"""
    return [
        (3, 17, [(1023, 2, 0.5), (1024, 3, 1.0), (1024, 2, 0.25), (1024, 2, 0.25), (17, 4, 1.0)], [(5, 0), (7, 1)]),
        (-1, 4, [], [(9, 1)]),                                    # no en_de factor
        (0, V - 1, [(0, 2, 1.0), (V - 1, 3, 2.0)], []),
        (-1, 0, [], []),
        (5, 1024, [(1023, 4, 1.0), (1022, 4, 1.0)], [(3, 0), (3, 1), (V - 1, 0)]),
    ]


def unary_inputs(V, vars_):
    sp, giv = [], []
    sp_off, giv_off = [0], [0]
    for d, y, s, g in vars_:
        sp += s
        giv += g
        sp_off.append(len(sp))
        giv_off.append(len(giv))
    i32 = lambda x: np.asarray(x, dtype=np.int32).reshape(-1)
    return dict(var_de=i32([v[0] for v in vars_]), var_label=i32([v[1] for v in vars_]), sp_off=i32(sp_off),
                sp_en=i32([x[0] for x in sp] or [0]), sp_feat=i32([x[1] for x in sp] or [0]),
                sp_val=np.asarray([x[2] for x in sp] or [0], dtype=np.float32), giv_off=i32(giv_off),
                giv_label=i32([x[0] for x in giv] or [0]), giv_gap1=i32([x[1] for x in giv] or [0]))


def unary_reference(m, vars_):
    """float64: psi_v = exp(phi_v . theta_ed) over the dense en_de features of the variable's German word (oracle
    dense_phi_en_de), and the en_en given-token factors' expectations from the oracle's T / T1 / G / G1 / G1w"""
    V = m['V']
    tb = orc.Tables(m, THETA_EE, THETA_ED)
    out = []
    for d, y, s, g in vars_:
        g9 = np.zeros(9)
        if d >= 0:
            phi = orc.dense_phi_en_de(m, types.SimpleNamespace(sparse=[(e, d, f, val) for e, f, val in s]))[:, d, :]
            psi = np.exp(phi @ THETA_ED)
            S0 = psi.sum()
            g9[3:9] = phi[y] - psi @ phi / S0
        else:
            psi, S0 = None, 1.0
        for o, gap in g:
            T, Gp = (tb.T1, tb.G1) if gap else (tb.T, tb.G)
            g9[0] += m['pmi'][y, o] - Gp[:, o].sum() / T[:, o].sum()
            if gap:
                g9[1] += m['pmi_w1'][y, o] - tb.G1w[:, o].sum() / tb.T1[:, o].sum()
        out.append(dict(psi=psi, S0=S0, g=g9))
    return tb, out


def colsums_of(tb):
    return np.stack([tb.T.sum(0), tb.T1.sum(0), tb.G.sum(0), tb.G1.sum(0), tb.G1w.sum(0), tb.T.sum(1), tb.T1.sum(1)])


def test_unary_stats(lib):
    V, Vd, ldf = 2050, 9, 2052
    m, pl = unary_model(V, Vd, ldf, 53)
    vars_ = unary_batch(V)
    x = unary_inputs(V, vars_)
    tb, ref = unary_reference(m, vars_)
    psi = np.exp(THETA_ED[0] * m['ed'] + THETA_ED[1] * m['ped'] + THETA_ED[5])
    edstats = np.stack([psi.sum(0), (psi * m['ed']).sum(0), (psi * m['ped']).sum(0)], axis=1)
    nv = len(vars_)
    inv = torch.full((nv + 1,), SENT32, dtype=torch.float64, device='cuda')
    gu = torch.full((nv + 1, 9), SENT32, dtype=torch.float64, device='cuda')
    t = {k: dev(v) for k, v in x.items()}
    t.update({k: dev(v) for k, v in pl.items()}, edstats=dev(edstats), cs=dev(colsums_of(tb)))
    _lib.check(lib.mlbp_unary_stats(nv, P(t['var_de']), P(t['var_label']), P(t['sp_off']), P(t['sp_en']), P(t['sp_feat']),
                                    P(t['sp_val']), P(t['giv_off']), P(t['giv_label']), P(t['giv_gap1']), P(t['pmi']),
                                    P(t['w1']), P(t['edT']), P(t['pedT']), V, ldf,
                                    THETA_ED.ctypes.data_as(ctypes.c_void_p), P(t['edstats']), P(t['cs']),
                                    P(inv), P(gu), S()))
    torch.cuda.synchronize()
    I, G = inv.cpu().numpy(), gu.cpu().numpy()
    for v, r in enumerate(ref):
        assert abs(I[v] - 1.0 / r['S0']) <= 1e-12 / r['S0'], v
        # float64 throughout; the bias entries are 1 - 1 (0 on the device, ~1e-16 in the dense reference)
        assert np.all(np.abs(G[v] - r['g']) <= 1e-11), (v, G[v], r['g'])
    assert I[nv] == SENT32 and (G[nv] == SENT32).all()


def test_unary_products(lib):
    """U[v] = V psi_v / sum(psi_v) times V T[:, o] / sum T[:, o] per given token (gap / no-gap planes), variables without an
    en_de factor, duplicate sparse features on one word, sparse words on both sides of the 1 024-column chunk boundary and
    V % 4 != 0: the row tail [V, roundup(V, 4)) is written as 0, nothing beyond it"""
    V, Vd, ldf, s = 2050, 9, 2052, 9
    ldv = roundup(V, 64)
    m, pl = unary_model(V, Vd, ldf, 57)
    vars_ = unary_batch(V)
    x = unary_inputs(V, vars_)
    tb, ref = unary_reference(m, vars_)
    planes = np.zeros((8, V, ldv), dtype=np.float16)
    for p, W in ((2, tb.Tt), (6, tb.T1t)):                         # Tt / T1t hi, lo: row o = column o of T / T1
        planes[p, :, :V], planes[p + 1, :, :V] = split16(W * 2.0 ** s)
    cs = colsums_of(tb)
    inv_sigma = np.array([1.0 / r['S0'] for r in ref])
    nv = len(vars_)
    U = torch.full((nv + 1, ldv), SENT32, dtype=torch.float32, device='cuda')
    t = {k: dev(v) for k, v in x.items()}
    t.update(edT=dev(pl['edT']), pedT=dev(pl['pedT']), inv=dev(inv_sigma), planes=dev(planes), cs=dev(cs))
    _lib.check(lib.mlbp_unary_products(nv, P(t['var_de']), P(t['sp_off']), P(t['sp_en']), P(t['sp_feat']), P(t['sp_val']),
                                       P(t['giv_off']), P(t['giv_label']), P(t['giv_gap1']), P(t['edT']),
                                       P(t['pedT']), V, ldf, THETA_ED.ctypes.data_as(ctypes.c_void_p), P(t['inv']),
                                       P(t['planes']), V * ldv, ldv, s, P(t['cs']), P(U), S()))
    torch.cuda.synchronize()
    got = U.cpu().numpy().astype(np.float64)
    for v, ((d, y, sp, giv), r) in enumerate(zip(vars_, ref)):
        want = V * r['psi'] / r['S0'] if d >= 0 else np.ones(V)
        for o, gap in giv:
            p = 6 if gap else 2
            tab = planes[p, o, :V].astype(np.float64) + planes[p + 1, o, :V].astype(np.float64)
            want = want * V * tab * 2.0 ** -s / cs[1 if gap else 0, o]
        # the en_de factor: expf (<= 2 ulp) of an fp32 fma chain whose inputs theta and log(V / S0) are rounded to fp32
        # (each term's error <= 2^-24 of its magnitude); each given token 4 fp32 roundings (scale, hi + lo, two products)
        if d >= 0:
            lsc = THETA_ED[5] + math.log(V / r['S0'])
            arg_abs = 2 * np.abs(THETA_ED[0] * pl['edT'][d, :V]) + 3 * np.abs(THETA_ED[1] * pl['pedT'][d, :V]) + 3 * abs(lsc)
            rel = arg_abs * U32 + 4 * U32                          # + expf's 2 ulp
        else:
            rel = np.zeros(V)
        rel = rel + 4 * len(giv) * U32 + U32
        assert np.all(np.abs(got[v, :V] - want) <= rel * want), v
        assert (got[v, V:roundup(V, 4)] == 0).all() and (got[v, roundup(V, 4):] == SENT32).all(), v
    assert (got[nv] == SENT32).all()


def test_const_rows(lib):
    """row 0 = 1.0 over the whole padded row; rows 1..4 = colsums rows 5, 0, 6, 1 mean-one scaled, padding 0; an all-zero
    sum leaves its row unscaled"""
    V, ldv = 1001, 1024
    rng = np.random.default_rng(59)
    cs = rng.random((7, V)) * 100 + 1
    cs[6] = 0.0
    rows = torch.full((6, ldv), SENT32, dtype=torch.float32, device='cuda')
    tcs = dev(cs)
    _lib.check(lib.mlbp_const_rows(P(tcs), V, ldv, P(rows), S()))
    torch.cuda.synchronize()
    got = rows.cpu().numpy().astype(np.float64)
    assert (got[0] == 1.0).all() and (got[5] == SENT32).all()
    for t, src in enumerate((5, 0, 6, 1), start=1):
        ssum = cs[src].sum()
        want = cs[src] * V / ssum if ssum > 0 else cs[src]
        assert np.all(np.abs(got[t, :V] - want) <= U32 * np.abs(want) * 1.01), t     # one fp32 rounding
        assert (got[t, V:] == 0).all()


@pytest.mark.parametrize('V', [1001, 64, 3])
def test_fill_uniform_rows(lib, V):
    ld = roundup(V, 64)
    rows = np.array([3, 7, 0], dtype=np.int32)
    hi_w, lo_w = split16(np.float32(SCALE) / np.float32(V))
    rng = np.random.default_rng(V)
    keep = (rng.random(V) < 0.6).astype(np.uint8)
    for k in (None, keep):
        Ah = torch.full((9, ld), SENT16, dtype=torch.float16, device='cuda')
        Al = torch.full((9, ld), SENT16, dtype=torch.float16, device='cuda')
        trows, tkeep = dev(rows), dev(k) if k is not None else None
        _lib.check(lib.mlbp_fill_uniform_rows(P(Ah), P(Al), ld, V, P(trows), len(rows), P(tkeep), S()))
        torch.cuda.synchronize()
        h, l = Ah.cpu().numpy(), Al.cpu().numpy()
        on = np.ones(V, dtype=bool) if k is None else k.astype(bool)
        for r in range(9):
            if r in rows:
                assert (h[r, :V][on] == hi_w).all() and (l[r, :V][on] == lo_w).all()
                assert (h[r, :V][~on] == 0).all() and (l[r, :V][~on] == 0).all()
                assert (h[r, V:] == 0).all() and (l[r, V:] == 0).all()            # the padding of a filled row is zeroed
            else:
                assert (h[r] == SENT16).all() and (l[r] == SENT16).all()


def test_topk_mask_rows_ties_at_threshold(lib):
    """exactly K entries survive per row, none of them below the K-th largest value, every entry above it survives (ties at
    the threshold are cut to fill K); rows outside [row0, row0 + n_rows) and the row padding are untouched"""
    V, K = 700, 100
    ld = roundup(V, 64)
    rng = np.random.default_rng(61)
    n = 6
    X = rng.random((n, V)) * 0.5 + 0.25
    X[1, rng.permutation(V)[:90]] = 0.9 + 0.05 * rng.random(90)      # 90 above, then 40 tied at the K-th value
    X[1, np.argsort(X[1])[:-90][rng.permutation(V - 90)[:40]]] = 0.8
    X[2, :] = 0.3                                                     # every entry tied
    X[3, :K + 1] = 0.7                                                # K + 1 tied at the top
    X[3, K + 1:] *= 0.5
    h, l = split16(X)
    Ah = np.full((n + 2, ld), SENT16, dtype=np.float16)
    Al = np.full((n + 2, ld), SENT16, dtype=np.float16)
    Ah[1:n + 1, :V], Al[1:n + 1, :V] = h, l
    tA, tL = dev(Ah), dev(Al)
    _lib.check(lib.mlbp_topk_mask_rows(P(tA), P(tL), ld, V, 1, n, K, S()))
    torch.cuda.synchronize()
    gh, gl = tA.cpu().numpy(), tL.cpu().numpy()
    assert np.array_equal(gh[0], Ah[0]) and np.array_equal(gh[n + 1], Ah[n + 1])
    assert (gh[:, V:] == SENT16).all() and (gl[:, V:] == SENT16).all()
    for i in range(n):
        val = h[i].astype(np.float32) + l[i].astype(np.float32)    # the order the kernel ranks by: fp32 hi + lo
        kth = np.sort(val)[::-1][K - 1]
        kept = (gh[1 + i, :V] != 0) | (gl[1 + i, :V] != 0)
        assert kept.sum() == K, (i, kept.sum())
        assert (val[kept] >= kth).all() and kept[val > kth].all()
        assert np.array_equal(gh[1 + i, :V][kept], h[i][kept]) and np.array_equal(gl[1 + i, :V][kept], l[i][kept])
        assert (gh[1 + i, :V][~kept] == 0).all() and (gl[1 + i, :V][~kept] == 0).all()
    assert (X[1] == 0.8).sum() == 40
    # K >= V: nothing to mask
    _lib.check(lib.mlbp_topk_mask_rows(P(tA), P(tL), ld, V, 1, n, V, S()))
    torch.cuda.synchronize()
    assert np.array_equal(tA.cpu().numpy(), gh)
