"""GPU tier, kernel level: K5 near-tie flags (mlbp_marginals) and K5b's exact re-score (mlbp_rescore_candidates) through the
C ABI, called as Engine.run calls them, on the engineered near-ties of rescore_cases.py against float64 decisions.

Per case: K5's products, flags, arg-max, rank, aux and counts equal the exact host model of the kernel; every decision K5 gets
wrong is flagged; after K5b every arg-max and every rank that can matter (<= 50) is the float64 one, exact ties going to the
first index; unflagged and skipped variables keep K5's answers; the counters count what happened; the result does not depend
on the order of the flagged list."""
import ctypes
import os
import sys

import numpy as np
import pytest
import torch

from macaronicusermodeling_b200 import _lib, build

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)

import rescore_cases as rc  # noqa: E402

pytestmark = pytest.mark.gpu

DEV = 'cuda'
SENT = -5
ERR_INVALID = 1


@pytest.fixture(scope='module')
def lib():
    build.build()
    return _lib.require_device()


def P(t, byte_offset=0):
    return ctypes.c_void_p(t.data_ptr() + byte_offset) if t is not None else None


def S():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def sync():
    torch.cuda.synchronize()


def dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).to(DEV)


_CACHE = {}


def case_on_device(V):
    """one case per V (two-pass bands below V = 8192, one-pass bands above, as the engine picks them), built once and kept
    on the device while the tests of that V run; the 20 planes are gathered from the pool on the device"""
    if V not in _CACHE:
        _CACHE.clear()
        c = rc.build_case(V, seed=V, bands='two_pass' if V < 8192 else 'one_pass', profile='many' if V < 2048 else 'few')
        d = {k: dev(c[k]) for k in ('grp_u', 'grp_off', 'in_row', 'label', 'U', 'D', 'blocks')}
        d['A_hi'], d['A_lo'] = dev(c['A_hi']), dev(c['A_lo'])
        pool_hi, pool_lo = dev(c['pool_hi']), dev(c['pool_lo'])
        planes = torch.empty((2 * rc.N_PLANE_PAIRS, V, c['ld']), dtype=torch.float16, device=DEV)
        for p in range(rc.N_PLANE_PAIRS):
            rm = dev(c['rowmap'][p])
            planes[2 * p] = pool_hi.index_select(0, rm)
            planes[2 * p + 1] = pool_lo.index_select(0, rm)
        d['planes'] = planes
        del pool_hi, pool_lo
        _CACHE[V] = (c, d)
    return _CACHE[V]


def k5(lib, c, d, range_log2):
    n = c['n_groups']
    o = dict(logp=torch.full((n,), -7.0, dtype=torch.float64, device=DEV),
             top1=torch.full((n,), SENT, dtype=torch.int32, device=DEV), rank=torch.full((n,), SENT, dtype=torch.int32, device=DEV),
             aux=torch.full((n, 2), -7.0, dtype=torch.float64, device=DEV), cnts=torch.full((n, 2), SENT, dtype=torch.int32, device=DEV),
             flags=torch.full((n,), SENT, dtype=torch.int32, device=DEV), flagged=torch.full((n,), SENT, dtype=torch.int32, device=DEV),
             words=torch.zeros(16, dtype=torch.int32, device=DEV))
    _lib.check(lib.mlbp_marginals(n, P(d['grp_u']), P(d['grp_off']), P(d['in_row']), P(d['label']), P(d['U']), P(d['D']), c['ld'],
                                  c['V'], P(o['logp']), P(o['top1']), P(o['rank']), None, range_log2, c['max_in'], c['tau'],
                                  c['tau_label'], P(o['aux']), P(o['cnts']), P(o['flags']), P(o['flagged']), P(o['words']), S()))
    return o


def k5b(lib, c, d, o, range_log2, **bad):
    """mlbp_rescore_candidates on K5's outputs o (top1 / rank overwritten in place, counters in o['words'][8:]); keyword
    arguments replace single arguments (refused calls)"""
    a = dict(n_vars=c['n_groups'], flagged=P(o['flagged']), n_flagged=P(o['words']), flags=P(o['flags']), grp_u=P(d['grp_u']),
             grp_off=P(d['grp_off']), in_row=P(d['in_row']), label=P(d['label']), U=P(d['U']), D=P(d['D']), ldv=c['ld'],
             V=c['V'], A_hi=P(d['A_hi']), A_lo=P(d['A_lo']), planes=P(d['planes']), plane_stride=c['V'] * c['ld'],
             msg_blocks=P(d['blocks']), n_blocks=len(c['blocks']), n_msg_rows=c['n_a'], aux=P(o['aux']), cnts=P(o['cnts']),
             tau=c['tau'], tau_label=c['tau_label'], range_log2=range_log2, top1=P(o['top1']), rank=P(o['rank']),
             counters=P(o['words'], 32))
    a.update(bad)
    return lib.mlbp_rescore_candidates(*a.values(), S())


def host(o):
    return {k: v.cpu().numpy().copy() for k, v in o.items()}


def check_k5b(c, h5, h, range_log2):
    """h5: outputs of K5 alone, h: after K5b"""
    fp64 = not (0.0 <= range_log2 < 100.0)
    n, nf = c['n_groups'], int(h5['words'][0])
    flagged = np.zeros(n, dtype=bool)
    flagged[h5['flagged'][:nf]] = True
    assert nf >= 1 and len(set(h5['flagged'][:nf].tolist())) == nf and (flagged == (h5['flags'] != 0)).all()
    skipped = {'mass': 0, 'degenerate': 0}
    for g, spec in enumerate(c['groups']):
        m = rc.k5_model(c, g, fp64)
        # K5 against its exact model: same products in the same type and order, so every decision and count is equal
        assert (h5['flags'][g], h5['top1'][g], h5['rank'][g]) == (m['flags'], m['top1'], m['rank']), (g, spec['kind'])
        if m['ok']:
            assert tuple(h5['aux'][g]) == (m['best'], m['plab']) and tuple(h5['cnts'][g]) == (m['icnt'], m['inh']), g
        kept = (h['top1'][g], h['rank'][g]) == (h5['top1'][g], h5['rank'][g])
        if spec['kind'] in rc.KEEPS_K5:
            assert flagged[g] and kept, (g, spec['kind'])
            skipped[spec['kind']] += 1
            continue
        if spec['fp64_only'] and not fp64:
            assert not m['ok'] and not flagged[g] and kept
            continue
        L, lab = rc.reference(c, g), int(c['label'][g])
        # flag safety: every decision K5 gets wrong is flagged, and what is not flagged is left alone
        if not rc.top1_ok(L, h5['top1'][g]):
            assert h5['flags'][g] & 1, (g, spec['kind'], 'a wrong arg-max was not flagged')
        if not rc.rank_ok(L, lab, h5['rank'][g]):
            assert h5['flags'][g] & 2, (g, spec['kind'], 'a wrong rank was not flagged')
        if not flagged[g]:
            assert kept, g
        # decisions after the re-score
        assert rc.top1_ok(L, h['top1'][g]), (g, spec['kind'], h['top1'][g], rc.decisions(L, lab), h5['top1'][g])
        assert rc.rank_ok(L, lab, h['rank'][g]), (g, spec['kind'], h['rank'][g], rc.decisions(L, lab), h5['rank'][g])
        for e1, e2 in spec['ties']:                        # exact float64 ties: the first index, never counted above
            if L[e1] == L.max():
                assert h['top1'][g] == e1, (g, spec['kind'])
    cnt = h['words'][8:13]
    n_mass = sum(s['kind'] == 'mass' for s in c['groups'])
    n_deg = sum(s['kind'] == 'degenerate' for s in c['groups'])
    assert (cnt[1], cnt[2]) == (n_mass, n_deg) == (skipped['mass'], skipped['degenerate']), cnt
    assert cnt[0] == nf - cnt[1] - cnt[2], (cnt, nf)
    assert cnt[3] == int((h['top1'] != h5['top1']).sum()) and cnt[4] == int((h['rank'] != h5['rank']).sum()), cnt
    assert cnt[3] > 0 and cnt[4] > 0, cnt                    # the re-score did change decisions
    return nf


@pytest.mark.parametrize('V,range_log2', [(1001, 50.0), (1001, -1.0), (1001, 99.9), (1001, 100.0), (1001, 120.0),
                                          (4608, 50.0), (4608, -1.0), (10000, 50.0), (10000, -1.0)])
def test_rescore_restores_float64_decisions(lib, V, range_log2):
    """fp32 products (0 <= range_log2 < 100) and fp64 products (else) in both kernels: 99.9 / 100 pin the shared switch"""
    c, d = case_on_device(V)
    o = k5(lib, c, d, range_log2)
    sync()
    h5 = host(o)
    assert int(h5['words'][8:].sum()) == 0
    _lib.check(k5b(lib, c, d, o, range_log2))
    sync()
    h = host(o)
    nf = check_k5b(c, h5, h, range_log2)
    if V == 1001:
        assert nf >= 1500, nf                              # more flagged variables than K5b's grid has CTAs (8 per SM)
    # the flagged list is filled by atomics in no particular order: a permuted list gives the same results
    nf = int(h5['words'][0])
    perm = np.random.default_rng(V).permutation(h5['flagged'][:nf])
    o2 = {k: dev(v) for k, v in h5.items()}
    o2['flagged'][:nf] = dev(perm.astype(np.int32))
    _lib.check(k5b(lib, c, d, o2, range_log2))
    sync()
    h2 = host(o2)
    for k in ('top1', 'rank'):
        assert np.array_equal(h2[k], h[k]), k
    assert np.array_equal(h2['words'][8:13], h['words'][8:13])
    assert _lib.load().mlbp_gemm_barrier_timeout_code() == 0


def test_rescore_refused_calls_leave_outputs(lib):
    """bad bands, a row pitch that is not a multiple of 64, misaligned operands and a null pointer: MLBP_ERR_INVALID and
    nothing launched (top1, rank and the counters keep their sentinels)"""
    c, d = case_on_device(1001)
    o = k5(lib, c, d, 50.0)
    sync()
    ref = host(o)
    o['words'][8:] = SENT
    for bad in (dict(tau=0.5), dict(tau_label=0.5), dict(ldv=c['ld'] - 8), dict(planes=P(d['planes'], 2)),
                dict(A_hi=P(d['A_hi'], 2)), dict(A_lo=P(d['A_lo'], 8)), dict(aux=None), dict(flagged=None),
                dict(msg_blocks=None)):
        assert k5b(lib, c, d, o, 50.0, **bad) == ERR_INVALID, bad
        sync()
        h = host(o)
        assert np.array_equal(h['top1'], ref['top1']) and np.array_equal(h['rank'], ref['rank']), bad
        assert (h['words'][8:] == SENT).all(), bad
