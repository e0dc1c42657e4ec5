"""CPU tier of the near-tie cases in rescore_cases.py: the builder puts every engineered gap where it should be, the stored
rows' perturbation really reverses decisions (else the GPU test of the exact re-score would prove nothing), every decision it
reverses is flagged by the model of K5, and the log-space reference equals a direct float64 evaluation."""
import math
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)

import rescore_cases as rc  # noqa: E402


@pytest.fixture(scope='module')
def case():
    return rc.build_case(1001, seed=1)


def test_engineered_gaps_are_where_intended(case):
    c = case
    fp32_excess = 0.0
    for g, spec in enumerate(c['groups']):
        if spec['kind'] == 'degenerate':
            continue
        L = rc.reference(c, g)
        m = rc.k5_model(c, g, fp64=True)                # products of the stored rows, rounded only in float64
        with np.errstate(divide='ignore', invalid='ignore'):
            lp = np.log(m['p'])
            d = (lp - L)[np.isfinite(L)]
        for x, y, lg, flip in spec['pairs']:
            # U is rounded to fp32 after the levels are set: each of the two beliefs moves by at most 2^-24
            assert abs((L[x] - L[y]) - lg) <= 2.0 ** -23 + 1e-15, (g, spec['kind'], x, y, L[x] - L[y], lg)
            if flip:
                assert np.sign(lp[x] - lp[y]) == -np.sign(lg), (g, spec['kind'], lp[x] - lp[y], lg)
        for e1, e2 in spec['ties']:
            assert L[e1] == L[e2] and m['p'][e1] == m['p'][e2] and e1 < e2
        if spec['kind'] in ('argmax', 'argmax_tie', 'zero_label', 'deep', 'deep_underflow'):
            top = [e for e in range(c['V']) if L[e] >= L.max() - 1e-3]
            assert len(top) == 2 + (spec['kind'] == 'argmax_tie') and m['flags'] & 1, (g, spec['kind'], top)
        if spec['kind'] == 'rank':
            assert rc.decisions(L, spec['label'])[1] < 50 and m['flags'] & 2
        # the stored rows deviate from the float64 rows by at most eps (+ fp32 roundings) on every element
        if spec['m'] and spec['kind'] != 'deep_underflow':
            fp32_excess = max(fp32_excess, float(np.abs(d - np.median(d)).max()) - 2 * c['eps'])
    assert fp32_excess <= 2e-5, fp32_excess
    kinds = {}
    for g, spec in enumerate(c['groups']):
        kinds.setdefault(spec['kind'], []).append(g)
    for g in kinds['edge_best']:                       # runner-up exactly at best * (1 - tau) in fp32: flagged (>=)
        a, b = c['groups'][g]['edge']
        m = rc.k5_model(c, g, fp64=False)
        assert m['p'][b] == m['best'] * (np.float32(1) - np.float32(c['tau'])) and m['flags'] & 1 and m['b0'][b]
    for g in kinds['edge_lab']:                        # neighbours exactly at plab * (1 +- tau_label) in fp32: inside the band
        hi, lo = c['groups'][g]['edge']
        m = rc.k5_model(c, g, fp64=False)
        one = np.float32(1)
        assert m['p'][hi] == np.float32(m['plab']) * (one + np.float32(c['tau_label']))
        assert m['p'][lo] == np.float32(m['plab']) * (one - np.float32(c['tau_label']))
        assert m['b2'][hi] and m['b2'][lo] and m['inh'] == 1 and m['flags'] == 2
        assert rc.decisions(rc.reference(c, g), c['label'][g])[1] == m['icnt'] == 11
    for g in kinds['bit1_50'] + kinds['bit1_51']:
        m = rc.k5_model(c, g, fp64=False)
        above = int(c['groups'][g]['kind'][-2:])
        assert m['icnt'] == above and m['inh'] == 0 and m['inl'] == 1
        assert rc.decisions(rc.reference(c, g), c['label'][g])[1] == above + 1
        assert bool(m['flags'] & 2) == (above == 50)
    for g in kinds['mass']:
        m = rc.k5_model(c, g, fp64=False)
        assert m['flags'] & 1 and m['n_cand'] > rc.MAX_CAND
    for g in kinds['degenerate']:
        spec = c['groups'][g]
        a = spec['a0'] + spec['zero_rows'][0]
        assert np.isneginf(rc.reference(c, g)).all() and (c['A_hi'][a, :c['V']] == 0).all()
        assert (c['D'][rc.D_CONST_ROWS + a, :c['V']] > 0).all() and rc.k5_model(c, g, fp64=False)['flags'] & 1
    for g in kinds['zero_label']:
        m = rc.k5_model(c, g, fp64=False)
        assert m['plab'] == 0 and m['flags'] == 1
    for g in kinds['deep'] + kinds['deep_underflow']:
        assert len(rc.group_rows(c, g)) == rc.MAX_IN
    g, = kinds['deep_underflow']
    assert not rc.k5_model(c, g, fp64=False)['ok'] and rc.k5_model(c, g, fp64=True)['flags'] & 1
    # only the engineered variables are skipped by K5b
    n_mass = sum(rc.k5_model(c, g, fp64=False)['n_cand'] > rc.MAX_CAND for g in range(c['n_groups']))
    assert n_mass == len(kinds['mass'])


@pytest.mark.parametrize('fp64', [False, True], ids=['fp32', 'fp64'])
def test_eps_reverses_decisions_and_every_reversal_is_flagged(case, fp64):
    c = case
    wrong_top, wrong_rank, flagged = 0, 0, 0
    for g, spec in enumerate(c['groups']):
        m = rc.k5_model(c, g, fp64)
        flagged += m['flags'] != 0
        if spec['kind'] == 'degenerate' or not m['ok']:
            continue
        L = rc.reference(c, g)
        if not rc.top1_ok(L, m['top1']):
            wrong_top += 1
            assert m['flags'] & 1, (g, spec['kind'])
        if not rc.rank_ok(L, c['label'][g], m['rank']):
            wrong_rank += 1
            assert m['flags'] & 2, (g, spec['kind'])
    assert wrong_top >= 100 and wrong_rank >= 100, (wrong_top, wrong_rank)
    assert flagged >= 1500, flagged                    # more than the 8 x 148 CTAs of K5b's grid on a B200


def test_reference_equals_direct_float64_product():
    c = rc.build_case(96, seed=3, profile='small')
    V = c['V']
    A = c['A_hi'][:, :V].astype(np.float64) + c['A_lo'][:, :V].astype(np.float64)
    tables = [rc.planes_exact(c, t) for t in range(4)]
    for g in range(c['n_groups']):
        p = c['U'][c['grp_u'][g], :V].astype(np.float64)
        for r in rc.group_rows(c, g):
            if r >= rc.D_CONST_ROWS:
                a = r - rc.D_CONST_ROWS
                B = tables[c['row_table'][a]]
                p = p * np.array([math.fsum(A[a] * B[e]) for e in range(V)])
            elif r >= 0:
                p = p * c['D'][r, :V].astype(np.float64)
        L = rc.reference(c, g)
        np.testing.assert_allclose(L, np.log(p), rtol=0, atol=1e-12)
        lab = c['label'][g]
        assert rc.decisions(L, lab) == (int(np.argmax(p)), int((p > p[lab]).sum()))
    # the layout: message rows in ascending contiguous blocks covering every A row, each message table in several blocks
    b = c['blocks']
    assert (b[:, 1] == np.concatenate([[0], np.cumsum(b[:, 3])[:-1]])).all() and b[:, 3].sum() == c['n_a']
    assert (b[:, 2] == b[:, 1] + rc.D_CONST_ROWS).all()
    full = rc.build_case(1001, seed=1, profile='few')
    assert all((full['blocks'][:, 0] == t).sum() >= 2 for t in range(4))
    for arr in (full['U'], full['D'], full['A_hi'], full['A_lo'], full['pool_hi'], full['pool_lo']):
        assert np.isnan(arr[:, full['V']:]).all()        # row padding: poisoned
    stack = rc.plane_stack(c)
    for p in range(rc.N_PLANE_PAIRS):                   # every plane pair differs from every other
        for q in range(p):
            assert not np.array_equal(stack[2 * p, :, :V], stack[2 * q, :, :V])
