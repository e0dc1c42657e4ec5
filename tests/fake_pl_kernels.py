"""TEST DOUBLE for K13 (mlbp_pseudo_likelihood, csrc/pseudo.cu): FakeKernels plus the entry point, emulated through the
plane-level reference (tests/pl_oracle.py) on host pointers, with the kernel's refusals (raised as the error the library's
return code becomes).  Never imported by the package."""
import numpy as np

from fake_kernels import FakeKernels, _arr
from macaronicusermodeling_b200._lib import MlbpError
from macaronicusermodeling_b200.engine import Corpus
import pl_oracle

MAX_K = 49                   # MLBP_PL_MAX_K


def _refuse(code, what):
    raise MlbpError('libmlbp error %d: %s' % (code, what))


class PLKernels(FakeKernels):
    """FakeKernels plus mlbp_pseudo_likelihood"""

    def mlbp_pseudo_likelihood(self, n_sent, max_k, n_vars, var_off, pair_off, pair_v0, pair_v1, pair_gap1, var_label, var_de,
                               sp_off, sp_en, sp_feat, sp_val, giv_off, giv_label, giv_gap1, U, planes, ps, ldv, V, scale_exp,
                               colsums, pmi, pmi_w1, edT, pedT, ldf, range_log2, logp_var, top1, rank, grad, beliefs):
        live = lambda p: p is not None and getattr(p, 'value', p)
        if not all(live(p) for p in (var_off, pair_off, pair_v0, pair_v1, pair_gap1, var_label, giv_off, giv_label, giv_gap1, U,
                                     planes, colsums, logp_var, top1, rank)):
            _refuse(1, 'pseudo_likelihood: null pointer')
        want_grad = live(grad)
        if want_grad and not all(live(p) for p in (var_de, sp_off, sp_en, sp_feat, sp_val, pmi, pmi_w1, edT, pedT)):
            _refuse(1, 'pseudo_likelihood: the gradient needs var_de, the sparse lists and the feature planes')
        if n_sent < 0 or n_vars < 0 or V < 1 or ldv < V or ldv % 8 or ps % 8 or ps < V * ldv or \
                (want_grad and (ldf < V or ldf % 8)):
            _refuse(1, 'pseudo_likelihood: bad n_sent / n_vars / V / ldv / plane_stride / ldf')
        al = U.value | planes.value | (beliefs.value if live(beliefs) else 0) | ((edT.value | pedT.value) if want_grad else 0)
        if al % 16:
            _refuse(1, 'pseudo_likelihood: misaligned rows')
        if n_sent and max_k < 1:
            _refuse(1, 'pseudo_likelihood: max_k < 1')
        if max_k > MAX_K:
            _refuse(3, 'pseudo_likelihood: sentences of %d variables' % max_k)
        if n_sent == 0 or n_vars == 0:
            return
        i32 = lambda p, n: _arr(p, np.int32, max(n, 1))[:n].copy()
        vo, po = i32(var_off, n_sent + 1), i32(pair_off, n_sent + 1)
        assert int(np.diff(vo).max()) <= max_k
        npairs, ng = int(po[-1]), None
        go = i32(giv_off, n_vars + 1)
        ng = int(go[-1])
        so = i32(sp_off, n_vars + 1) if want_grad else np.zeros(n_vars + 1, dtype=np.int32)
        ns = int(so[-1])
        c = Corpus(var_off=vo, var_de=i32(var_de, n_vars) if want_grad else np.full(n_vars, -1, dtype=np.int32),
                   var_label=i32(var_label, n_vars), var_pos=np.zeros(n_vars, dtype=np.int32), sp_off=so,
                   sp_en=i32(sp_en, ns) if want_grad else so[:0], sp_feat=i32(sp_feat, ns) if want_grad else so[:0],
                   sp_val=_arr(sp_val, np.float32, max(ns, 1))[:ns].copy() if want_grad else np.zeros(0, dtype=np.float32),
                   giv_off=go, giv_label=i32(giv_label, ng), giv_gap1=i32(giv_gap1, ng), pair_off=po,
                   pair_v0=i32(pair_v0, npairs), pair_v1=i32(pair_v1, npairs), pair_gap1=i32(pair_gap1, npairs))
        n_planes = 20 if want_grad else 8
        pl = _arr(planes, np.float16, n_planes * ps)
        pls = [pl[p * ps:p * ps + V * ldv].reshape(V, ldv) for p in range(n_planes)] + [None] * (20 - n_planes)
        Um = _arr(U, np.float32, n_vars * ldv).reshape(n_vars, ldv)
        cs = _arr(colsums, np.float64, 7 * V).reshape(7, V)
        f64 = not (0.0 <= range_log2 < 100.0)
        mat = lambda p, rows: _arr(p, np.float32, rows * ldf).reshape(rows, ldf) if want_grad else None
        Vd = int(c.var_de.max()) + 1 if want_grad and n_vars else 0
        lp, t1, rk, g, rows, _ = pl_oracle.planes_reference(c, Um, pls, cs, scale_exp, mat(pmi, V), mat(pmi_w1, V),
                                                            mat(edT, max(Vd, 1)), mat(pedT, max(Vd, 1)), f64, want_grad)
        _arr(logp_var, np.float64, n_vars)[:] = lp
        _arr(top1, np.int32, n_vars)[:] = t1
        _arr(rank, np.int32, n_vars)[:] = rk
        if want_grad:
            _arr(grad, np.float64, n_vars * 9).reshape(n_vars, 9)[:] = g
        if live(beliefs):
            _arr(beliefs, np.float32, n_vars * ldv).reshape(n_vars, ldv)[:, :V] = rows
