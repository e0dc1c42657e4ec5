"""TEST DOUBLE for K12 (mlbp_gibbs_sample, mlbp_gibbs_reduce; csrc/gibbs.cu): FakeKernels plus the two entry points, emulated
through the NumPy reference sampler (tests/gibbs_oracle.py) on host pointers, with the kernels' refusals (raised as the error the
library's return code becomes).  Never imported by the package."""
import numpy as np

from fake_kernels import FakeKernels, _arr
from macaronicusermodeling_b200._lib import MlbpError
import gibbs_oracle

MAX_K = 64                   # MLBP_GIBBS_MAX_K


def _refuse(code, what):
    raise MlbpError('libmlbp error %d: %s' % (code, what))


class GibbsKernels(FakeKernels):
    """FakeKernels plus mlbp_gibbs_sample and mlbp_gibbs_reduce"""

    def mlbp_gibbs_sample(self, n_sent, max_k, n_vars, var_off, pair_off, pair_v0, pair_v1, pair_gap1, sent_id, U, planes, ps, ldv,
                          V, scale_exp, colsums, chains, burn_in, n_keep, seed, range_log2, acc, samples):
        live = lambda p: p is not None and getattr(p, 'value', p)
        if not all(live(p) for p in (var_off, pair_off, pair_v0, pair_v1, pair_gap1, sent_id, U, planes, colsums, acc)):
            _refuse(1, 'gibbs_sample: null pointer')
        if n_sent < 0 or n_vars < 0 or V < 1 or ldv < V or ldv % 8 or ps % 8 or ps < V * ldv:
            _refuse(1, 'gibbs_sample: bad n_sent / n_vars / V / ldv / plane_stride')
        if (U.value | planes.value | acc.value) % 16:
            _refuse(1, 'gibbs_sample: misaligned rows')
        if chains < 1 or n_keep < 1 or burn_in < 0:
            _refuse(1, 'gibbs_sample: chains and n_keep must be >= 1, burn_in >= 0')
        if n_sent and max_k < 1:
            _refuse(1, 'gibbs_sample: max_k < 1')
        if max_k > MAX_K:
            _refuse(3, 'gibbs_sample: sentences of %d variables' % max_k)
        if n_sent == 0:
            return
        i32 = lambda p, n: _arr(p, np.int32, max(n, 1))[:n].copy()
        vo, po = i32(var_off, n_sent + 1), i32(pair_off, n_sent + 1)
        assert int(np.diff(vo).max()) <= max_k
        npairs = int(po[-1])
        pl = _arr(planes, np.float16, 8 * ps)
        pls = [pl[p * ps:p * ps + V * ldv].reshape(V, ldv) for p in range(8)]
        Um = _arr(U, np.float32, n_vars * ldv).reshape(n_vars, ldv)
        cs = _arr(colsums, np.float64, 7 * V).reshape(7, V)
        f64 = not (0.0 <= range_log2 < 100.0)
        a, s, _ = gibbs_oracle.sample(vo, po, i32(pair_v0, npairs), i32(pair_v1, npairs), i32(pair_gap1, npairs),
                                      i32(sent_id, n_sent), Um, pls, cs, scale_exp, int(seed) & 0xffffffffffffffff, chains,
                                      burn_in, n_keep, f64)
        _arr(acc, np.float32, chains * n_vars * ldv).reshape(chains, n_vars, ldv)[:, :, :V] = a
        if live(samples):
            _arr(samples, np.int32, chains * n_keep * n_vars).reshape(chains, n_keep, n_vars)[:] = s

    def mlbp_gibbs_reduce(self, n_vars, chains, n_keep, acc, ldv, V, var_label, marginals, label_prob, logp_var, top1, rank):
        if not all(p is not None and p.value for p in (acc, var_label, marginals, label_prob, logp_var, top1, rank)):
            _refuse(1, 'gibbs_reduce: null pointer')
        if n_vars < 0 or V < 1 or ldv < V or ldv % 8 or (acc.value | marginals.value) % 16 or chains < 1 or n_keep < 1:
            _refuse(1, 'gibbs_reduce: bad arguments')
        if n_vars == 0:
            return
        a = _arr(acc, np.float32, chains * n_vars * ldv).reshape(chains, n_vars, ldv)[:, :, :V]
        m, lp, logp, t1, rk = gibbs_oracle.reduce(a, _arr(var_label, np.int32, n_vars), n_keep)
        _arr(marginals, np.float32, n_vars * ldv).reshape(n_vars, ldv)[:, :V] = m
        _arr(label_prob, np.float64, n_vars * chains).reshape(n_vars, chains)[:] = lp
        _arr(logp_var, np.float64, n_vars)[:] = logp
        _arr(top1, np.int32, n_vars)[:] = t1
        _arr(rank, np.int32, n_vars)[:] = rk
