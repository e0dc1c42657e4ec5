"""TEST DOUBLE for K10 / K11 (mlbp_factor_to_var_maxprod, mlbp_assignment_score; csrc/maxprod.cu): FakeKernels plus max-product
message rows and assignment scores, emulated in NumPy on host pointers with the kernels' conventions (rows normalised by their
max, the centred table formed from the fp32 feature planes, columns k >= V unused, a zero row gives a zero D row) and their
range checks.  Never imported by the package."""
import numpy as np

from fake_kernels import FakeKernels, _arr
from macaronicusermodeling_b200.engine import Corpus
import maxprod_oracle


class MapKernels(FakeKernels):
    """FakeKernels plus mlbp_factor_to_var_maxprod and mlbp_assignment_score"""

    def mlbp_factor_to_var_maxprod(self, A_hi, A_lo, a_rows_total, a_row0, n_rows, table, pmi, pmi_w1, V, ldv, ldf, h_theta_ee,
                                   centre_exp, D, d_row0, ldd):
        assert 0 <= table <= 3 and V >= 1 and min(ldv, ldf, ldd) >= V and 0 <= a_row0 and a_row0 + n_rows <= a_rows_total
        if n_rows == 0:
            return
        th = _arr(h_theta_ee, np.float64, 3)
        P = _arr(pmi, np.float32, V * ldf).reshape(V, ldf)[:, :V].astype(np.float64)
        W = _arr(pmi_w1, np.float32, V * ldf).reshape(V, ldf)[:, :V].astype(np.float64)
        z = th[0] * P + th[2] - centre_exp * np.log(2.0) + (th[1] * W if table in (2, 3) else 0.0)
        T = np.exp(z).astype(np.float32)                             # T[a, b]; B[n][k] = T[n, k] or T[k, n]
        B = T.T if table in (1, 3) else T                            # B[n, k] -> max over k of a[k] * B[n, k]
        n = (a_row0 + n_rows) * ldv
        H = _arr(A_hi, np.float16, n).reshape(-1, ldv)[a_row0:, :V].astype(np.float32)
        L = _arr(A_lo, np.float16, n).reshape(-1, ldv)[a_row0:, :V].astype(np.float32)
        a = H + L
        amax = a.max(axis=1)
        out = maxprod_oracle.max_times(a, B.T.astype(np.float64)).astype(np.float32)
        with np.errstate(invalid='ignore', divide='ignore'):
            out = np.where(amax[:, None] > 0, out / np.where(amax > 0, amax, 1.0)[:, None], np.float32(0)).astype(np.float32)
        _arr(D, np.float32, (d_row0 + n_rows) * ldd).reshape(-1, ldd)[d_row0:d_row0 + n_rows, :V] = out

    def mlbp_assignment_score(self, n_sent, n_vars, n_given, var_off, x, var_de, sp_off, sp_en, sp_feat, sp_val, giv_off, giv_label,
                              giv_gap1, pair_off, pair_v0, pair_v1, pair_gap1, pmi, pmi_w1, edT, pedT, V, ldf, h_theta_ee,
                              h_theta_ed, score):
        if n_sent == 0:
            return
        i32 = lambda p, n: _arr(p, np.int32, max(n, 1))[:n].copy()
        vo = i32(var_off, n_sent + 1)
        go, po = i32(giv_off, n_vars + 1), i32(pair_off, n_sent + 1)
        assert int(vo[-1]) == n_vars and int(go[-1]) == n_given
        xs, gl = i32(x, n_vars), i32(giv_label, n_given)
        assert ((xs >= 0) & (xs < V)).all() and ((gl >= 0) & (gl < V)).all(), 'an index outside [0, V)'
        de = i32(var_de, n_vars)
        so = i32(sp_off, n_vars + 1)
        ns, np_ = int(so[-1]), int(po[-1])
        c = Corpus(var_off=vo, var_de=de, var_label=xs, var_pos=np.zeros(n_vars, dtype=np.int32), sp_off=so, sp_en=i32(sp_en, ns),
                   sp_feat=i32(sp_feat, ns), sp_val=_arr(sp_val, np.float32, max(ns, 1))[:ns].copy(), giv_off=go, giv_label=gl,
                   giv_gap1=i32(giv_gap1, n_given), pair_off=po, pair_v0=i32(pair_v0, np_), pair_v1=i32(pair_v1, np_),
                   pair_gap1=i32(pair_gap1, np_))
        Vd = int(de.max()) + 1
        plane = lambda p, rows: _arr(p, np.float32, rows * ldf).reshape(rows, ldf)[:, :V]
        model = {'pmi': plane(pmi, V), 'pmi_w1': plane(pmi_w1, V), 'ed': plane(edT, Vd).T, 'ped': plane(pedT, Vd).T}
        _arr(score, np.float64, n_sent)[:] = maxprod_oracle.assignment_scores(model, _arr(h_theta_ee, np.float64, 3),
                                                                             _arr(h_theta_ed, np.float64, 6), c, xs)
