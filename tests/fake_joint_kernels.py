"""TEST DOUBLE for K9 (mlbp_joint_logp, csrc/joint.cu): FakeKernels plus the joint log-likelihood, emulated in NumPy float64 on
host pointers with the kernel's checks, row conventions (mk_row < 0 reads D row 0) and -inf rule.  Never imported by the
package."""
import numpy as np

from fake_kernels import FakeKernels, _arr


class JointKernels(FakeKernels):
    """FakeKernels plus mlbp_joint_logp"""

    def mlbp_joint_logp(self, n_sent, n_pairs, sent_var_off, sent_fac_off, logp_var, c_row, r_row, m0_row, m1_row, pair_v0,
                        pair_v1, var_label, pair_gap1, pair_stats, A_hi, A_lo, D, ldv, V, pmi, pmi_w1, ldf, h_theta_ee,
                        z_scale_log2, pair_term, logp_joint):
        assert n_sent >= 0 and n_pairs >= 0
        if n_sent == 0:
            return
        vo, fo = _arr(sent_var_off, np.int32, n_sent + 1), _arr(sent_fac_off, np.int32, n_sent + 1)
        assert int(fo[-1]) == n_pairs
        lv = _arr(logp_var, np.float64, int(vo[-1]))
        term = np.zeros(n_pairs)
        if n_pairs:
            idx = lambda p: _arr(p, np.int32, n_pairs)
            cr, rr, m0, m1, v0, v1, g1 = (idx(p) for p in (c_row, r_row, m0_row, m1_row, pair_v0, pair_v1, pair_gap1))
            lab = _arr(var_label, np.int32, int(vo[-1]))
            a_rows = int(max(cr.max(), rr.max())) + 1
            H = _arr(A_hi, np.float16, a_rows * ldv).reshape(-1, ldv)[:, :V].astype(np.float32)
            L = _arr(A_lo, np.float16, a_rows * ldv).reshape(-1, ldv)[:, :V].astype(np.float32)
            Dm = _arr(D, np.float32, (int(max(m0.max(), m1.max(), 0)) + 1) * ldv).reshape(-1, ldv)[:, :V]
            st = _arr(pair_stats, np.float64, 3 * n_pairs).reshape(-1, 3)
            th = _arr(h_theta_ee, np.float64, 3)
            P = _arr(pmi, np.float32, V * ldf).reshape(V, ldf)
            W = _arr(pmi_w1, np.float32, V * ldf).reshape(V, ldf)
            with np.errstate(divide='ignore', invalid='ignore'):
                for f in range(n_pairs):
                    y0, y1 = int(lab[v0[f]]), int(lab[v1[f]])
                    mu0, mu1 = Dm[max(int(m0[f]), 0)], Dm[max(int(m1[f]), 0)]
                    o0 = ((H[cr[f]] + L[cr[f]]) * mu0).astype(np.float64).sum()
                    o1 = ((H[rr[f]] + L[rr[f]]) * mu1).astype(np.float64).sum()
                    log_t = th[0] * float(P[y0, y1]) + th[2] + (th[1] * float(W[y0, y1]) if g1[f] else 0.0)
                    log_z = np.log(st[f, 0]) - z_scale_log2 * np.log(2.0)
                    term[f] = log_t - log_z + np.log(o0) + np.log(o1) - np.log(float(mu0[y0])) - np.log(float(mu1[y1]))
            _arr(pair_term, np.float64, n_pairs)[:] = term
        out = _arr(logp_joint, np.float64, n_sent)
        for s in range(n_sent):
            x = lv[vo[s]:vo[s + 1]]
            out[s] = -np.inf if (x == -99.99).any() else x.sum() + term[fo[s]:fo[s + 1]].sum()
