// K9: the joint log-likelihood of each sentence's labels, estimated from the final messages (Bethe free energy).
//
// The model's joint is p(y) ∝ prod_i U_i(y_i) prod_F T_F(y_i, y_j).  Its loopy-BP estimate, written around the per-variable
// log-marginals logp_var that K5 already produced, is
//     log p_B(y) = sum_i logp_var_i
//                + sum_F [ log T_F(y_i, y_j) - log Z_F + sum_{k in F} ( log O_{F,k} - log mu_{F->k}(y_k) ) ]
//     Z_F = nu_{i->F}' T_F nu_{j->F},   O_{F,k} = nu_{k->F} . mu_{F->k}
// with nu the final variable->factor messages (the c / r rows K6a reads) and mu the final factor->variable messages (the D rows
// K5 reads).  Every stored row enters once with + and once with -, so the arbitrary scales of the rows cancel; only Z_F, which
// K6a formed against the scaled table planes, carries a known power of two.  Exact on trees.
//
// Two launches: one warp per pairwise factor for the two V-length dots (HBM-bound, 16 V bytes per factor) and the gathers,
// then one warp per sentence for the segmented sum.  Both in a fixed order: deterministic.
#include "common.cuh"

namespace mlbp {

constexpr int JOINT_WARPS = 8;

__device__ __forceinline__ void dot8(const uint4 h8, const uint4 l8, const float4 d0, const float4 d1, double &acc) {
    const __half2 *hh = reinterpret_cast<const __half2 *>(&h8), *ll = reinterpret_cast<const __half2 *>(&l8);
    const float d[8] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const float2 h = __half22float2(hh[q]), l = __half22float2(ll[q]);
        acc += (double)((h.x + l.x) * d[2 * q]);
        acc += (double)((h.y + l.y) * d[2 * q + 1]);
    }
}

// VEC: every row base is 16-byte aligned (8 fp16 / 4 fp32 per load); otherwise element loads
template <bool VEC>
__global__ void __launch_bounds__(32 * JOINT_WARPS)
joint_pair_kernel(int n_pairs, const int32_t *__restrict__ c_row, const int32_t *__restrict__ r_row,
                  const int32_t *__restrict__ m0_row, const int32_t *__restrict__ m1_row, const int32_t *__restrict__ pair_v0,
                  const int32_t *__restrict__ pair_v1, const int32_t *__restrict__ var_label,
                  const int32_t *__restrict__ gap1, const double *__restrict__ pair_stats, const __half *__restrict__ A_hi,
                  const __half *__restrict__ A_lo, const float *__restrict__ D, int ldv, int V, const float *__restrict__ pmi,
                  const float *__restrict__ w1, int ldf, double th0, double th1, double th2, double log_z_scale,
                  double *__restrict__ pair_term) {
    const int f = blockIdx.x * JOINT_WARPS + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (f >= n_pairs) return;
    // a factor->variable message still at its uniform initial value is read as the constant-one row D[0] (as K3 / K5 do)
    const size_t cr = (size_t)c_row[f] * ldv, rr = (size_t)r_row[f] * ldv;
    const float *d0 = D + (size_t)max(m0_row[f], 0) * ldv, *d1 = D + (size_t)max(m1_row[f], 0) * ldv;
    const __half *ch = A_hi + cr, *cl = A_lo + cr, *rh = A_hi + rr, *rl = A_lo + rr;
    // O_0 = c . mu_0, O_1 = r . mu_1: fp32 products, float64 sums per lane, lanes combined in a fixed butterfly
    double o0 = 0.0, o1 = 0.0;
    int k = lane;
    if (VEC) {
        const int n8 = V >> 3;
        for (int k8 = lane; k8 < n8; k8 += 32) {
            const uint4 ch8 = __ldg(reinterpret_cast<const uint4 *>(ch) + k8), cl8 = __ldg(reinterpret_cast<const uint4 *>(cl) + k8);
            const uint4 rh8 = __ldg(reinterpret_cast<const uint4 *>(rh) + k8), rl8 = __ldg(reinterpret_cast<const uint4 *>(rl) + k8);
            const float4 a0 = __ldg(reinterpret_cast<const float4 *>(d0) + 2 * k8), a1 = __ldg(reinterpret_cast<const float4 *>(d0) + 2 * k8 + 1);
            const float4 b0 = __ldg(reinterpret_cast<const float4 *>(d1) + 2 * k8), b1 = __ldg(reinterpret_cast<const float4 *>(d1) + 2 * k8 + 1);
            dot8(ch8, cl8, a0, a1, o0);
            dot8(rh8, rl8, b0, b1, o1);
        }
        k = 8 * n8 + lane;                                         // the padding of a row is never read (it may hold anything)
    }
    for (; k < V; k += 32) {
        o0 += (double)((__half2float(ch[k]) + __half2float(cl[k])) * d0[k]);
        o1 += (double)((__half2float(rh[k]) + __half2float(rl[k])) * d1[k]);
    }
    o0 = warp_sum(o0);
    o1 = warp_sum(o1);
    if (lane == 0) {
        const int y0 = var_label[pair_v0[f]], y1 = var_label[pair_v1[f]];
        const size_t cell = (size_t)y0 * ldf + y1;
        // log T(y0, y1) from the feature planes in float64 (train.py:218-219, :252-253), on the scale of the unscaled table
        double log_t = th0 * (double)pmi[cell] + th2;
        if (gap1[f]) log_t += th1 * (double)w1[cell];
        const double log_z = log(pair_stats[3 * (size_t)f]) - log_z_scale;
        pair_term[f] = log_t - log_z + log(o0) + log(o1) - log((double)d0[y0]) - log((double)d1[y1]);
    }
}

// one warp per sentence; the variables are summed in the order of mlbp_gradient_reduce's logp_sent, so a sentence without
// pairwise factors reports exactly its logp_sent
__global__ void joint_reduce_kernel(int n_sent, const int32_t *__restrict__ sent_var_off, const int32_t *__restrict__ sent_fac_off,
                                    const double *__restrict__ logp_var, const double *__restrict__ pair_term,
                                    double *__restrict__ logp_joint) {
    const int s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (s >= n_sent) return;
    double lp = 0.0, pt = 0.0;
    bool zero = false;
    for (int v = sent_var_off[s] + lane; v < sent_var_off[s + 1]; v += 32) {
        const double x = logp_var[v];
        zero = zero || x == -99.99;                                 // K5's value for a label of belief 0 (LBP.py:247-259)
        lp += x;
    }
    for (int f = sent_fac_off[s] + lane; f < sent_fac_off[s + 1]; f += 32) pt += pair_term[f];
    lp = warp_sum(lp);
    pt = warp_sum(pt);
    zero = __any_sync(0xffffffffu, zero);
    if (lane == 0) logp_joint[s] = zero ? -INFINITY : lp + pt;
}

}  // namespace mlbp

using namespace mlbp;

extern "C" int mlbp_joint_logp(int n_sent, int n_pairs, const int32_t *sent_var_off, const int32_t *sent_fac_off,
                               const double *logp_var, const int32_t *c_row, const int32_t *r_row, const int32_t *m0_row,
                               const int32_t *m1_row, const int32_t *pair_v0, const int32_t *pair_v1, const int32_t *var_label,
                               const int32_t *pair_gap1, const double *pair_stats, const void *A_hi, const void *A_lo,
                               const float *D, int ldv, int V, const float *pmi, const float *pmi_w1, int ldf,
                               const double *h_theta_ee, int z_scale_log2, double *pair_term, double *logp_joint,
                               void *stream) {
    MLBP_CHECK_ARG(n_sent >= 0 && n_pairs >= 0, "joint_logp: negative count");
    if (n_sent == 0 && n_pairs == 0) return MLBP_OK;
    MLBP_CHECK_ARG(n_sent > 0, "joint_logp: pairwise factors without sentences");
    MLBP_CHECK_ARG(sent_var_off && sent_fac_off && logp_var && logp_joint, "joint_logp: null pointer");
    if (n_pairs > 0) {
        MLBP_CHECK_ARG(c_row && r_row && m0_row && m1_row && pair_v0 && pair_v1 && var_label && pair_gap1 && pair_stats && A_hi &&
                       A_lo && D && pmi && pmi_w1 && h_theta_ee && pair_term, "joint_logp: null pointer");
        MLBP_CHECK_ARG(V > 0 && ldv >= V && ldf >= V, "joint_logp: bad V / ldv / ldf");
        MLBP_CHECK_ARG(z_scale_log2 > -1000 && z_scale_log2 < 1000, "joint_logp: z_scale_log2 out of range");
        for (int i = 0; i < 3; ++i)
            MLBP_CHECK_ARG(h_theta_ee[i] == h_theta_ee[i] && h_theta_ee[i] - h_theta_ee[i] == 0.0, "joint_logp: theta_ee not finite");
    }
    const cudaStream_t st = as_stream(stream);
    if (n_pairs > 0) {
        const bool vec = (ldv % 8) == 0 && ((reinterpret_cast<uintptr_t>(A_hi) | reinterpret_cast<uintptr_t>(A_lo) |
                                             reinterpret_cast<uintptr_t>(D)) % 16) == 0;
        const double lzs = (double)z_scale_log2 * 0.69314718055994530942;
        const int blocks = (n_pairs + JOINT_WARPS - 1) / JOINT_WARPS;
        auto kern = vec ? joint_pair_kernel<true> : joint_pair_kernel<false>;
        kern<<<blocks, 32 * JOINT_WARPS, 0, st>>>(n_pairs, c_row, r_row, m0_row, m1_row, pair_v0, pair_v1, var_label, pair_gap1,
                                                  pair_stats, (const __half *)A_hi, (const __half *)A_lo, D, ldv, V, pmi, pmi_w1,
                                                  ldf, h_theta_ee[0], h_theta_ee[1], h_theta_ee[2], lzs, pair_term);
        MLBP_LAUNCH_CHECK();
    }
    const int threads = 128, warps_per_block = threads / 32;
    joint_reduce_kernel<<<(n_sent + warps_per_block - 1) / warps_per_block, threads, 0, st>>>(n_sent, sent_var_off, sent_fac_off,
                                                                                             logp_var, pair_term, logp_joint);
    MLBP_LAUNCH_CHECK();
    return MLBP_OK;
}
