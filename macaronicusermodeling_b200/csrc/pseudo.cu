// K13: the pseudo-likelihood of the learner's guesses (include/mlbp.h).  For every variable i the exact conditional
//     p(y_i | y_-i) = q_i(y_i) / Z_i,   Z_i = sum_x q_i(x)
// of the model p(x) ~ prod_i U_i(x_i) prod_(a, b) T_g(x_a, x_b), with q_i formed exactly as K12 forms a Gibbs conditional
// (conditional.cuh) but with the other variables' labels as the conditioning words, and the exact gradient of its log,
//     phi(y_i) - E_{q_i / Z_i}[phi]   summed over the en_de unary factor, the given tokens and the pairwise factors touching i
// (every factor's normaliser is a constant in x_i and cancels).  No messages, no schedule, no GEMM.
#include "conditional.cuh"

#include <limits.h>

namespace mlbp {

constexpr int PK = MLBP_PL_MAX_K;

// p * G / T of one column.  Unlike the conditional, the expectations need no bit-exact reference, so the division is the
// approximate __fdividef (~2 ulp): its error is far below the 2^-22 rounding of the planes it divides.
__device__ __forceinline__ float ratio_term(float p, float g, float t) { return p > 0.f ? p * __fdividef(g, t) : 0.f; }

// E_p[feature] over this thread's 8 columns e0 .. for the plane row pair at `t_off` (the table row of the factor) and `g_off`
// (the same row of a gradient table G = T o PMI): feature(x) = G(x) / T(x)
__device__ __forceinline__ float expect8(const float p[8], const __half *__restrict__ planes, int64_t ps, int64_t t_off,
                                         int64_t g_off, int e0) {
    float th[8], tl[8], gh[8], gl[8];
    halves8(planes + t_off + e0, th);
    halves8(planes + t_off + ps + e0, tl);
    halves8(planes + g_off + e0, gh);
    halves8(planes + g_off + ps + e0, gl);
    float s = 0.f;
#pragma unroll
    for (int jj = 0; jj < 8; ++jj) s += ratio_term(p[jj], gh[jj] + gl[jj], th[jj] + tl[jj]);
    return s;
}

// grid: one CTA of GT threads per variable.  Thread t owns the E consecutive columns [t E, t E + E) as in K12; q lives in
// shared memory at qs[j * GT + t], followed by the neighbour lists of the variable's sentence.  Three CTAs per SM on the fp32
// path (at four, 64 registers, ptxas spills), two on the fp64 path.
template <typename Q>
__global__ void __launch_bounds__(GT, sizeof(Q) == 4 ? 3 : 2)
pseudo_kernel(int n_sent, int max_k, int n_vars, const int32_t *__restrict__ var_off, const int32_t *__restrict__ pair_off,
              const int32_t *__restrict__ pair_v0, const int32_t *__restrict__ pair_v1, const int32_t *__restrict__ pair_gap1,
              const int32_t *__restrict__ var_label, const int32_t *__restrict__ var_de, const int32_t *__restrict__ sp_off,
              const int32_t *__restrict__ sp_en, const int32_t *__restrict__ sp_feat, const float *__restrict__ sp_val,
              const int32_t *__restrict__ giv_off, const int32_t *__restrict__ giv_label,
              const int32_t *__restrict__ giv_gap1, const float *__restrict__ U, const __half *__restrict__ planes, int64_t ps,
              int ldv, int V, int E, double unscale, const double *__restrict__ colsums, const float *__restrict__ pmi,
              const float *__restrict__ w1, const float *__restrict__ edT, const float *__restrict__ pedT, int ldf,
              double *__restrict__ logp_var, int32_t *__restrict__ top1, int32_t *__restrict__ rank, double *__restrict__ grad,
              float *__restrict__ q_out) {
    extern __shared__ __align__(16) unsigned char smem[];
    Q *qs = reinterpret_cast<Q *>(smem);
    uint16_t *nb = reinterpret_cast<uint16_t *>(smem + (size_t)E * GT * sizeof(Q));   // [max_k (max_k - 1)]
    __shared__ int x[PK], nb_off[PK + 1];
    __shared__ int64_t row_off[PK];
    __shared__ float row_f[PK];
    __shared__ double obs[PK][2];                                     // observed pmi, pmi_w1 of each pairwise factor
    __shared__ double warp_tot[GW], red[32];
    __shared__ double s_tot, s_best[GT];
    __shared__ int s_idx[GT];
    __shared__ int s_v0, s_k, s_bad, s_cnt;

    const int i = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int e_beg = tid * E;
    if (tid == 0) {
        int lo = 0, hi = n_sent;                                      // the sentence s with var_off[s] <= i < var_off[s + 1]
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (var_off[mid] <= i) lo = mid;
            else hi = mid;
        }
        const int v0 = var_off[lo], k = var_off[lo + 1] - v0;
        int bad = !(v0 >= 0 && v0 <= i && i < v0 + k && k <= max_k && v0 + k <= n_vars);
        if (!bad) {
            const int p0 = pair_off[lo];
            bad = build_neighbours(k, p0, pair_off[lo + 1] - p0, pair_v0, pair_v1, pair_gap1, nb_off, x, nb);
        }
        s_v0 = v0;
        s_k = k;
        s_bad = bad;
        s_cnt = 0;
    }
    __syncthreads();
    const int v0 = s_v0, k = s_k, li = i - v0;
    if (!s_bad) {
        const int g0 = giv_off[i], g1 = giv_off[i + 1];                                                     // every conditioning word must name a row of the tables
        if (tid < k) {
            const int y = var_label[v0 + tid];
            x[tid] = y;
            if (y < 0 || y >= V) s_bad = 1;
        }
        for (int j = g0 + tid; j < g1; j += GT)
            if (giv_label[j] < 0 || giv_label[j] >= V) s_bad = 1;
        if (tid == 0 && g1 < g0) s_bad = 1;
    }
    __syncthreads();
    if (s_bad) {                                                      // nothing readable to condition on: NaN outputs
        const double nan = __longlong_as_double(0x7ff8000000000000ll);
        if (tid == 0) {
            logp_var[i] = nan;
            top1[i] = -1;
            rank[i] = INT_MAX;
        }
        if (grad && tid < 9) grad[(size_t)i * 9 + tid] = nan;
        if (q_out)
            for (int e = tid; e < V; e += GT) q_out[(size_t)i * ldv + e] = __int_as_float(0x7fc00000);
        return;
    }
    const int deg = nb_off[li + 1] - nb_off[li];
    if (tid < deg) {
        const int yi = x[li];
        const int ent = nb[nb_off[li] + tid];
        factor_row(ent, x, ps, ldv, V, unscale, colsums, row_off[tid], row_f[tid]);
        if (grad) {
            const int y = x[ent & 63];
            const size_t cell = (ent >> 6) & 1 ? (size_t)y * ldf + yi : (size_t)yi * ldf + y;
            obs[tid][0] = (double)pmi[cell];
            obs[tid][1] = (ent >> 7) & 1 ? (double)w1[cell] : 0.0;
        }
    }
    __syncthreads();
    // q over this thread's columns and their float64 sum in column order; Z in K12's block order
    const float *urow = U + (size_t)i * ldv;
    double t_sum = 0.0;
    for (int j0 = 0; j0 < E; j0 += 8) {
        const int e0 = e_beg + j0;
        Q q[8];
        if (e0 < V) conditional8(q, urow, e0, deg, planes, row_off, row_f, ps);
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) {
            const Q v = (e0 + jj < V) ? q[jj] : Q(0);
            qs[(j0 + jj) * GT + tid] = v;
            t_sum = __dadd_rn(t_sum, to_d(v));
        }
    }
    const double base = scan_base(t_sum, warp_tot, lane, warp);
    if (e_beg <= V - 1 && V - 1 < e_beg + E) s_tot = __dadd_rn(base, t_sum);
    __syncthreads();
    const double Z = s_tot;
    const int yi = x[li];
    const int g0 = giv_off[i], g1 = giv_off[i + 1];
    const Q qy = qs[(yi % E) * GT + yi / E];
    // arg-max (first index on ties) and rank of the label over this thread's columns
    double best = -1.0;
    int bi = INT_MAX, cnt = 0;
    for (int j = 0; j < E && e_beg + j < V; ++j) {
        const Q qv = qs[j * GT + tid];
        if (to_d(qv) > best) {
            best = to_d(qv);
            bi = e_beg + j;
        }
        cnt += qv > qy;
    }
    s_best[tid] = best;
    s_idx[tid] = bi;
    atomicAdd(&s_cnt, cnt);
    const bool ok = Z > 0.0;
    if (q_out) {                                                      // normalised row, coalesced
        for (int e = tid; e < V; e += GT)
            q_out[(size_t)i * ldv + e] = ok ? (float)__ddiv_rn(to_d(qs[(e % E) * GT + e / E]), Z) : 0.f;
    }
    if (grad) {
        // E_p of pmi, pmi_w1 (pairwise factors and given tokens) and of ed, ped (the en_de factor): fp32 per thread, float64
        // across the block.  p(x) = q(x) / Z; a column with p(x) = 0 contributes 0 (the planes are not divided there).
        const double invz = ok ? 1.0 / Z : 0.0;
        const int d = var_de[i];
        float e_pmi = 0.f, e_w1 = 0.f, e_ed = 0.f, e_ped = 0.f;
        for (int j0 = 0; j0 < E; j0 += 8) {
            const int e0 = e_beg + j0;
            if (e0 >= V) break;
            float p[8];
#pragma unroll
            for (int jj = 0; jj < 8; ++jj) p[jj] = (float)(to_d(qs[(j0 + jj) * GT + tid]) * invz);
#pragma unroll 1
            for (int m = 0; m < deg; ++m) {
                const int ent = nb[nb_off[li] + m];
                const int dim1 = (ent >> 6) & 1, g = (ent >> 7) & 1;
                const int64_t yrow = (int64_t)x[ent & 63] * ldv;
                // gradient rows at the table row's orientation: G / G1 (planes 8 / 10) for dim 1, Gt / G1t (14 / 16) for dim 0
                e_pmi += expect8(p, planes, ps, row_off[m], (dim1 ? (g ? 10 : 8) : (g ? 16 : 14)) * ps + yrow, e0);
                if (g) e_w1 += expect8(p, planes, ps, row_off[m], (dim1 ? 12 : 18) * ps + yrow, e0);
            }
#pragma unroll 1
            for (int j = g0; j < g1; ++j) {                          // given tokens: row o of Tt / T1t, as K1 reads them
                const int g = giv_gap1[j] ? 1 : 0;
                const int64_t orow = (int64_t)giv_label[j] * ldv;
                const int64_t t_off = (g ? 6 : 2) * ps + orow;
                e_pmi += expect8(p, planes, ps, t_off, (g ? 16 : 14) * ps + orow, e0);
                if (g) e_w1 += expect8(p, planes, ps, t_off, 18 * ps + orow, e0);
            }
            if (d >= 0) {
                const float4 a0 = *reinterpret_cast<const float4 *>(edT + (size_t)d * ldf + e0);
                const float4 a1 = *reinterpret_cast<const float4 *>(edT + (size_t)d * ldf + e0 + 4);
                const float4 b0 = *reinterpret_cast<const float4 *>(pedT + (size_t)d * ldf + e0);
                const float4 b1 = *reinterpret_cast<const float4 *>(pedT + (size_t)d * ldf + e0 + 4);
                const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
                const float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
                for (int jj = 0; jj < 8; ++jj) {
                    e_ed += p[jj] > 0.f ? p[jj] * a[jj] : 0.f;
                    e_ped += p[jj] > 0.f ? p[jj] * b[jj] : 0.f;
                }
            }
        }
        const double E_pmi = block_sum((double)e_pmi, red), E_w1 = block_sum((double)e_w1, red);
        const double E_ed = block_sum((double)e_ed, red), E_ped = block_sum((double)e_ped, red);
        if (tid == 0) {
            double o_pmi = 0.0, o_w1 = 0.0, g_ed = 0.0, g_ped = 0.0, g_sp[3] = {0.0, 0.0, 0.0};
            for (int m = 0; m < deg; ++m) {
                o_pmi += obs[m][0];
                o_w1 += obs[m][1];
            }
            for (int j = g0; j < g1; ++j) {
                const size_t cell = (size_t)yi * ldf + giv_label[j];
                o_pmi += (double)pmi[cell];
                if (giv_gap1[j]) o_w1 += (double)w1[cell];
            }
            if (d >= 0) {
                g_ed = (double)edT[(size_t)d * ldf + yi] - E_ed;
                g_ped = (double)pedT[(size_t)d * ldf + yi] - E_ped;
                for (int s = sp_off[i]; s < sp_off[i + 1]; ++s) {   // sparse features: val at x = sp_en only
                    const int e = sp_en[s], f = sp_feat[s];
                    const double pe = (e >= 0 && e < V) ? to_d(qs[(e % E) * GT + e / E]) * invz : 0.0;
                    const double t = (double)sp_val[s] * ((e == yi ? 1.0 : 0.0) - pe);
#pragma unroll
                    for (int c = 0; c < 3; ++c) g_sp[c] += f == 2 + c ? t : 0.0;
                }
            }
            double *gr = grad + (size_t)i * 9;                         // bias components: exactly 0
            gr[0] = o_pmi - E_pmi;
            gr[1] = o_w1 - E_w1;
            gr[2] = 0.0;
            gr[3] = g_ed;
            gr[4] = g_ped;
            gr[5] = g_sp[0];
            gr[6] = g_sp[1];
            gr[7] = g_sp[2];
            gr[8] = 0.0;
        }
    }
    __syncthreads();
    if (tid == 0) {
        for (int t = 1; t < GT; ++t)
            if (s_best[t] > best || (s_best[t] == best && s_idx[t] < bi)) best = s_best[t], bi = s_idx[t];
        top1[i] = bi;
        rank[i] = s_cnt;
        logp_var[i] = (to_d(qy) > 0.0 && ok) ? log(__ddiv_rn(to_d(qy), Z)) : -99.99;
    }
}

}  // namespace mlbp

using namespace mlbp;

extern "C" int mlbp_pseudo_likelihood(int n_sent, int max_k, int n_vars, const int32_t *var_off, const int32_t *pair_off,
                                      const int32_t *pair_v0, const int32_t *pair_v1, const int32_t *pair_gap1,
                                      const int32_t *var_label, const int32_t *var_de, const int32_t *sp_off, const int32_t *sp_en,
                                      const int32_t *sp_feat, const float *sp_val, const int32_t *giv_off,
                                      const int32_t *giv_label, const int32_t *giv_gap1, const float *U, const void *planes,
                                      int64_t plane_stride, int ldv, int V, int scale_exp, const double *colsums,
                                      const float *pmi, const float *pmi_w1, const float *edT, const float *pedT, int ldf,
                                      float range_log2, double *logp_var, int32_t *top1, int32_t *rank, double *grad,
                                      float *beliefs, void *stream) {
    MLBP_CHECK_ARG(var_off && pair_off && pair_v0 && pair_v1 && pair_gap1 && var_label && giv_off && giv_label && giv_gap1 && U &&
                   planes && colsums && logp_var && top1 && rank, "pseudo_likelihood: null pointer");
    MLBP_CHECK_ARG(!grad || (var_de && sp_off && sp_en && sp_feat && sp_val && pmi && pmi_w1 && edT && pedT),
                   "pseudo_likelihood: the gradient needs var_de, the sparse lists and the feature planes");
    MLBP_CHECK_ARG(n_sent >= 0 && n_vars >= 0 && V >= 1 && ldv >= V && ldv % 8 == 0 && plane_stride % 8 == 0 &&
                   plane_stride >= (int64_t)V * ldv && (!grad || (ldf >= V && ldf % 8 == 0)),
                   "pseudo_likelihood: bad n_sent / n_vars / V / ldv / plane_stride / ldf");
    MLBP_CHECK_ARG(((reinterpret_cast<uintptr_t>(U) | reinterpret_cast<uintptr_t>(planes) | reinterpret_cast<uintptr_t>(beliefs) |
                     (grad ? reinterpret_cast<uintptr_t>(edT) | reinterpret_cast<uintptr_t>(pedT) : 0)) % 16) == 0,
                   "pseudo_likelihood: U, planes, beliefs, edT and pedT need 16-byte aligned rows");
    MLBP_CHECK_ARG(n_sent == 0 || max_k >= 1, "pseudo_likelihood: max_k < 1");
    if (max_k > MLBP_PL_MAX_K) {
        set_error("pseudo_likelihood: sentences of %d variables, at most %d are supported", max_k, MLBP_PL_MAX_K);
        return MLBP_ERR_UNSUPPORTED;
    }
    if (n_sent == 0 || n_vars == 0) return MLBP_OK;
    const bool f64 = !(range_log2 >= 0.0f && range_log2 < 100.0f);
    const int E = ((V + 8 * GT - 1) / (8 * GT)) * 8;
    const size_t shm = (size_t)E * GT * (f64 ? 8 : 4) + (size_t)max_k * (max_k - 1) * 2;
    int dev = 0, optin = 0;
    MLBP_CUDA(cudaGetDevice(&dev));
    MLBP_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    if (shm + 8192 > (size_t)optin) {
        set_error("pseudo_likelihood: V = %d needs %zu bytes of shared memory per CTA (%s products), the device has %d", V, shm,
                  f64 ? "fp64" : "fp32", optin);
        return MLBP_ERR_UNSUPPORTED;
    }
    auto kern = f64 ? pseudo_kernel<double> : pseudo_kernel<float>;
    MLBP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)shm));
    kern<<<n_vars, GT, shm, as_stream(stream)>>>(n_sent, max_k, n_vars, var_off, pair_off, pair_v0, pair_v1, pair_gap1, var_label,
                                                 var_de, sp_off, sp_en, sp_feat, sp_val, giv_off, giv_label, giv_gap1, U,
                                                 (const __half *)planes, plane_stride, ldv, V, E, ldexp(1.0, -scale_exp), colsums,
                                                 pmi, pmi_w1, edT, pedT, ldf, logp_var, top1, rank, grad, beliefs);
    MLBP_LAUNCH_CHECK();
    return MLBP_OK;
}
