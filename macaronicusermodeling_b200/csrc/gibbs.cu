// K12: a systematic-scan Gibbs sampler of each sentence's joint guesses, and its chain-averaging reduction (include/mlbp.h).
//
// One CTA of MLBP_GIBBS_THREADS threads runs one (sentence, chain).  An update of variable i forms the full conditional
// q_i(x) for every x < V from K1's row U_i and one table row per pairwise factor that touches i (the other variables' current
// words act like given tokens), takes the float64 running sum of q in a fixed block-wide order, draws x_i with a counter-based
// Philox uniform and, in kept sweeps, adds q_i / sum to the chain's Rao-Blackwell row.  Everything is ordered so that a NumPy
// emulation (tests/gibbs_oracle.py) reproduces every q, every sum and every draw bit for bit.
#include "conditional.cuh"

#include <limits.h>

namespace mlbp {

// Philox4x32-10 (Salmon et al., SC'11; the constants of Random123), counter c, key (k0, k1)
__host__ __device__ __forceinline__ void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1) {
    for (int r = 0; r < 10; ++r) {
        const uint64_t p0 = (uint64_t)0xD2511F53u * c[0], p1 = (uint64_t)0xCD9E8D57u * c[2];
        const uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0, hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
        c[0] = hi1 ^ c[1] ^ k0;
        c[1] = lo1;
        c[2] = hi0 ^ c[3] ^ k1;
        c[3] = lo0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
}

// grid: n_sent * chains CTAs, blockIdx.x = s * chains + c.  Thread t owns the E consecutive columns [t E, t E + E) (E a multiple
// of 8); its q values live in shared memory at qs[j * GT + t] (conflict-free), followed by the neighbour lists.
// 4 CTAs per SM at 64 registers on the fp32 path (V = 10 000: 41 KB of shared memory each); the fp64 path holds two
template <typename Q>
__global__ void __launch_bounds__(GT, sizeof(Q) == 4 ? 4 : 2)
gibbs_kernel(int max_k, const int32_t *__restrict__ var_off, const int32_t *__restrict__ pair_off,
             const int32_t *__restrict__ pair_v0, const int32_t *__restrict__ pair_v1, const int32_t *__restrict__ pair_gap1,
             const int32_t *__restrict__ sent_id, const float *__restrict__ U, const __half *__restrict__ planes, int64_t ps,
             int ldv, int V, int E, double unscale, const double *__restrict__ colsums, int chains, int burn_in, int n_keep,
             uint32_t key0, uint32_t key1, int n_vars, float *__restrict__ acc, int32_t *__restrict__ samples) {
    extern __shared__ __align__(16) unsigned char smem[];
    Q *qs = reinterpret_cast<Q *>(smem);
    uint16_t *nb = reinterpret_cast<uint16_t *>(smem + (size_t)E * GT * sizeof(Q));   // [max_k (max_k - 1)]
    __shared__ int x[MLBP_GIBBS_MAX_K], nb_off[MLBP_GIBBS_MAX_K + 1];
    __shared__ int64_t row_off[MLBP_GIBBS_MAX_K];
    __shared__ float row_f[MLBP_GIBBS_MAX_K];
    __shared__ double warp_tot[GW];
    __shared__ double s_tot;
    __shared__ int s_hit, s_last, s_bad;

    const int s = blockIdx.x / chains, c = blockIdx.x % chains;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int v0 = var_off[s], k = var_off[s + 1] - v0;
    const int p0 = pair_off[s], n_p = pair_off[s + 1] - p0;
    const int e_beg = tid * E;
    if (k < 1 || k > max_k || v0 < 0 || v0 + k > n_vars) return;     // outside the caller's stated bounds: nothing to own
    if (tid == 0) s_bad = build_neighbours(k, p0, n_p, pair_v0, pair_v1, pair_gap1, nb_off, x, nb);   // x: fill cursor
    __syncthreads();
    if (s_bad) {                                                       // a pair list the sampler cannot read: NaN rows
        for (int i = 0; i < k; ++i)
            for (int e = tid; e < V; e += GT) acc[((size_t)c * n_vars + v0 + i) * ldv + e] = __int_as_float(0x7fc00000);
        return;
    }
    const uint32_t sid = (uint32_t)sent_id[s];
    const int n_sweeps = 1 + burn_in + n_keep;
    for (int sw = 0; sw < n_sweeps; ++sw) {
        const bool kept = sw > burn_in;
        for (int i = 0; i < k; ++i) {
            const int deg = sw == 0 ? 0 : nb_off[i + 1] - nb_off[i];    // sweep 0 draws from U_i alone
            if (tid < deg) {
                const int ent = nb[nb_off[i] + tid];
                factor_row(ent, x, ps, ldv, V, unscale, colsums, row_off[tid], row_f[tid]);
            }
            if (tid == 0) {
                s_hit = INT_MAX;
                s_last = -1;
            }
            __syncthreads();
            // q over this thread's columns, and their float64 sum in column order
            const float *urow = U + (size_t)(v0 + i) * ldv;
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
            const double base = scan_base(t_sum, warp_tot, lane, warp);   // C(e) = base + (running sum of this thread up to e)
            if (e_beg <= V - 1 && V - 1 < e_beg + E) s_tot = __dadd_rn(base, t_sum);
            __syncthreads();
            const double tot = s_tot;                                  // C(V - 1)
            uint32_t ctr[4] = {sid, (uint32_t)c, (uint32_t)sw, (uint32_t)i};
            philox4x32_10(ctr, key0, key1);
            const double u = ((double)(ctr[0] >> 5) * 67108864.0 + (double)(ctr[1] >> 6)) * 0x1p-53;
            const bool ok = tot > 0.0 && tot - tot == 0.0;
            if (ok) {                                                  // smallest x with C(x) > u C(V - 1)
                const double target = __dmul_rn(u, tot);
                double run = 0.0;
                int hit = INT_MAX, last = -1;
                for (int j = 0; j < E && e_beg + j < V; ++j) {
                    const Q qv = qs[j * GT + tid];
                    run = __dadd_rn(run, to_d(qv));
                    if (hit == INT_MAX && __dadd_rn(base, run) > target) hit = e_beg + j;
                    if (qv > Q(0)) last = e_beg + j;
                }
                if (hit != INT_MAX) atomicMin(&s_hit, hit);
                if (last >= 0) atomicMax(&s_last, last);
            }
            __syncthreads();
            // no x qualifies only when u C(V - 1) rounds up to C(V - 1): the last word of positive mass.  A zero or non-finite
            // sum draws uniformly (K3's fallback)
            const int xi = ok ? (s_hit != INT_MAX ? s_hit : s_last) : min((int)(u * (double)V), V - 1);
            if (tid == 0) x[i] = xi;
            if (kept) {                                                // Rao-Blackwell row: acc += fp32(q / C(V - 1))
                float *arow = acc + ((size_t)c * n_vars + v0 + i) * ldv;
                const bool first = sw == burn_in + 1;
                const float uni = (float)(1.0 / (double)V);
                for (int j0 = 0; j0 < E; j0 += 8) {
                    const int e0 = e_beg + j0;
                    if (e0 >= V) break;
                    const bool full = e0 + 8 <= V;
                    float a[8];
                    if (!first && full) {
                        const float4 aa = *reinterpret_cast<const float4 *>(arow + e0);
                        const float4 ab = *reinterpret_cast<const float4 *>(arow + e0 + 4);
                        a[0] = aa.x; a[1] = aa.y; a[2] = aa.z; a[3] = aa.w;
                        a[4] = ab.x; a[5] = ab.y; a[6] = ab.z; a[7] = ab.w;
                    } else {
#pragma unroll
                        for (int jj = 0; jj < 8; ++jj) a[jj] = (!first && e0 + jj < V) ? arow[e0 + jj] : 0.f;
                    }
#pragma unroll
                    for (int jj = 0; jj < 8; ++jj) {
                        const float term = ok ? (float)__ddiv_rn(to_d(qs[(j0 + jj) * GT + tid]), tot) : uni;
                        a[jj] = first ? term : __fadd_rn(a[jj], term);
                    }
                    if (full) {
                        *reinterpret_cast<float4 *>(arow + e0) = make_float4(a[0], a[1], a[2], a[3]);
                        *reinterpret_cast<float4 *>(arow + e0 + 4) = make_float4(a[4], a[5], a[6], a[7]);
                    } else {
#pragma unroll
                        for (int jj = 0; jj < 8; ++jj)
                            if (e0 + jj < V) arow[e0 + jj] = a[jj];
                    }
                }
            }
            __syncthreads();                                           // x[i] visible; q, rows and flags free for the next update
        }
        if (kept && samples && tid < k) samples[((size_t)c * n_keep + (sw - burn_in - 1)) * n_vars + v0 + tid] = x[tid];
    }
}

// one CTA per variable: the chain average in float64 (chains in ascending order) and K5's per-variable outputs on it
__global__ void __launch_bounds__(256)
gibbs_reduce_kernel(int n_vars, int chains, int n_keep, const float *__restrict__ acc, int ldv, int V,
                    const int32_t *__restrict__ var_label, float *__restrict__ marg, double *__restrict__ label_prob,
                    double *__restrict__ logp_var, int32_t *__restrict__ top1, int32_t *__restrict__ rank) {
    __shared__ double s_best[256];
    __shared__ int s_idx[256];
    __shared__ int s_cnt;
    const int i = blockIdx.x, tid = threadIdx.x;
    const double den = (double)chains * (double)n_keep;
    const int lab = var_label[i];
    const bool lv = lab >= 0 && lab < V;
    auto mean = [&](int x) {
        double s = 0.0;
        for (int c = 0; c < chains; ++c) s = __dadd_rn(s, (double)acc[((size_t)c * n_vars + i) * ldv + x]);
        return __ddiv_rn(s, den);
    };
    const double ml = lv ? mean(lab) : __longlong_as_double(0x7ff8000000000000ll);
    if (tid == 0) s_cnt = 0;
    __syncthreads();
    double best = -1.0;
    int bi = INT_MAX, cnt = 0;
    for (int x = tid; x < V; x += 256) {
        const double m = mean(x);
        marg[(size_t)i * ldv + x] = (float)m;
        if (m > best) {
            best = m;
            bi = x;
        }
        cnt += m > ml;
    }
    s_best[tid] = best;
    s_idx[tid] = bi;
    atomicAdd(&s_cnt, cnt);
    for (int c = tid; c < chains; c += 256)
        label_prob[(size_t)i * chains + c] =
            lv ? __ddiv_rn((double)acc[((size_t)c * n_vars + i) * ldv + lab], (double)n_keep) : ml;
    __syncthreads();
    if (tid == 0) {
        for (int t = 1; t < 256; ++t)
            if (s_best[t] > best || (s_best[t] == best && s_idx[t] < bi)) best = s_best[t], bi = s_idx[t];
        top1[i] = bi;
        rank[i] = s_cnt;
        logp_var[i] = ml > 0.0 ? log(ml) : (lv ? -99.99 : ml);
    }
}

}  // namespace mlbp

using namespace mlbp;

extern "C" int mlbp_gibbs_sample(int n_sent, int max_k, int n_vars, const int32_t *var_off, const int32_t *pair_off,
                                 const int32_t *pair_v0, const int32_t *pair_v1, const int32_t *pair_gap1, const int32_t *sent_id,
                                 const float *U, const void *planes, int64_t plane_stride, int ldv, int V, int scale_exp,
                                 const double *colsums, int chains, int burn_in, int n_keep, uint64_t seed, float range_log2,
                                 float *acc, int32_t *samples, void *stream) {
    MLBP_CHECK_ARG(var_off && pair_off && pair_v0 && pair_v1 && pair_gap1 && sent_id && U && planes && colsums && acc,
                   "gibbs_sample: null pointer");
    MLBP_CHECK_ARG(n_sent >= 0 && n_vars >= 0 && V >= 1 && ldv >= V && ldv % 8 == 0 && plane_stride % 8 == 0 &&
                   plane_stride >= (int64_t)V * ldv, "gibbs_sample: bad n_sent / n_vars / V / ldv / plane_stride");
    MLBP_CHECK_ARG(((reinterpret_cast<uintptr_t>(U) | reinterpret_cast<uintptr_t>(planes) | reinterpret_cast<uintptr_t>(acc)) %
                    16) == 0, "gibbs_sample: U, planes and acc need 16-byte aligned rows");
    MLBP_CHECK_ARG(chains >= 1 && n_keep >= 1 && burn_in >= 0, "gibbs_sample: chains and n_keep must be >= 1, burn_in >= 0");
    MLBP_CHECK_ARG((int64_t)burn_in + n_keep < INT_MAX, "gibbs_sample: too many sweeps");
    MLBP_CHECK_ARG(n_sent == 0 || max_k >= 1, "gibbs_sample: max_k < 1");
    if (max_k > MLBP_GIBBS_MAX_K) {
        set_error("gibbs_sample: sentences of %d variables, at most %d are supported", max_k, MLBP_GIBBS_MAX_K);
        return MLBP_ERR_UNSUPPORTED;
    }
    if (n_sent == 0) return MLBP_OK;
    MLBP_CHECK_ARG((int64_t)n_sent * chains < INT_MAX, "gibbs_sample: too many (sentence, chain) pairs");
    const bool f64 = !(range_log2 >= 0.0f && range_log2 < 100.0f);
    const int E = ((V + 8 * GT - 1) / (8 * GT)) * 8;
    const size_t shm = (size_t)E * GT * (f64 ? 8 : 4) + (size_t)max_k * (max_k - 1) * 2;
    int dev = 0, optin = 0;
    MLBP_CUDA(cudaGetDevice(&dev));
    MLBP_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    if (shm + 2048 > (size_t)optin) {
        set_error("gibbs_sample: V = %d needs %zu bytes of shared memory per CTA (%s products), the device has %d", V, shm,
                  f64 ? "fp64" : "fp32", optin);
        return MLBP_ERR_UNSUPPORTED;
    }
    auto kern = f64 ? gibbs_kernel<double> : gibbs_kernel<float>;
    MLBP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)shm));
    kern<<<n_sent * chains, GT, shm, as_stream(stream)>>>(max_k, var_off, pair_off, pair_v0, pair_v1, pair_gap1, sent_id, U,
                                                           (const __half *)planes, plane_stride, ldv, V, E,
                                                           ldexp(1.0, -scale_exp), colsums, chains, burn_in, n_keep,
                                                           (uint32_t)(seed & 0xffffffffu), (uint32_t)(seed >> 32), n_vars, acc,
                                                           samples);
    MLBP_LAUNCH_CHECK();
    return MLBP_OK;
}

extern "C" int mlbp_gibbs_reduce(int n_vars, int chains, int n_keep, const float *acc, int ldv, int V, const int32_t *var_label,
                                 float *marginals, double *label_prob, double *logp_var, int32_t *top1, int32_t *rank,
                                 void *stream) {
    MLBP_CHECK_ARG(acc && var_label && marginals && label_prob && logp_var && top1 && rank, "gibbs_reduce: null pointer");
    MLBP_CHECK_ARG(n_vars >= 0 && V >= 1 && ldv >= V && ldv % 8 == 0, "gibbs_reduce: bad n_vars / V / ldv");
    MLBP_CHECK_ARG(((reinterpret_cast<uintptr_t>(acc) | reinterpret_cast<uintptr_t>(marginals)) % 16) == 0,
                   "gibbs_reduce: acc and marginals need 16-byte aligned rows");
    MLBP_CHECK_ARG(chains >= 1 && n_keep >= 1, "gibbs_reduce: chains and n_keep must be >= 1");
    if (n_vars == 0) return MLBP_OK;
    gibbs_reduce_kernel<<<n_vars, 256, 0, as_stream(stream)>>>(n_vars, chains, n_keep, acc, ldv, V, var_label, marginals,
                                                               label_prob, logp_var, top1, rank);
    MLBP_LAUNCH_CHECK();
    return MLBP_OK;
}
