// K10: max-product factor->variable messages; K11: the log-potential of a whole assignment.
//
// Max-product BP changes one update of sum-product: the pairwise factor->variable message becomes mu(x) = max_y T(x, y) nu(y).
// Tensor cores have no (max, x) semiring, so K10 is a CUDA-core kernel: a 128 x 128 output tile per CTA of 256 threads, 8 x 8
// outputs per thread, k in steps of 32.  Operands sit in shared memory as fp32 PAIRS along k, so one packed multiply (FMUL2)
// forms two products and one three-input max (FMNMX3) folds both into the accumulator: one instruction per multiply-max.
//
// The table entries are formed in the B-tile loader from the fp32 feature planes with K2's compensated argument and exp_f2
// (~1 ulp).  K2's fp16 planes are not read: their hi halves are rounded stochastically, so two equal entries may differ after
// hi + lo, and a max would break such an exact tie differently from float64.
//
// Row normalisation by the max: D = max_k (a_k / amax) T'[n, k] lies within [min T', max T'] (up to the roundings of one
// product and one division), the same 2^(+-half_range_log2) window around 2^-centre_exp as a sum-product D row, so the
// range_log2 bound of K3 and K5 holds unchanged.  Without it a flat message would land log2 V below its table.
//
// A max is exact and order-free: the output is bit-identical for any tiling, slicing or launch order.
#include <vector>

#include "common.cuh"

namespace mlbp {

constexpr int MP_BM = 128, MP_BN = 128, MP_BK = 32, MP_THREADS = 256;

struct MaxprodSmem {
    float2 a[MP_BK / 2][MP_BM];      // a[r, k] as pairs (k, k + 1) along k
    float2 b[MP_BK / 2][MP_BN];      // T'[n, k], same pairing
    __half ah[MP_BM][MP_BK];         // raw tiles, filled by cp.async while the previous tile is multiplied
    __half al[MP_BM][MP_BK];
    float p[MP_BN * MP_BK];          // pmi: [n][k], or [k][n] for the transposed tables
    float w[MP_BN * MP_BK];          // pmi_w1 (T1 / T1T)
    float amax[2][MP_BM];
};

__device__ __forceinline__ void cp_async16(void *smem, const void *gmem, bool pred) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(s), "l"(gmem), "r"(pred ? 16 : 0));
}
__device__ __forceinline__ float max3(float a, float b, float c) {
    float d;
    asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
    return d;
}

// table: MLBP_TABLE_T (B[n][k] = T[n, k]), TT (T[k, n]), T1, T1T; every operand with k >= V is 0 (the padding of A is not
// initialised, and exp of a padded PMI column would be exp(theta_bias))
template <bool TRANS, bool W1>
__global__ void __launch_bounds__(MP_THREADS, 2)
maxprod_kernel(const __half *__restrict__ A_hi, const __half *__restrict__ A_lo, int64_t a_row0, int n_rows,
               const float *__restrict__ pmi, const float *__restrict__ w1, int V, int ldv, int ldf, F2 t_pmi, F2 t_w1,
               F2 t_bias, float *__restrict__ D, int64_t d_row0, int ldd) {
    extern __shared__ __align__(16) unsigned char mp_raw[];
    MaxprodSmem &s = *reinterpret_cast<MaxprodSmem *>(mp_raw);
    const int t = threadIdx.x;
    const int m0 = blockIdx.x * MP_BM, n0 = blockIdx.y * MP_BN;
    const int nk = (V + MP_BK - 1) / MP_BK;

    auto load = [&](int k0) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {                             // A: 128 rows x 32 halves, hi and lo, 16-byte chunks
            const int c = t + MP_THREADS * i, lo = c >> 9, r = (c >> 2) & 127, k = k0 + (c & 3) * 8;
            const bool in = m0 + r < n_rows && k < V;
            const __half *src = (lo ? A_lo : A_hi) + (in ? (a_row0 + m0 + r) * (int64_t)ldv + k : 0);
            cp_async16(lo ? &s.al[r][(c & 3) * 8] : &s.ah[r][(c & 3) * 8], src, in);
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {                             // B: 128 n x 32 k floats per feature plane
            const int c = t + MP_THREADS * i;
            int row, col, off;
            bool in;
            if (TRANS) {                                          // T'[n, k] = T[k, n]: rows k of the plane, 128 n wide
                const int kk = c >> 5;
                row = k0 + kk; col = n0 + (c & 31) * 4; off = kk * MP_BN + (c & 31) * 4;
            } else {                                              // rows n, 32 k wide
                const int nn = c >> 3;
                row = n0 + nn; col = k0 + (c & 7) * 4; off = nn * MP_BK + (c & 7) * 4;
            }
            in = row < V && col < V;                              // ldf % 4 == 0: a chunk that starts below V ends inside the row
            const int64_t g = in ? (int64_t)row * ldf + col : 0;
            cp_async16(&s.p[off], pmi + g, in);
            if (W1) cp_async16(&s.w[off], w1 + g, in);
        }
        asm volatile("cp.async.commit_group;\n" ::);
    };

    // conversion: thread (row / column r = t % 128, half h = t / 128) owns k = 16 h .. 16 h + 15 of the tile
    const int cr = t & 127, ch = t >> 7;
    float amax = 0.f;
    auto convert = [&](int k0) {
        const F2 zero = {0.f, 0.f};
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int k = k0 + 16 * ch + 2 * j;
            const float2 h = __half22float2(*reinterpret_cast<const __half2 *>(&s.ah[cr][16 * ch + 2 * j]));
            const float2 l = __half22float2(*reinterpret_cast<const __half2 *>(&s.al[cr][16 * ch + 2 * j]));
            const float x0 = k < V ? h.x + l.x : 0.f, x1 = k + 1 < V ? h.y + l.y : 0.f;   // exact: 22 bits
            amax = max3(amax, x0, x1);
            s.a[8 * ch + j][cr] = make_float2(x0, x1);
        }
#pragma unroll 2
        for (int j = 0; j < 8; ++j) {
            const int k = k0 + 16 * ch + 2 * j;
            float e[2];
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                const int kl = 16 * ch + 2 * j + q;
                const int o = TRANS ? kl * MP_BN + cr : cr * MP_BK + kl;
                float v = exp_f2(axpb(t_pmi, s.p[o], t_bias));
                if (W1) v *= exp_f2(axpb(t_w1, s.w[o], zero));      // exp(z + th_w1 w) = exp(z) exp(th_w1 w), as K2
                e[q] = (k + q < V && n0 + cr < V) ? v : 0.f;
            }
            s.b[8 * ch + j][cr] = make_float2(e[0], e[1]);
        }
    };

    const int tx = t & 15, ty = t >> 4;                          // outputs: rows 4 ty + {0..3}, 64 + ..; columns 4 tx + {0..3}, 64 + ..
    float acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

    load(0);
    asm volatile("cp.async.wait_group 0;\n" ::: "memory");
    __syncthreads();
    convert(0);
    __syncthreads();
    for (int kt = 0; kt < nk; ++kt) {
        if (kt + 1 < nk) load((kt + 1) * MP_BK);                  // raw buffers are free: the last conversion is behind a barrier
#pragma unroll 1
        for (int kp = 0; kp < MP_BK / 2; ++kp) {
            float2 a[8], b[8];
            const float4 *ap = reinterpret_cast<const float4 *>(&s.a[kp][0]), *bp = reinterpret_cast<const float4 *>(&s.b[kp][0]);
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                const float4 x0 = ap[2 * ty + q], x1 = ap[32 + 2 * ty + q], y0 = bp[2 * tx + q], y1 = bp[32 + 2 * tx + q];
                a[2 * q] = make_float2(x0.x, x0.y); a[2 * q + 1] = make_float2(x0.z, x0.w);
                a[4 + 2 * q] = make_float2(x1.x, x1.y); a[4 + 2 * q + 1] = make_float2(x1.z, x1.w);
                b[2 * q] = make_float2(y0.x, y0.y); b[2 * q + 1] = make_float2(y0.z, y0.w);
                b[4 + 2 * q] = make_float2(y1.x, y1.y); b[4 + 2 * q + 1] = make_float2(y1.z, y1.w);
            }
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float2 p = __fmul2_rn(a[i], b[j]);
                    acc[i][j] = max3(acc[i][j], p.x, p.y);
                }
        }
        if (kt + 1 < nk) {
            asm volatile("cp.async.wait_group 0;\n" ::: "memory");
            __syncthreads();                                      // every thread is done with s.a / s.b and the raw tile is in
            convert((kt + 1) * MP_BK);
            __syncthreads();
        }
    }
    s.amax[ch][cr] = amax;
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int r = (i < 4 ? 4 * ty + i : 64 + 4 * ty + i - 4);
        if (m0 + r >= n_rows) continue;
        const float am = fmaxf(s.amax[0][r], s.amax[1][r]);
        float *out = D + (d_row0 + m0 + r) * (int64_t)ldd;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int n = n0 + (j < 4 ? 4 * tx + j : 64 + 4 * tx + j - 4);
            if (n < V) out[n] = am > 0.f ? __fdiv_rn(acc[i][j], am) : 0.f;   // a zero row: K3 turns it into a uniform message
        }
    }
}

struct ScoreTheta { double ee[3], ed[6]; };

// K11: one warp per sentence; per-lane sums in a fixed order, then a fixed butterfly: deterministic
__global__ void assignment_score_kernel(int n_sent, const int32_t *__restrict__ var_off, const int32_t *__restrict__ x,
                                        const int32_t *__restrict__ var_de, const int32_t *__restrict__ sp_off,
                                        const int32_t *__restrict__ sp_en, const int32_t *__restrict__ sp_feat,
                                        const float *__restrict__ sp_val, const int32_t *__restrict__ giv_off,
                                        const int32_t *__restrict__ giv_label, const int32_t *__restrict__ giv_gap1,
                                        const int32_t *__restrict__ pair_off, const int32_t *__restrict__ pair_v0,
                                        const int32_t *__restrict__ pair_v1, const int32_t *__restrict__ pair_gap1,
                                        const float *__restrict__ pmi, const float *__restrict__ w1, const float *__restrict__ edT,
                                        const float *__restrict__ pedT, int ldf, ScoreTheta th, double *__restrict__ score) {
    const int s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (s >= n_sent) return;
    auto pair_log = [&](int a, int b, int gap1) {                 // log of pot_en_en / pot_en_en_w1 at (a, b), train.py:218-219
        const size_t cell = (size_t)a * ldf + b;
        double l = th.ee[0] * (double)pmi[cell] + th.ee[2];
        if (gap1) l += th.ee[1] * (double)w1[cell];
        return l;
    };
    const int v0 = var_off[s];
    double acc = 0.0;
    for (int v = v0 + lane; v < var_off[s + 1]; v += 32) {
        const int xi = x[v], d = var_de[v];
        double u = 0.0;
        if (d >= 0) {                                             // en_de factor (train.py:240, :251) with its sparse features
            const size_t cell = (size_t)d * ldf + xi;
            u = th.ed[0] * (double)edT[cell] + th.ed[1] * (double)pedT[cell] + th.ed[5];
            for (int q = sp_off[v]; q < sp_off[v + 1]; ++q)
                if (sp_en[q] == xi) u += th.ed[sp_feat[q]] * (double)sp_val[q];
        }
        for (int j = giv_off[v]; j < giv_off[v + 1]; ++j) u += pair_log(xi, giv_label[j], giv_gap1[j]);
        acc += u;
    }
    for (int f = pair_off[s] + lane; f < pair_off[s + 1]; f += 32)
        acc += pair_log(x[v0 + pair_v0[f]], x[v0 + pair_v1[f]], pair_gap1[f]);
    acc = warp_sum(acc);
    if (lane == 0) score[s] = acc;
}

}  // namespace mlbp

using namespace mlbp;

extern "C" int mlbp_factor_to_var_maxprod(const void *A_hi, const void *A_lo, int64_t a_rows_total, int a_row0, int n_rows,
                                          int table, const float *pmi, const float *pmi_w1, int V, int ldv, int ldf,
                                          const double *h_theta_ee, int centre_exp, float *D, int64_t d_row0, int ldd,
                                          void *stream) {
    MLBP_CHECK_ARG(A_hi && A_lo && pmi && pmi_w1 && h_theta_ee && D, "factor_to_var_maxprod: null pointer");
    MLBP_CHECK_ARG(table >= MLBP_TABLE_T && table <= MLBP_TABLE_T1T, "factor_to_var_maxprod: unknown table id %d", table);
    MLBP_CHECK_ARG(V >= 1 && ldv >= V && ldf >= V && ldd >= V, "factor_to_var_maxprod: bad V / ld (%d, %d, %d, %d)", V, ldv, ldf, ldd);
    MLBP_CHECK_ARG(a_row0 >= 0 && n_rows >= 0 && d_row0 >= 0 && (int64_t)a_row0 + n_rows <= a_rows_total,
                   "factor_to_var_maxprod: rows [%d, +%d) outside the %lld A rows", a_row0, n_rows, (long long)a_rows_total);
    MLBP_CHECK_ARG((ldv % 8) == 0 && (ldf % 4) == 0 &&
                   ((reinterpret_cast<uintptr_t>(A_hi) | reinterpret_cast<uintptr_t>(A_lo) | reinterpret_cast<uintptr_t>(pmi) |
                     reinterpret_cast<uintptr_t>(pmi_w1)) % 16) == 0,
                   "factor_to_var_maxprod: operands must be 16-byte aligned rows (ldv %% 8, ldf %% 4)");
    MLBP_CHECK_ARG(centre_exp > -1000 && centre_exp < 1000, "factor_to_var_maxprod: centre_exp out of range");
    for (int i = 0; i < 3; ++i)
        MLBP_CHECK_ARG(h_theta_ee[i] == h_theta_ee[i] && h_theta_ee[i] - h_theta_ee[i] == 0.0, "factor_to_var_maxprod: theta_ee not finite");
    if (n_rows == 0) return MLBP_OK;
    const bool trans = table == MLBP_TABLE_TT || table == MLBP_TABLE_T1T, with_w = table == MLBP_TABLE_T1 || table == MLBP_TABLE_T1T;
    auto kern = trans ? (with_w ? maxprod_kernel<true, true> : maxprod_kernel<true, false>)
                      : (with_w ? maxprod_kernel<false, true> : maxprod_kernel<false, false>);
    const int smem = (int)sizeof(MaxprodSmem);
    static bool attr_set_dev[MLBP_MAX_DEVICES][4] = {};
    const int dev = current_device(), variant = (trans ? 2 : 0) + (with_w ? 1 : 0);
    if (!attr_set_dev[dev][variant]) {
        MLBP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        attr_set_dev[dev][variant] = true;
    }
    // T' = exp(th_pmi pmi [+ th_w1 pmi_w1] + th_bias - centre_exp ln 2): the centring of the sum-product D rows
    const F2 bias = split_double(h_theta_ee[2] - (double)centre_exp * 0.69314718055994530942);
    const dim3 grid((unsigned)((n_rows + MP_BM - 1) / MP_BM), (unsigned)((V + MP_BN - 1) / MP_BN));
    kern<<<grid, MP_THREADS, smem, as_stream(stream)>>>((const __half *)A_hi, (const __half *)A_lo, a_row0, n_rows, pmi, pmi_w1, V,
                                                       ldv, ldf, split_double(h_theta_ee[0]), split_double(h_theta_ee[1]), bias, D,
                                                       d_row0, ldd);
    MLBP_LAUNCH_CHECK();
    return MLBP_OK;
}

extern "C" int mlbp_assignment_score(int n_sent, int n_vars, int n_given, const int32_t *var_off, const int32_t *x,
                                     const int32_t *var_de, const int32_t *sp_off, const int32_t *sp_en, const int32_t *sp_feat,
                                     const float *sp_val, const int32_t *giv_off, const int32_t *giv_label,
                                     const int32_t *giv_gap1, const int32_t *pair_off, const int32_t *pair_v0,
                                     const int32_t *pair_v1, const int32_t *pair_gap1, const float *pmi, const float *pmi_w1,
                                     const float *edT, const float *pedT, int V, int ldf, const double *h_theta_ee,
                                     const double *h_theta_ed, double *score, void *stream) {
    MLBP_CHECK_ARG(n_sent >= 0 && n_vars >= 0 && n_given >= 0, "assignment_score: negative count");
    if (n_sent == 0) return MLBP_OK;
    MLBP_CHECK_ARG(var_off && x && var_de && sp_off && sp_en && sp_feat && sp_val && giv_off && giv_label && giv_gap1 && pair_off &&
                   pair_v0 && pair_v1 && pair_gap1 && pmi && pmi_w1 && edT && pedT && h_theta_ee && h_theta_ed && score,
                   "assignment_score: null pointer");
    MLBP_CHECK_ARG(V >= 1 && ldf >= V, "assignment_score: bad V / ldf (%d, %d)", V, ldf);
    ScoreTheta th;
    for (int i = 0; i < 9; ++i) {
        const double v = i < 3 ? h_theta_ee[i] : h_theta_ed[i - 3];
        MLBP_CHECK_ARG(v == v && v - v == 0.0, "assignment_score: theta not finite");
        (i < 3 ? th.ee[i] : th.ed[i - 3]) = v;
    }
    // every index the kernel gathers a feature cell with must lie in [0, V): checked on the host (this synchronises the stream)
    const cudaStream_t st = as_stream(stream);
    int32_t ends[2] = {0, 0};
    std::vector<int32_t> h((size_t)n_vars + n_given + 1);
    cudaError_t e = cudaMemcpyAsync(&ends[0], var_off + n_sent, sizeof(int32_t), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && n_vars) e = cudaMemcpyAsync(&ends[1], giv_off + n_vars, sizeof(int32_t), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && n_vars) e = cudaMemcpyAsync(h.data(), x, sizeof(int32_t) * n_vars, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && n_given) e = cudaMemcpyAsync(h.data() + n_vars, giv_label, sizeof(int32_t) * n_given, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    int bad = -1;
    for (int i = 0; e == cudaSuccess && i < n_vars + n_given && bad < 0; ++i)
        if (h[i] < 0 || h[i] >= V) bad = i;
    MLBP_CUDA(e);
    MLBP_CHECK_ARG(ends[0] == n_vars && ends[1] == n_given, "assignment_score: var_off / giv_off end at %d / %d, not n_vars %d / n_given %d",
                   ends[0], ends[1], n_vars, n_given);
    MLBP_CHECK_ARG(bad < 0, "assignment_score: %s %d is outside [0, %d)", bad < n_vars ? "assignment of variable" : "given label",
                   bad < n_vars ? bad : bad - n_vars, V);
    const int threads = 128, warps = threads / 32;
    assignment_score_kernel<<<(n_sent + warps - 1) / warps, threads, 0, st>>>(n_sent, var_off, x, var_de, sp_off, sp_en, sp_feat,
                                                                             sp_val, giv_off, giv_label, giv_gap1, pair_off, pair_v0,
                                                                             pair_v1, pair_gap1, pmi, pmi_w1, edT, pedT, ldf, th, score);
    MLBP_LAUNCH_CHECK();
    return MLBP_OK;
}
