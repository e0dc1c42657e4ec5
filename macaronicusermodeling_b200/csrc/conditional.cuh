// The full conditional of one token given words for the other tokens of its sentence, shared by K12 (gibbs.cu: the chain's
// current words) and K13 (pseudo.cu: the learner's guesses):
//     q_i(x) = U_i(x) * prod over the factors touching i, in pair-list order, of (hi + lo) * f
// with one table-plane row per factor read at the neighbour's word and K1's mean-one factor f (include/mlbp.h, K12).
#pragma once
#include "common.cuh"

namespace mlbp {

constexpr int GT = MLBP_GIBBS_THREADS;
constexpr int GW = GT / 32;

__device__ __forceinline__ double to_d(float v) { return (double)v; }
__device__ __forceinline__ double to_d(double v) { return v; }
// one factor of the conditional: q * ((hi + lo) * f), every operation rounded on its own (no contraction)
__device__ __forceinline__ float mul_factor(float q, float t, float f) { return __fmul_rn(q, __fmul_rn(t, f)); }
__device__ __forceinline__ double mul_factor(double q, float t, float f) { return __dmul_rn(q, __dmul_rn((double)t, (double)f)); }

__device__ __forceinline__ void halves8(const __half *p, float *out) {
    const uint4 w = *reinterpret_cast<const uint4 *>(p);
    const __half2 *h = reinterpret_cast<const __half2 *>(&w);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const float2 f = __half22float2(h[j]);
        out[2 * j] = f.x;
        out[2 * j + 1] = f.y;
    }
}

// One thread: per variable of a k-variable sentence, the factors that touch it in pair-list order, as
// nb[nb_off[i] .. nb_off[i + 1]) = neighbour | (1 if the variable is dim 1) << 6 | gap1 << 7.  cursor: k ints of scratch.
// Returns nonzero for a pair list that cannot be read (a variable outside [0, k), a self pair, more than k - 1 factors on a
// variable); nb is then incomplete.
__device__ __forceinline__ int build_neighbours(int k, int p0, int n_p, const int32_t *__restrict__ pair_v0,
                                                const int32_t *__restrict__ pair_v1, const int32_t *__restrict__ pair_gap1,
                                                int *nb_off, int *cursor, uint16_t *nb) {
    int bad = n_p < 0 || 2 * n_p > k * (k - 1);
    for (int i = 0; i <= k; ++i) nb_off[i] = 0;
    for (int p = 0; p < n_p && !bad; ++p) {
        const int a = pair_v0[p0 + p], b = pair_v1[p0 + p];
        if (a < 0 || a >= k || b < 0 || b >= k || a == b) bad = 1;
        else ++nb_off[a + 1], ++nb_off[b + 1];
    }
    for (int i = 0; i < k && !bad; ++i) {
        bad = nb_off[i + 1] > k - 1;
        nb_off[i + 1] += nb_off[i];
        cursor[i] = nb_off[i];                                         // fill cursor
    }
    for (int p = 0; p < n_p && !bad; ++p) {
        const int a = pair_v0[p0 + p], b = pair_v1[p0 + p], g = pair_gap1[p0 + p] ? 1 : 0;
        nb[cursor[a]++] = (uint16_t)(b | (g << 7));
        nb[cursor[b]++] = (uint16_t)(a | (1 << 6) | (g << 7));
    }
    return bad;
}

// The table row of neighbour entry `ent` read at the neighbour's word (words[neighbour]), and its mean-one factor.  dim 0:
// T[x, y] is row y of TT / T1T (planes 2 / 6) with the column sums; dim 1: T[y, x] is row y of T / T1 (planes 0 / 4) with the
// row sums (colsums rows 5 / 6)
__device__ __forceinline__ void factor_row(int ent, const int *words, int64_t ps, int ldv, int V, double unscale,
                                           const double *__restrict__ colsums, int64_t &row_off, float &row_f) {
    const int j = ent & 63, dim1 = (ent >> 6) & 1, g = (ent >> 7) & 1;
    const int y = words[j];
    const int plane = dim1 ? (g ? 4 : 0) : (g ? 6 : 2);
    const int sum = dim1 ? (g ? 6 : 5) : (g ? 1 : 0);
    row_off = (int64_t)plane * ps + (int64_t)y * ldv;
    row_f = (float)(unscale * (double)V / colsums[(size_t)sum * V + y]);
}

// q at the 8 columns e0 .. e0 + 7 (e0 < V; columns from V on hold whatever the padding gives and are masked by the caller):
// U_i's row, then every factor row in order
template <typename Q>
__device__ __forceinline__ void conditional8(Q q[8], const float *urow, int e0, int deg, const __half *__restrict__ planes,
                                             const int64_t *row_off, const float *row_f, int64_t ps) {
    const float4 ua = *reinterpret_cast<const float4 *>(urow + e0);
    const float4 ub = *reinterpret_cast<const float4 *>(urow + e0 + 4);
    q[0] = ua.x; q[1] = ua.y; q[2] = ua.z; q[3] = ua.w;
    q[4] = ub.x; q[5] = ub.y; q[6] = ub.z; q[7] = ub.w;
    int m = 0;
    for (; m + 4 <= deg; m += 4) {                                     // 8 independent 16-byte row loads in flight
        float h[4][8], l[4][8];
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            halves8(planes + row_off[m + r] + e0, h[r]);
            halves8(planes + row_off[m + r] + ps + e0, l[r]);
        }
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const float f = row_f[m + r];
#pragma unroll
            for (int jj = 0; jj < 8; ++jj) q[jj] = mul_factor(q[jj], __fadd_rn(h[r][jj], l[r][jj]), f);
        }
    }
    for (; m < deg; ++m) {
        float h[8], l[8];
        halves8(planes + row_off[m] + e0, h);
        halves8(planes + row_off[m] + ps + e0, l);
        const float f = row_f[m];
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) q[jj] = mul_factor(q[jj], __fadd_rn(h[jj], l[jj]), f);
    }
}

// Block exclusive scan of the threads' float64 sums: Kogge-Stone inside a warp, the warp totals added in warp order.  Returns
// O_w + E_t, the sum of every earlier thread's t_sum in that order (include/mlbp.h, K12).  Holds a block barrier.
__device__ __forceinline__ double scan_base(double t_sum, double *warp_tot, int lane, int warp) {
    double v = t_sum;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const double y = __shfl_up_sync(0xffffffffu, v, d);
        if (lane >= d) v = __dadd_rn(v, y);
    }
    double ex = __shfl_up_sync(0xffffffffu, v, 1);
    if (lane == 0) ex = 0.0;
    if (lane == 31) warp_tot[warp] = v;
    __syncthreads();
    double o = 0.0;
    for (int w = 0; w < warp; ++w) o = __dadd_rn(o, warp_tot[w]);
    return __dadd_rn(o, ex);
}

}  // namespace mlbp
