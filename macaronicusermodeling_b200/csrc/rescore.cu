// K5b: exact re-score of near-tied candidates.
//
// Reference: VariableNode.get_marginal / get_max_vocab (LBP.py:392-411) and FactorGraph.get_precision_counts (LBP.py:80-106)
// take the arg-max and the label's rank of a float64 belief.  The contract is a bit-exact top-1, and no finite-precision
// pipeline can promise that for candidates whose beliefs differ by less than its own error.  K5 (marginals_kernel) therefore
// FLAGS every variable whose two largest products lie within a relative band tau of each other (or whose label has a
// neighbour inside tau_label while its rank can still matter, i.e. at most 50 candidates are certainly above it), and this
// kernel re-evaluates exactly those candidates: for every incoming pairwise message it recomputes the ONE element
//     D_j[e] = sum_k (A_hi + A_lo)[row_j, k] * (B_hi + B_lo)[table_j][e, k]
// from the full 22-bit operands (fp32 products, float64 block reduction: ~1e-8 relative, an order better than the
// three-pass tensor-core row), multiplies the ratios to a reference candidate in float64 and decides arg-max (first index on
// exact ties, np.argmax) and rank from those.  What this buys: message rows may drop the lo half of A (two tensor-core
// passes instead of three, MLBP_GEMM_A_HI_ONLY) -- the rounding of the LAST hop into a belief is the only error of that
// scheme that is not damped by a further contraction (measured: 2.3e-6 relative rms on a belief at V = 10 000 against 1e-7 for
// everything upstream), and the last hop is what this kernel redoes for every decision that error could change.
//
// One CTA walks flagged variables (persistent: the flagged count is only known on the device).
#include "common.cuh"

namespace mlbp {

constexpr int RS_THREADS = 256;
constexpr int RS_MAX_CAND = 64;
constexpr int RS_MAX_IN = 64;      // = marginals_kernel's input capacity

// product of all incoming messages at element e -- the SAME expression, in the same order, as marginals_kernel uses, so
// both kernels see bit-identical values
template <typename T>
__device__ __forceinline__ T belief_product(const float *urow, const float *const *rows, int nn, int e) {
    T p = (T)__ldg(urow + e);
    for (int j = 0; j < nn; ++j)
        if (rows[j]) p *= (T)__ldg(rows[j] + e);
    return p;
}

// 8 fp16 hi + 8 fp16 lo -> 8 floats hi + lo (exact: 22 significant bits)
__device__ __forceinline__ void unpack8(const uint4 h, const uint4 l, float (&x)[8]) {
    const __half2 *hh = reinterpret_cast<const __half2 *>(&h), *ll = reinterpret_cast<const __half2 *>(&l);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float2 a = __half22float2(hh[i]), b = __half22float2(ll[i]);
        x[2 * i] = a.x + b.x;
        x[2 * i + 1] = a.y + b.y;
    }
}

template <typename T>
__global__ void __launch_bounds__(RS_THREADS)
rescore_kernel(const int32_t *__restrict__ flagged, const int32_t *__restrict__ n_flagged,
               const int32_t *__restrict__ flags, const int32_t *__restrict__ grp_u, const int32_t *__restrict__ grp_off,
               const int32_t *__restrict__ in_row, const int32_t *__restrict__ label, const float *__restrict__ U,
               const float *__restrict__ D, int ldv, int V, const __half *__restrict__ A_hi,
               const __half *__restrict__ A_lo, const __half *__restrict__ planes, int64_t plane_stride,
               const int32_t *__restrict__ blocks, int n_blocks, int n_msg_rows, const double *__restrict__ aux,
               const int32_t *__restrict__ cnts, float tau, float tau_label, int32_t *__restrict__ top1,
               int32_t *__restrict__ rank, int32_t *__restrict__ counters) {
    __shared__ double red[32];
    __shared__ const float *s_rows[RS_MAX_IN];
    __shared__ int s_drow[RS_MAX_IN];
    __shared__ int s_table[RS_MAX_IN];
    __shared__ int s_cand[RS_MAX_CAND];
    __shared__ int s_bits[RS_MAX_CAND];
    __shared__ double s_score[RS_MAX_CAND];
    __shared__ double s_dot[RS_MAX_CAND];
    __shared__ int s_nc, s_ref;
    const int total = *n_flagged;
    for (int it = blockIdx.x; it < total; it += gridDim.x) {
        const int g = flagged[it];
        const int flag = flags[g];
        const int i0 = grp_off[g], n = grp_off[g + 1] - i0;
        const int nn = min(n, RS_MAX_IN);
        const float *urow = U + (size_t)grp_u[g] * ldv;
        const int lab = label[g];
        __syncthreads();                                          // shared state of the previous variable is dead
        if (threadIdx.x < RS_MAX_IN) {
            const int r = threadIdx.x < nn ? in_row[i0 + threadIdx.x] : -1;
            s_rows[threadIdx.x] = r >= 0 ? D + (size_t)r * ldv : nullptr;
            s_drow[threadIdx.x] = r;
            int t = -1;                                           // table of a message row: its (level, table) block
            const int a_row = r - MLBP_D_CONST_ROWS;
            if (r >= MLBP_D_CONST_ROWS && a_row < n_msg_rows) {
                int lo = 0, hi = n_blocks - 1;
                while (lo < hi) {                                 // last block with a0 <= a_row
                    const int mid = (lo + hi + 1) >> 1;
                    if (blocks[4 * mid + 1] <= a_row) lo = mid; else hi = mid - 1;
                }
                if (n_blocks > 0 && blocks[4 * lo + 1] <= a_row && a_row < blocks[4 * lo + 1] + blocks[4 * lo + 3]) t = blocks[4 * lo];
            }
            s_table[threadIdx.x] = t;
        }
        if (threadIdx.x == 0) { s_cand[0] = lab; s_bits[0] = 4; s_nc = 1; }
        __syncthreads();
        // ---- candidates: everything inside the band of the best product (bit 1) / of the label's product (bit 2)
        const T best = (T)aux[2 * (size_t)g], plab = (T)aux[2 * (size_t)g + 1];
        const T best_lo = best * (T)(1.0f - tau);
        const T lab_lo = plab * (T)(1.0f - tau_label), lab_hi = plab * (T)(1.0f + tau_label);
        // four elements per thread and iteration, each with its own chain of loads: the products are bit-identical to
        // marginals_kernel's (same factors, same order), the loads of the four chains overlap
        for (int e0 = threadIdx.x; e0 < V; e0 += 4 * RS_THREADS) {
            T p[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) p[u] = e0 + u * RS_THREADS < V ? (T)__ldg(urow + e0 + u * RS_THREADS) : (T)0;
            for (int j = 0; j < nn; ++j) {
                const float *r = s_rows[j];
                if (!r) continue;
#pragma unroll
                for (int u = 0; u < 4; ++u)
                    if (e0 + u * RS_THREADS < V) p[u] *= (T)__ldg(r + e0 + u * RS_THREADS);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int e = e0 + u * RS_THREADS;
                if (e >= V) continue;
                int bits = 0;
                if ((flag & 1) && p[u] >= best_lo) bits |= 1;
                if ((flag & 2) && e != lab && p[u] >= lab_lo && p[u] <= lab_hi) bits |= 2;
                if (bits) {
                    if (e == lab) { atomicOr(&s_bits[0], bits); }
                    else {
                        const int k = atomicAdd(&s_nc, 1);
                        if (k < RS_MAX_CAND) { s_cand[k] = e; s_bits[k] = bits; }
                    }
                }
            }
        }
        __syncthreads();
        const int nc = s_nc;
        if (nc > RS_MAX_CAND) {                                   // an (almost) exact tie of many candidates: keep K5's answer
            if (threadIdx.x == 0) atomicAdd(&counters[1], 1);
            continue;
        }
        // scores are ratios to one reference candidate.  The arg-max does not depend on the label, so with bit 0 the reference
        // is the bit-0 candidate of smallest index (a label whose product is 0 must not stop the arg-max re-score); else the label
        if (threadIdx.x == 0) {
            int k = 0;
            for (int c = 1; c < nc; ++c)
                if ((s_bits[c] & 1) && (!(s_bits[k] & 1) || s_cand[c] < s_cand[k])) k = c;
            s_ref = k;
        }
        __syncthreads();
        const int ref = s_ref;
        if (threadIdx.x < nc) s_score[threadIdx.x] = (double)__ldg(urow + s_cand[threadIdx.x]) / (double)__ldg(urow + s_cand[ref]);
        __syncthreads();
        // ---- exact last hop, one incoming message at a time
        bool bad = false;
        for (int j = 0; j < nn; ++j) {
            const int r = s_drow[j];
            if (r < 0) continue;                                  // still the uniform initial message
            const int t = s_table[j];
            if (t < 0) {                                          // constant-folded row (exact per-theta sums): use it as stored
                if (threadIdx.x < nc) s_dot[threadIdx.x] = (double)__ldg(s_rows[j] + s_cand[threadIdx.x]);
            } else {
                const size_t arow = (size_t)(r - MLBP_D_CONST_ROWS) * ldv;
                const __half *bh = planes + (size_t)(2 * t) * plane_stride, *bl = planes + (size_t)(2 * t + 1) * plane_stride;
                // 16-byte chunks of 8 fp16; rows are padded to ldv (a multiple of 64) so the last chunk may be loaded whole,
                // but the padding of the A rows is never written (uninitialised memory, possibly NaN): it is masked below
                const int n8 = (V + 7) >> 3;
                const uint4 *ah8 = reinterpret_cast<const uint4 *>(A_hi + arow), *al8 = reinterpret_cast<const uint4 *>(A_lo + arow);
                for (int c0 = 0; c0 < nc; c0 += 4) {
                    float acc[4] = {0.f, 0.f, 0.f, 0.f};
                    const uint4 *bh8[4], *bl8[4];
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        const size_t o = (size_t)s_cand[min(c0 + c, nc - 1)] * ldv;
                        bh8[c] = reinterpret_cast<const uint4 *>(bh + o); bl8[c] = reinterpret_cast<const uint4 *>(bl + o);
                    }
                    for (int k8 = threadIdx.x; k8 < n8; k8 += RS_THREADS) {
                        float a[8];
                        unpack8(__ldg(ah8 + k8), __ldg(al8 + k8), a);
                        if (8 * k8 + 8 > V) {
#pragma unroll
                            for (int i = 0; i < 8; ++i)
                                if (8 * k8 + i >= V) a[i] = 0.f;
                        }
#pragma unroll
                        for (int c = 0; c < 4; ++c)
                            if (c0 + c < nc) {                     // block-uniform
                                float b[8];
                                unpack8(__ldg(bh8[c] + k8), __ldg(bl8[c] + k8), b);
                                if (8 * k8 + 8 > V) {
#pragma unroll
                                    for (int i = 0; i < 8; ++i)
                                        if (8 * k8 + i >= V) b[i] = 0.f;
                                }
#pragma unroll
                                for (int i = 0; i < 8; ++i) acc[c] = fmaf(a[i], b[i], acc[c]);
                            }
                    }
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        const double s = block_sum((double)acc[c], red);
                        if (threadIdx.x == 0 && c0 + c < nc) s_dot[c0 + c] = s;
                    }
                }
            }
            __syncthreads();
            const double d0 = s_dot[ref];
            if (!(d0 > 0.0) || !isfinite(d0)) bad = true;          // block-uniform
            if (!bad && threadIdx.x < nc) s_score[threadIdx.x] *= s_dot[threadIdx.x] / d0;
            __syncthreads();
        }
        if (threadIdx.x == 0) {
            bool ok = !bad && (!(flag & 2) || s_score[0] > 0.0);  // a rank needs a positive label product
            for (int c = 0; c < nc; ++c) ok = ok && isfinite(s_score[c]);
            if (!ok) {
                atomicAdd(&counters[2], 1);                        // degenerate products: keep K5's answer
            } else {
                if (flag & 1) {
                    int bi = -1;
                    double bs = -1.0;
                    for (int c = 0; c < nc; ++c)
                        if ((s_bits[c] & 1) && (s_score[c] > bs || (s_score[c] == bs && s_cand[c] < bi))) { bs = s_score[c]; bi = s_cand[c]; }
                    if (bi >= 0) {
                        if (top1[g] != bi) atomicAdd(&counters[3], 1);     // decisions the exact last hop changed
                        top1[g] = bi;
                    }
                }
                if (flag & 2) {
                    int above = 0;
                    for (int c = 1; c < nc; ++c)
                        if ((s_bits[c] & 2) && s_score[c] > s_score[0]) ++above;
                    const int rk = cnts[2 * (size_t)g] - cnts[2 * (size_t)g + 1] + above;
                    if (rank[g] != rk) atomicAdd(&counters[4], 1);
                    rank[g] = rk;
                }
                atomicAdd(&counters[0], 1);
            }
        }
    }
}

}  // namespace mlbp

using namespace mlbp;

extern "C" int mlbp_rescore_candidates(int n_vars, const int32_t *flagged, const int32_t *n_flagged, const int32_t *flags,
                                       const int32_t *grp_u, const int32_t *grp_off, const int32_t *in_row,
                                       const int32_t *label, const float *U, const float *D, int ldv, int V,
                                       const void *A_hi, const void *A_lo, const void *planes, int64_t plane_stride,
                                       const int32_t *msg_blocks, int n_blocks, int n_msg_rows, const double *aux,
                                       const int32_t *cnts, float tau, float tau_label, float range_log2, int32_t *top1,
                                       int32_t *rank, int32_t *counters, void *stream) {
    if (n_vars == 0) return MLBP_OK;
    MLBP_CHECK_ARG(n_vars > 0 && flagged && n_flagged && flags && grp_u && grp_off && in_row && label && U && D && A_hi &&
                   A_lo && planes && aux && cnts && top1 && rank && counters && (msg_blocks || n_blocks == 0),
                   "rescore_candidates: null pointer");
    MLBP_CHECK_ARG(tau >= 0.f && tau < 0.5f && tau_label >= 0.f && tau_label < 0.5f, "rescore_candidates: bad band");
    MLBP_CHECK_ARG((ldv % 64) == 0 && ldv >= V && (plane_stride % 8) == 0 &&
                   ((reinterpret_cast<uintptr_t>(A_hi) | reinterpret_cast<uintptr_t>(A_lo) | reinterpret_cast<uintptr_t>(planes)) % 16) == 0,
                   "rescore_candidates: rows must be 16-byte aligned and padded to a multiple of 64");
    int dev = 0, sms = 0;
    MLBP_CUDA(cudaGetDevice(&dev));
    MLBP_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int grid = n_vars < 8 * sms ? n_vars : 8 * sms;
    if (range_log2 >= 0.f && range_log2 < 100.f)
        rescore_kernel<float><<<grid, RS_THREADS, 0, as_stream(stream)>>>(
            flagged, n_flagged, flags, grp_u, grp_off, in_row, label, U, D, ldv, V, (const __half *)A_hi, (const __half *)A_lo,
            (const __half *)planes, plane_stride, msg_blocks, n_blocks, n_msg_rows, aux, cnts, tau, tau_label, top1, rank, counters);
    else
        rescore_kernel<double><<<grid, RS_THREADS, 0, as_stream(stream)>>>(
            flagged, n_flagged, flags, grp_u, grp_off, in_row, label, U, D, ldv, V, (const __half *)A_hi, (const __half *)A_lo,
            (const __half *)planes, plane_stride, msg_blocks, n_blocks, n_msg_rows, aux, cnts, tau, tau_label, top1, rank, counters);
    MLBP_LAUNCH_CHECK();
    return MLBP_OK;
}
