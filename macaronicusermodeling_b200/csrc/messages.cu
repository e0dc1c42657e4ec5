// K3 (variable -> factor messages) and K5 (marginals / log-posterior / argmax / rank).
//
// Both multiply the messages coming into one variable.  The reference does it one np.multiply per incoming
// message and per OUTGOING edge (LBP.py:377-389, :717-730): O(deg^2) vector passes per variable and sweep.
// Here every needed leave-one-out product of a (variable, schedule level) group comes from a prefix / suffix product
// in registers.  Phase 1 sums every outgoing product (the renormalisation of Message.renormalize, LBP.py:649-657);
// phase 2 recomputes it, scales to 2^14 / sum and splits into the fp16 hi / lo operand rows the pairwise GEMM (K4)
// consumes through TMA.  The sums only have to be deterministic, not exact: a row-uniform factor cancels downstream.
//
// Two kernels:
//   var_to_factor_resident_kernel  (default) a thread-block cluster per group keeps the inputs in shared memory
//                                  (bulk-async copies), exchanges partial sums by st.async pushes: every input is
//                                  read from HBM once.  fp32 products; needs the slices to fit (V = 10k: 8 CTAs).
//   var_to_factor_kernel           one CTA per group, inputs streamed from HBM in both phases; T = float when the
//                                  caller's bound (range_log2) proves that no product can leave the fp32 range, else
//                                  double (the reference multiplies fp64 values of size 1/V and never rescales,
//                                  LBP.py:381-385).  Measured on B200 the fp64 pipe issues only ~3 lanes/clk/SM
//                                  (profiles/README.md): the double variant is compute-bound at ~16 % of HBM bandwidth;
//                                  it is the always-safe fallback.
#include <stdlib.h>

#include <cooperative_groups.h>
#include <cuda/std/type_traits>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace mlbp {

constexpr int K3_THREADS = 256;
constexpr int K3_WARPS = K3_THREADS / 32;
constexpr int K3R_THREADS = 256;                  // resident kernel (224 = three balanced passes over 640 column pairs: measured no faster)
constexpr int K3R_WARPS = K3R_THREADS / 32;
constexpr int K3_RESIDENT_SMEM = 100 * 1024;     // per CTA: two CTAs per SM keep loads and stores overlapped

__global__ void fill_uniform_rows_kernel(__half *__restrict__ A_hi, __half *__restrict__ A_lo, int ldv, int V,
                                         const int32_t *__restrict__ rows, const uint8_t *__restrict__ keep) {
    const size_t r = (size_t)rows[blockIdx.x];
    __half hi, lo;
    split_f16(ldexpf(1.0f, MLBP_A_SCALE_LOG2) / (float)V, hi, lo);
    const __half z = __float2half_rn(0.f);
    for (int e = threadIdx.x; e < ldv; e += blockDim.x) {
        const bool on = e < V && (!keep || keep[e]);
        A_hi[r * ldv + e] = on ? hi : z;
        A_lo[r * ldv + e] = on ? lo : z;
    }
}

// One output element of a leave-one-out product -> fp16 hi/lo rows of every GEMM block that reads this message.
// `first` = element offset of the first destination row (the common case: exactly one reader); further readers are
// walked by a rolled loop so that the unrolled per-input code around it stays small (instruction-cache resident).
__device__ __forceinline__ void k3_store(float x, size_t first, int nd, const int32_t *__restrict__ dest, int d0, int ldv,
                                         int col, __half *__restrict__ A_hi, __half *__restrict__ A_lo) {
    __half hi, lo;
    split_f16(x, hi, lo);
    A_hi[first] = hi;
    A_lo[first] = lo;
    if (nd > 1) {
#pragma unroll 1
        for (int t = 1; t < nd; ++t) {
            const size_t o = (size_t)dest[d0 + t] * ldv + col;
            A_hi[o] = hi;
            A_lo[o] = lo;
        }
    }
}

template <int NMAX, typename T, int OCC>
__global__ void __launch_bounds__(K3_THREADS, OCC)
var_to_factor_kernel(const int32_t *__restrict__ grp_u, const int32_t *__restrict__ grp_off,
                     const int32_t *__restrict__ in_row, const int32_t *__restrict__ dest_off,
                     const int32_t *__restrict__ dest, const int32_t *__restrict__ first_dest,
                     const int32_t *__restrict__ second_dest, const float *__restrict__ U, const float *__restrict__ D, int ldv, int V,
                     __half *__restrict__ A_hi, __half *__restrict__ A_lo) {
    __shared__ const float *s_src[NMAX];
    __shared__ int s_d0[NMAX], s_nd[NMAX];
    __shared__ size_t s_first[NMAX];
    __shared__ double s_warp[K3_WARPS][NMAX];
    // the normaliser in T: in fp64 the sums reach far outside the fp32 range (2^14 / t is 0 above t = 2^163, inf below
    // t = 2^-114), and a float scale would turn those messages uniform or infinite
    __shared__ T s_scale[NMAX];
    const int g = blockIdx.x;
    const int i0 = grp_off[g], n = grp_off[g + 1] - i0;
    const float *urow = U + (size_t)grp_u[g] * ldv;
    if (threadIdx.x < NMAX) {
        const int j = threadIdx.x;
        // a message still at its uniform initial value, and the unused slots up to NMAX, read the constant-one row
        // D[0] (messages are scale-free): every load below is unconditional
        const int r = j < n ? in_row[i0 + j] : -1;
        s_src[j] = D + (size_t)(r >= 0 ? r : 0) * ldv;
        const int d0 = j < n ? dest_off[i0 + j] : 0, d1 = j < n ? dest_off[i0 + j + 1] : 0;
        s_d0[j] = d0;
        s_nd[j] = d1 - d0;
        s_first[j] = d1 > d0 ? (size_t)first_dest[i0 + j] * ldv : 0;
    }
    __syncthreads();

    // ---- phase 1: sums of the leave-one-out products
    T acc[NMAX];
#pragma unroll
    for (int j = 0; j < NMAX; ++j) acc[j] = (T)0;
    for (int e = threadIdx.x; e < V; e += K3_THREADS) {
        float d[NMAX];
#pragma unroll
        for (int j = 0; j < NMAX; ++j) d[j] = __ldg(s_src[j] + e);
        T pre[NMAX];
        T p = (T)__ldg(urow + e);
#pragma unroll
        for (int j = 0; j < NMAX; ++j) { pre[j] = p; p *= (T)d[j]; }
        T suf = (T)1;
#pragma unroll
        for (int j = NMAX - 1; j >= 0; --j) {
            acc[j] += pre[j] * suf;
            suf *= (T)d[j];
        }
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int j = 0; j < NMAX; ++j) {
        const double w = warp_sum((double)acc[j]);
        if (lane == 0) s_warp[warp][j] = w;
    }
    __syncthreads();
    if (threadIdx.x < NMAX) {
        double t = 0.0;
#pragma unroll
        for (int w = 0; w < K3_WARPS; ++w) t += s_warp[w][threadIdx.x];
        // sum <= 0 or non-finite -> uniform (Message.renormalize, LBP.py:650-657); flagged by a negative scale
        s_scale[threadIdx.x] = (t > 0.0 && isfinite(t)) ? (T)(ldexp(1.0, MLBP_A_SCALE_LOG2) / t) : (T)-1;
    }
    __syncthreads();

    // ---- phase 2: recompute, normalise, split, scatter to the consuming GEMM blocks
    // (walking the columns backwards to catch the L2-resident tail of phase 1 was measured 12 % slower)
    const float uni = ldexpf(1.0f, MLBP_A_SCALE_LOG2) / (float)V;
    for (int e = threadIdx.x; e < V; e += K3_THREADS) {
        float d[NMAX];
#pragma unroll
        for (int j = 0; j < NMAX; ++j) d[j] = __ldg(s_src[j] + e);
        T pre[NMAX];
        T p = (T)__ldg(urow + e);
#pragma unroll
        for (int j = 0; j < NMAX; ++j) { pre[j] = p; p *= (T)d[j]; }
        T suf = (T)1;
#pragma unroll
        for (int j = NMAX - 1; j >= 0; --j) {
            const int nd = s_nd[j];                               // 0 beyond n and for messages nobody reads
            if (nd > 0) {
                const T sc = s_scale[j];
                const float x = sc > (T)0 ? (float)(pre[j] * suf * sc) : uni;
                k3_store(x, s_first[j] + e, nd, dest, s_d0[j], ldv, e, A_hi, A_lo);
            }
            suf *= (T)d[j];
        }
    }
}

// Messages with more than TWO readers (the first two are written directly): the slice just written to the first reader's
// row is copied into the third and further readers' rows (L1/L2 hits).  The caller puts a __syncthreads() between the
// writes and this copy.
template <int NIN>
__device__ __forceinline__ void k3_copy_extras(const int *__restrict__ s_nd, const int *__restrict__ s_d0,
                                               const size_t *__restrict__ s_first, const int32_t *__restrict__ dest,
                                               int ldv, int col0, int ncol, __half *A_hi, __half *A_lo) {
#pragma unroll 1
    for (int j = 0; j < NIN; ++j) {
        const int nd = s_nd[j];
#pragma unroll 1
        for (int t = 2; t < nd; ++t) {
            const size_t src = s_first[j], dst = (size_t)dest[s_d0[j] + t] * ldv + col0;
            for (int e = threadIdx.x; e < ncol; e += K3_THREADS) {
                A_hi[dst + e] = A_hi[src + e];
                A_lo[dst + e] = A_lo[src + e];
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------------------------
// K3, single-read variant.  The leave-one-out sums need every input element before the first output element can be
// scaled, so a streaming kernel reads its inputs twice.  Here a thread-block CLUSTER owns one (variable, level) group:
// CTA q of C keeps the column slice [q*S, (q+1)*S) of all NIN+1 input rows in shared memory (bulk-async copies,
// cp.async.bulk + one mbarrier: the whole slice is in flight at once), phase 1 sums from shared memory, the C partial
// sums per output are exchanged through distributed shared memory in fixed rank order (deterministic), and phase 2
// re-reads shared memory, not HBM.  DRAM traffic = each input once + each output once.  The grid is persistent
// (resident clusters walk over the groups); the index records of the next group are fetched while the copies of
// the current one are in flight.  NIN is the exact row count the shared-memory slices are sized for.
__device__ __forceinline__ uint32_t k3_smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

template <int NIN>
__global__ void __launch_bounds__(K3R_THREADS, 2)
var_to_factor_resident_kernel(int n_groups, const int32_t *__restrict__ grp_u, const int32_t *__restrict__ grp_off,
                              const int32_t *__restrict__ in_row, const int32_t *__restrict__ dest_off,
                              const int32_t *__restrict__ dest, const int32_t *__restrict__ first_dest,
                              const int32_t *__restrict__ second_dest, const float *__restrict__ U, const float *__restrict__ D, int ldv, int V, int S,
                              __half *__restrict__ A_hi, __half *__restrict__ A_lo, long long *dbg) {
#ifdef MLBP_K3_STAGE_TIMES                                      // scripts/k3_probe.py: cycles per stage, per CTA
    long long tacc[6] = {0, 0, 0, 0, 0, 0}, tprev = clock64();
#define K3_TICK(i) do { const long long tn_ = clock64(); tacc[i] += tn_ - tprev; tprev = tn_; } while (0)
#else
#define K3_TICK(i) do { } while (0)
#endif
    extern __shared__ __align__(128) float s_rows[];          // [1 + NIN][S]: row 0 = U slice, row 1 + j = input j
    __shared__ __align__(8) unsigned long long s_bar;
    __shared__ const float *s_src[2][NIN + 1];                // [buffer][0] = U row, [1 + j] = input j (nullptr: ones)
    __shared__ int s_d0[2][NIN], s_nd[2][NIN];
    __shared__ size_t s_first[2][NIN], s_second[2][NIN];
    __shared__ double s_warp[K3R_WARPS][NIN];
    __shared__ double s_gather[2][8][NIN];                     // [exchange parity][source rank][output]
    __shared__ __align__(8) unsigned long long s_gbar[2];
    __shared__ float s_scale[NIN];
    cg::cluster_group cl = cg::this_cluster();
    const unsigned C = cl.num_blocks(), q = cl.block_rank();
    const int n_clusters = gridDim.x / C;
    const int col0 = (int)q * S;
    const int ncol = max(0, min(S, V - col0));                 // columns this CTA owns (S is a multiple of 4)
    const uint32_t bytes = (uint32_t)((ncol + 3) & ~3) * 4u;   // rows are padded to ld >= roundup(V, 64): in bounds
    const uint32_t bar = k3_smem_u32(&s_bar);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const float uni = ldexpf(1.0f, MLBP_A_SCALE_LOG2) / (float)V;

    // Index records of a group -> shared-memory buffer b (threads 0..NIN; thread 0 also owns the U row).  The chain
    // grp_off -> in_row / dest_off / first_dest is software-pipelined: (i0, n, u) of a group are loaded one iteration
    // before they are needed, so only ONE dependent load level is left, and it overlaps the bulk copies in flight.
    int nx_i0 = 0, nx_n = 0, nx_u = 0;
    auto fetch_head = [&](int g) {
        if (threadIdx.x <= NIN && g < n_groups) {
            nx_i0 = grp_off[g];
            nx_n = grp_off[g + 1] - nx_i0;
            nx_u = grp_u[g];
        }
    };
    auto fetch_body = [&](int b) {
        if (threadIdx.x <= NIN) {
            const int i0 = nx_i0, n = nx_n;
            if (threadIdx.x == 0) {
                s_src[b][0] = U + (size_t)nx_u * ldv + col0;
            } else {
                const int j = threadIdx.x - 1;
                const int r = j < n ? in_row[i0 + j] : -1;
                // a message still uniform, and the unused slots, copy the constant-one row D[0] (scale-free): every
                // group moves the same number of bytes and phase 1 / 2 need no special cases
                s_src[b][1 + j] = D + (size_t)(r >= 0 ? r : 0) * ldv + col0;
                const int d0 = j < n ? dest_off[i0 + j] : 0, d1 = j < n ? dest_off[i0 + j + 1] : 0;
                const int f = j < n ? first_dest[i0 + j] : -1, f2 = j < n ? second_dest[i0 + j] : -1;
                s_d0[b][j] = d0;
                s_nd[b][j] = d1 - d0;
                s_first[b][j] = f >= 0 ? (size_t)f * ldv + col0 : 0;
                s_second[b][j] = f2 >= 0 ? (size_t)f2 * ldv + col0 : 0;
            }
        }
    };

    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(1) : "memory");
        for (int k = 0; k < 2; ++k) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(k3_smem_u32(&s_gbar[k])), "r"(1) : "memory");
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;"
                         ::"r"(k3_smem_u32(&s_gbar[k])), "r"((uint32_t)(NIN * C * sizeof(double))) : "memory");
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    cl.sync();                                                     // once: every peer's barriers exist before the first push
    int it = 0;
    int g = blockIdx.x / C, b = 0;
    fetch_head(g);
    if (g < n_groups) fetch_body(0);
    fetch_head(g + n_clusters);
    __syncthreads();
    uint32_t parity = 0;
    // Two adjacent columns per thread: 8-byte shared-memory loads, packed fp32x2 multiplies (FMUL2 on sm_100), fp16x2
    // conversions and 4-byte stores.  With 100 KB of shared memory per CTA only 16 warps are resident per SM, so the
    // loops are written as straight-line code (no branch on a value loaded inside the loop): measured with clock64
    // per stage, a data-dependent branch per input cost ~100 cycles per input and column pair.
    const int npair = (ncol + 1) >> 1;
    for (; g < n_groups; g += n_clusters, b ^= 1) {
        if (ncol > 0) {
            if (threadIdx.x == 0)
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes * (NIN + 1)) : "memory");
            if (threadIdx.x <= NIN) {
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // earlier generic reads before the async writes
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                             ::"r"(k3_smem_u32(s_rows + (size_t)threadIdx.x * S)), "l"(s_src[b][threadIdx.x]), "r"(bytes), "r"(bar) : "memory");
            }
        }
        K3_TICK(0);
        if (g + n_clusters < n_groups) fetch_body(b ^ 1);                     // overlaps the copies in flight
        fetch_head(g + 2 * n_clusters);
        K3_TICK(1);
        if (ncol > 0) {
            uint32_t ok = 0;
            const unsigned long long t0 = clock64();
            while (!ok) {
                asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                             : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
                if (!ok && clock64() - t0 > 4000000000ull) __trap();   // a lost copy traps (launch error) instead of hanging the GPU
            }
            parity ^= 1u;
            if (ncol & 1) {                                        // odd V, last slice: the pair partner of the final column
                if (threadIdx.x <= NIN) s_rows[(size_t)threadIdx.x * S + ncol] = 1.0f;   // is row padding -> make it finite
                __syncthreads();
            }
        }
        K3_TICK(2);

        // ---- phase 1: partial sums of the leave-one-out products over this CTA's columns
        float acc[NIN];
#pragma unroll
        for (int j = 0; j < NIN; ++j) acc[j] = 0.f;
        for (int e2 = threadIdx.x; e2 < npair; e2 += K3R_THREADS) {
            const float2 *col = reinterpret_cast<const float2 *>(s_rows) + e2;
            const bool odd = 2 * e2 + 1 >= ncol;                  // the second column is padding
            float2 d[NIN];
#pragma unroll
            for (int j = 0; j < NIN; ++j) d[j] = col[(1 + j) * (S >> 1)];
            float2 pre[NIN];
            float2 p = col[0];
#pragma unroll
            for (int j = 0; j < NIN; ++j) { pre[j] = p; p = __fmul2_rn(p, d[j]); }
            float2 suf = make_float2(1.f, odd ? 0.f : 1.f);         // zero kills the padding column's contribution
#pragma unroll
            for (int j = NIN - 1; j >= 0; --j) {
                acc[j] = fmaf(pre[j].x, suf.x, acc[j]);
                acc[j] = fmaf(pre[j].y, suf.y, acc[j]);
                suf = __fmul2_rn(suf, d[j]);
            }
        }
#pragma unroll
        for (int j = 0; j < NIN; ++j) {
            const float w = warp_sum_f32(acc[j]);                  // fp32: the fp64 pipe is ~3 lanes/clk/SM, and the
            if (lane == 0) s_warp[warp][j] = (double)w;            // scale only has to be deterministic, not exact
        }
        __syncthreads();
        K3_TICK(3);
        // Exchange of the partial sums: every CTA PUSHES its NIN partial sums into each peer's gather buffer with
        // st.async, which completes on the PEER's mbarrier; a CTA only waits on its own barrier.  No cluster barrier in
        // the loop: barrier.cluster.arrive.release made every iteration wait for the previous phase-2 stores to drain
        // (7 % membar + 6 % cluster-barrier stalls in the ncu source view).  Buffers alternate by iteration parity; a
        // CTA can run at most one exchange ahead of a peer, because finishing exchange i needs the peer's sums of i.
        {
            const int par = it & 1;
            for (int i = threadIdx.x; i < NIN * (int)C; i += K3R_THREADS) {
                const int r = i / NIN, j = i - r * NIN;
                double t = 0.0;
#pragma unroll
                for (int w = 0; w < K3R_WARPS; ++w) t += s_warp[w][j];
                const uint32_t dst = k3_smem_u32(&s_gather[par][q][j]), rb = k3_smem_u32(&s_gbar[par]);
                asm volatile(
                    "{\n\t.reg .b32 ra, rm;\n\t"
                    "mapa.shared::cluster.u32 ra, %0, %2;\n\t"
                    "mapa.shared::cluster.u32 rm, %1, %2;\n\t"
                    "st.async.shared::cluster.mbarrier::complete_tx::bytes.b64 [ra], %3, [rm];\n\t}"
                    ::"r"(dst), "r"(rb), "r"(r), "l"(__double_as_longlong(t)) : "memory");
            }
            const uint32_t gb = k3_smem_u32(&s_gbar[par]), gpar = (uint32_t)(it >> 1) & 1u;
            uint32_t ok = 0;
            const unsigned long long t0 = clock64();
            while (!ok) {
                asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                             : "=r"(ok) : "r"(gb), "r"(gpar) : "memory");
                if (!ok && clock64() - t0 > 4000000000ull) __trap();
            }
            if (threadIdx.x < NIN) {
                double t = 0.0;
                for (unsigned r = 0; r < C; ++r) t += s_gather[par][r][threadIdx.x];     // fixed order: deterministic
                // sum <= 0 or non-finite -> uniform (Message.renormalize, LBP.py:650-657): flagged by a negative scale
                s_scale[threadIdx.x] = (t > 0.0 && isfinite(t)) ? (float)(ldexp(1.0, MLBP_A_SCALE_LOG2) / t) : -1.0f;
            }
        }
        __syncthreads();
        if (threadIdx.x == 0)                                      // re-arm this parity's barrier for exchange it + 2
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;"
                         ::"r"(k3_smem_u32(&s_gbar[it & 1])), "r"((uint32_t)(NIN * C * sizeof(double))) : "memory");
        ++it;
        K3_TICK(4);

        // ---- phase 2: recompute from shared memory, normalise, split, scatter to the consuming GEMM blocks
        unsigned omask = 0, multi = 0, many = 0;                   // bit j: message j has >= 1 / >= 2 / >= 3 readers
#pragma unroll
        for (int j = 0; j < NIN; ++j) {
            const int nd = s_nd[b][j];
            omask |= (nd > 0 ? 1u : 0u) << j;
            multi |= (nd > 1 ? 1u : 0u) << j;
            many |= (nd > 2 ? 1u : 0u) << j;
        }
        // two instantiations of the loop: levels whose messages all have one reader (most) do not carry the code and
        // registers of the second store
        auto phase2 = [&](auto second_tag) {
            constexpr bool SECOND = decltype(second_tag)::value;
            for (int e2 = threadIdx.x; e2 < npair; e2 += K3R_THREADS) {
                const float2 *col = reinterpret_cast<const float2 *>(s_rows) + e2;
                const bool odd = 2 * e2 + 1 >= ncol;
                float2 d[NIN];
    #pragma unroll
                for (int j = 0; j < NIN; ++j) d[j] = col[(1 + j) * (S >> 1)];
                float2 pre[NIN];
                float2 p = col[0];
    #pragma unroll
                for (int j = 0; j < NIN; ++j) { pre[j] = p; p = __fmul2_rn(p, d[j]); }
                float2 suf = make_float2(1.f, 1.f);
                // one output: scale, split into fp16 hi / lo pairs, store to the first reader's row
                auto emit = [&](int j, float2 sufj) {
                    const float sc = s_scale[j];
                    float2 x = __fmul2_rn(__fmul2_rn(pre[j], sufj), make_float2(sc, sc));
                    if (!(sc > 0.f)) x = make_float2(uni, uni);
                    const __half2 hi = __float22half2_rn(x);
                    const float2 back = __half22float2(hi);
                    const __half2 lo = __float22half2_rn(__fadd2_rn(x, make_float2(-back.x, -back.y)));
                    const size_t o = s_first[b][j] + 2 * (size_t)e2;              // even: 4-byte aligned
                    if (!odd) {
                        *reinterpret_cast<__half2 *>(A_hi + o) = hi;
                        *reinterpret_cast<__half2 *>(A_lo + o) = lo;
                    } else {
                        A_hi[o] = __low2half(hi);
                        A_lo[o] = __low2half(lo);
                    }
                    if (SECOND && ((multi >> j) & 1u)) {                // second reader (final versions: message GEMM + gradient stage)
                        const size_t o2 = s_second[b][j] + 2 * (size_t)e2;
                        if (!odd) {
                            *reinterpret_cast<__half2 *>(A_hi + o2) = hi;
                            *reinterpret_cast<__half2 *>(A_lo + o2) = lo;
                        } else {
                            A_hi[o2] = __low2half(hi);
                            A_lo[o2] = __low2half(lo);
                        }
                    }
                };
                // Outputs are walked four at a time: when all four have a reader (the common case) their chains are emitted
                // as ONE straight-line block, so the four dependent load -> multiply -> convert -> store chains overlap
                // instead of each paying its latency behind a branch (only 16 warps per SM are resident to hide it).
    #pragma unroll
                for (int j0 = NIN - 1; j0 >= 0; j0 -= 4) {
                    if (j0 >= 3 && ((omask >> (j0 - 3)) & 0xFu) == 0xFu) {
                        const float2 s0 = suf, s1 = __fmul2_rn(s0, d[j0]), s2 = __fmul2_rn(s1, d[j0 - 1]),
                                     s3 = __fmul2_rn(s2, d[j0 - 2]);
                        emit(j0, s0); emit(j0 - 1, s1); emit(j0 - 2, s2); emit(j0 - 3, s3);
                        suf = __fmul2_rn(s3, d[j0 - 3]);
                    } else {
    #pragma unroll
                        for (int j = j0; j > j0 - 4 && j >= 0; --j) {
                            if ((omask >> j) & 1u) emit(j, suf);           // register test: no load feeds this branch
                            suf = __fmul2_rn(suf, d[j]);
                        }
                    }
                }
            }
        };
        if (multi) phase2(cuda::std::true_type{}); else phase2(cuda::std::false_type{});
        if (many) {                                                // block-uniform, rare: third and further readers
            __syncthreads();                                       // the copy below reads elements other threads wrote
            k3_copy_extras<NIN>(s_nd[b], s_d0[b], s_first[b], dest, ldv, col0, ncol, A_hi, A_lo);
        }
        __syncthreads();                                           // shared memory is reused by the next group
        K3_TICK(5);
    }
#ifdef MLBP_K3_STAGE_TIMES
    if (dbg && threadIdx.x == 0)
        for (int i = 0; i < 6; ++i) dbg[(size_t)blockIdx.x * 6 + i] = tacc[i];
#endif
    // A CTA leaves its last exchange only after every peer's sums for it have ARRIVED here, and nothing is ever read from
    // a peer, so no CTA can exit while another still needs its shared memory.
}

// Top-K masking of message rows: the reference's approximate paths (use_approx_inference / use_approx_beliefs,
// LBP.py:506-507, :515-516, :554-563) contract only the K = 100 largest entries of a message
// (au.sparse_vec_mat_dot pyx:193-205, au.sparse_dot pyx:117-129).  Zeroing every other entry of the operand row and
// running the same dense GEMM gives the same sums.  One CTA per row: 4-pass radix select (8 bits per pass) on the bit
// patterns of hi + lo (non-negative floats order like their bits), then one masking pass; ties at the threshold are
// kept in arbitrary order up to K, like np.argpartition.
__global__ void __launch_bounds__(256)
topk_mask_rows_kernel(__half *__restrict__ A_hi, __half *__restrict__ A_lo, int ldv, int V, int64_t row0, int K) {
    __shared__ unsigned hist[256];
    __shared__ unsigned s_prefix, s_need, s_taken;
    __half *hi = A_hi + (size_t)(row0 + blockIdx.x) * ldv, *lo = A_lo + (size_t)(row0 + blockIdx.x) * ldv;
    auto bits_of = [&](int e) { return __float_as_uint(__half2float(hi[e]) + __half2float(lo[e])); };
    if (threadIdx.x == 0) { s_prefix = 0u; s_need = (unsigned)K; s_taken = 0u; }
    for (int shift = 24; shift >= 0; shift -= 8) {
        hist[threadIdx.x] = 0u;
        __syncthreads();
        const unsigned prefix = s_prefix;
        for (int e = threadIdx.x; e < V; e += 256) {
            const unsigned b = bits_of(e);
            if (shift == 24 || (b >> (shift + 8)) == (prefix >> (shift + 8))) atomicAdd(&hist[(b >> shift) & 255u], 1u);
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            unsigned cum = 0, need = s_need;
            for (int b = 255; b >= 0; --b) {
                if (cum + hist[b] >= need) { s_need = need - cum; s_prefix = prefix | ((unsigned)b << shift); break; }
                cum += hist[b];
            }
        }
        __syncthreads();
    }
    const unsigned thr = s_prefix, need = s_need;     // K-th largest bit pattern; keep `need` of the entries equal to it
    const __half z = __float2half_rn(0.f);
    for (int e = threadIdx.x; e < V; e += 256) {
        const unsigned b = bits_of(e);
        bool keep = b > thr;
        if (b == thr) keep = atomicAdd(&s_taken, 1u) < need;
        if (!keep) { hi[e] = z; lo[e] = z; }
    }
}

// one CTA per variable: total product of all incoming messages (T = float under the same range bound as K3).
// Optional near-tie detection (flags != nullptr; see rescore.cu): besides the arg-max and the label's rank the kernel keeps
// the SECOND largest product and counts the candidates inside a relative band around the label's product; variables whose
// decisions an error of relative size << tau could change are appended to `flagged` for the exact re-score.
template <typename T, bool VEC>
__global__ void __launch_bounds__(256)
marginals_kernel(const int32_t *__restrict__ grp_u, const int32_t *__restrict__ grp_off,
                 const int32_t *__restrict__ in_row, const int32_t *__restrict__ label, const float *__restrict__ U,
                 const float *__restrict__ D, int ldv, int V, double *__restrict__ logp, int32_t *__restrict__ top1,
                 int32_t *__restrict__ rank, float *__restrict__ beliefs, float tau, float tau_label,
                 double *__restrict__ aux, int32_t *__restrict__ cnts, int32_t *__restrict__ flags,
                 int32_t *__restrict__ flagged, int32_t *__restrict__ n_flagged) {
    __shared__ double red[32];
    __shared__ T s_best[8], s_second[8];
    __shared__ int s_besti[8];
    const int g = blockIdx.x;
    const int i0 = grp_off[g], n = grp_off[g + 1] - i0;
    const float *urow = U + (size_t)grp_u[g] * ldv;
    const int lab = label[g];
    __shared__ const float *s_rows[64];
    __shared__ int s_nn;
    const int n64 = min(n, 64);                                   // the host entry point rejects n > 64
    if (threadIdx.x == 0) {                                       // messages still uniform (row < 0) drop out: order is kept
        int c = 0;
        for (int j = 0; j < n64; ++j) {
            const int r = in_row[i0 + j];
            if (r >= 0) s_rows[c++] = D + (size_t)r * ldv;
        }
        s_nn = c;
    }
    __syncthreads();
    const int nn = s_nn;
    auto prod = [&](int e) {                                      // rescore.cu evaluates the same expression in the same order
        T p = (T)__ldg(urow + e);
        for (int j = 0; j < nn; ++j) p *= (T)__ldg(s_rows[j] + e);
        return p;
    };
    // four adjacent columns per thread: 16-byte loads, the loads of four rows issued before their multiplies (the products
    // are formed in the same left-to-right order as prod(), so every value is bit-identical to the scalar expression)
    auto prod4 = [&](int e, T p[4]) {
        const float4 u = __ldg(reinterpret_cast<const float4 *>(urow + e));
        p[0] = (T)u.x; p[1] = (T)u.y; p[2] = (T)u.z; p[3] = (T)u.w;
        int j = 0;
        for (; j + 4 <= nn; j += 4) {
            float4 d[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) d[q] = __ldg(reinterpret_cast<const float4 *>(s_rows[j + q] + e));
#pragma unroll
            for (int q = 0; q < 4; ++q) { p[0] *= (T)d[q].x; p[1] *= (T)d[q].y; p[2] *= (T)d[q].z; p[3] *= (T)d[q].w; }
        }
        for (; j < nn; ++j) {
            const float4 d = __ldg(reinterpret_cast<const float4 *>(s_rows[j] + e));
            p[0] *= (T)d.x; p[1] *= (T)d.y; p[2] *= (T)d.z; p[3] *= (T)d.w;
        }
    };
    const T plab = prod(lab);
    const T lab_lo = plab * (T)(1.0f - tau_label), lab_hi = plab * (T)(1.0f + tau_label);
    T sp = (T)0, best = (T)-1, second = (T)-1;
    int besti = 0x7fffffff, cnt = 0, near_hi = 0, near_lo = 0;
    auto visit = [&](int e, T p) {
        sp += p;
        cnt += (p > plab) ? 1 : 0;
        near_hi += (p > plab && p <= lab_hi) ? 1 : 0;
        near_lo += (e != lab && p <= plab && p >= lab_lo) ? 1 : 0;
        if (p > best) { second = best; best = p; besti = e; }     // ascending e inside a thread: first index wins per thread
        else if (p > second) second = p;
    };
    if (VEC) {
        for (int e = 4 * threadIdx.x; e < V; e += 4 * blockDim.x) {   // rows are padded to a multiple of 4: loads stay inside
            T p[4];
            prod4(e, p);
#pragma unroll
            for (int q = 0; q < 4; ++q)
                if (e + q < V) visit(e + q, p[q]);
        }
    } else {
        for (int e = threadIdx.x; e < V; e += blockDim.x) visit(e, prod(e));
    }
    double s = block_sum((double)sp, red);
    const double c = block_sum((double)cnt, red);
    const double nh = block_sum((double)near_hi, red), nl = block_sum((double)near_lo, red);
    // argmax with first-index tie break (np.argmax); the runner-up value rides along
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const T ob = __shfl_xor_sync(0xffffffffu, best, o), os = __shfl_xor_sync(0xffffffffu, second, o);
        const int oi = __shfl_xor_sync(0xffffffffu, besti, o);
        const T lose = ob < best ? ob : best;                     // the smaller of the two bests is a runner-up candidate
        second = second > os ? second : os;
        second = second > lose ? second : lose;
        if (ob > best || (ob == best && oi < besti)) { best = ob; besti = oi; }
    }
    __syncthreads();
    if ((threadIdx.x & 31) == 0) { s_best[threadIdx.x >> 5] = best; s_besti[threadIdx.x >> 5] = besti; s_second[threadIdx.x >> 5] = second; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w) {
            const T lose = s_best[w] < best ? s_best[w] : best;
            second = second > s_second[w] ? second : s_second[w];
            second = second > lose ? second : lose;
            if (s_best[w] > best || (s_best[w] == best && s_besti[w] < besti)) { best = s_best[w]; besti = s_besti[w]; }
        }
        const bool ok = s > 0.0 && isfinite(s);
        // renormalize falls back to uniform when the sum is not positive (LBP.py:650-657)
        const double b = ok ? (double)plab / s : 1.0 / (double)V;
        logp[g] = b > 0.0 ? log(b) : -99.99;                      // LBP.py:252-258
        top1[g] = ok ? besti : 0;
        rank[g] = ok ? (int)(c + 0.5) : 0;
        if (flags) {
            const int icnt = (int)(c + 0.5), inh = (int)(nh + 0.5), inl = (int)(nl + 0.5);
            int f = 0;
            if (ok && V > 1 && second >= best * (T)(1.0f - tau)) f |= 1;                 // the arg-max has a neighbour inside tau
            if (ok && (inh + inl) > 0 && icnt - inh <= 50) f |= 2;                        // the label's rank can change and can matter
            flags[g] = f;
            aux[2 * (size_t)g] = (double)best; aux[2 * (size_t)g + 1] = (double)plab;
            cnts[2 * (size_t)g] = icnt; cnts[2 * (size_t)g + 1] = inh;
            if (f) flagged[atomicAdd(n_flagged, 1)] = g;
        }
    }
    if (beliefs) {
        const bool ok = s > 0.0 && isfinite(s);
        float *brow = beliefs + (size_t)g * ldv;
        if (VEC) {
            for (int e = 4 * threadIdx.x; e < V; e += 4 * blockDim.x) {
                T p[4];
                prod4(e, p);
                float4 o;                                          // (columns >= V of the padded row: whatever the products are)
                o.x = ok ? (float)((double)p[0] / s) : 1.0f / (float)V; o.y = ok ? (float)((double)p[1] / s) : 1.0f / (float)V;
                o.z = ok ? (float)((double)p[2] / s) : 1.0f / (float)V; o.w = ok ? (float)((double)p[3] / s) : 1.0f / (float)V;
                if (e + 3 < V) *reinterpret_cast<float4 *>(brow + e) = o;
                else { const float ov[4] = {o.x, o.y, o.z, o.w}; for (int q = 0; q < 4 && e + q < V; ++q) brow[e + q] = ov[q]; }
            }
        } else {
            for (int e = threadIdx.x; e < V; e += blockDim.x) brow[e] = ok ? (float)((double)prod(e) / s) : 1.0f / (float)V;
        }
    }
}

}  // namespace mlbp

using namespace mlbp;

extern "C" int mlbp_fill_uniform_rows(void *A_hi, void *A_lo, int ldv, int V, const int32_t *rows, int n_rows,
                                      const uint8_t *keep, void *stream) {
    if (n_rows == 0) return MLBP_OK;
    MLBP_CHECK_ARG(A_hi && A_lo && rows && n_rows > 0 && V > 0 && ldv >= V, "fill_uniform_rows: bad argument");
    fill_uniform_rows_kernel<<<n_rows, 256, 0, as_stream(stream)>>>((__half *)A_hi, (__half *)A_lo, ldv, V, rows, keep);
    MLBP_LAUNCH_CHECK();
    return MLBP_OK;
}

static long long *g_k3_dbg = nullptr;
extern "C" void mlbp_debug_k3_times(long long *p) { g_k3_dbg = p; }

// resident (single-read) launch: cluster of C CTAs per group, (NIN + 1) * S floats of dynamic shared memory per CTA
template <int NIN>
static cudaError_t launch_resident(int n_groups, int C, int S, cudaStream_t st, const int32_t *grp_u,
                                   const int32_t *grp_off, const int32_t *in_row, const int32_t *dest_off,
                                   const int32_t *dest, const int32_t *first_dest, const int32_t *second_dest, const float *U,
                                   const float *D, int ldv, int V, __half *A_hi, __half *A_lo) {
    // function attributes and occupancy are per DEVICE: a process that drives several GPUs configures each one
    static bool configured[MLBP_MAX_DEVICES] = {};
    const int dev = current_device();
    auto kern = var_to_factor_resident_kernel<NIN>;
    if (!configured[dev]) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, K3_RESIDENT_SMEM);
        if (e != cudaSuccess) return e;
        configured[dev] = true;
    }
    const size_t smem = (size_t)(NIN + 1) * S * sizeof(float);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)C);                              // placeholder: set from the occupancy query below
    cfg.blockDim = dim3(K3R_THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)C; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    // persistent grid: as many clusters as the device keeps resident for this shared-memory size (queried once per C)
    static int resident_tab[MLBP_MAX_DEVICES][9] = {};
    int *resident = resident_tab[dev];
    if (!resident[C]) {
        int nc = 0;
        cudaError_t e = cudaOccupancyMaxActiveClusters(&nc, kern, &cfg);   // counts this device's SMs: nothing hard-coded
        if (e != cudaSuccess) return e;
        resident[C] = nc > 0 ? nc : 1;
        if (getenv("MLBP_DEBUG")) fprintf(stderr, "mlbp K3 resident<%d>: cluster %d, %zu B smem, %d resident clusters\n", NIN, C, smem, nc);
    }
    const int n_clusters = n_groups < resident[C] ? n_groups : resident[C];
    cfg.gridDim = dim3((unsigned)n_clusters * (unsigned)C);
    return cudaLaunchKernelEx(&cfg, kern, n_groups, grp_u, grp_off, in_row, dest_off, dest, first_dest, second_dest, U, D, ldv,
                              V, S, A_hi, A_lo, g_k3_dbg);
}

constexpr int K3_RESIDENT_MAX_IN = 24;

extern "C" int mlbp_var_to_factor(int n_groups, const int32_t *grp_u, const int32_t *grp_off, const int32_t *in_row,
                                  const int32_t *dest_off, const int32_t *dest, const int32_t *first_dest,
                                  const int32_t *second_dest, const float *U, const float *D, int ldv, int V, void *A_hi,
                                  void *A_lo, int max_in, float range_log2, void *stream) {
    if (n_groups == 0) return MLBP_OK;
    MLBP_CHECK_ARG(n_groups > 0 && grp_u && grp_off && in_row && dest_off && dest && first_dest && second_dest && U && D && A_hi && A_lo,
                   "var_to_factor: null pointer");
    const bool fp32_ok = range_log2 >= 0.f && range_log2 < 100.f;   // products provably stay inside 2^+-100
    MLBP_CHECK_ARG(V > 0 && ldv >= V && (ldv % 4) == 0, "var_to_factor: bad V/ldv");
    MLBP_CHECK_ARG(max_in >= 0, "var_to_factor: bad max_in");
    if (max_in > 48) {
        set_error("var_to_factor: a variable with %d pairwise factors exceeds the supported 48", max_in);
        return MLBP_ERR_UNSUPPORTED;
    }
    cudaStream_t st = as_stream(stream);
    // The resident single-read kernel runs whenever the products fit fp32 and the cluster's slices fit shared memory;
    // MLBP_K3_IMPL=1 forces the streaming two-read kernel (used by scripts/k3_probe.py to time both).
    const char *env_impl = getenv("MLBP_K3_IMPL");
    const int forced = env_impl ? atoi(env_impl) : 2;
    const int nin = max_in < 1 ? 1 : max_in;
    int C = 0, S = 0;
    if (fp32_ok && forced == 2 && nin <= K3_RESIDENT_MAX_IN && (((uintptr_t)U | (uintptr_t)D) & 15) == 0)
        for (int c = 1; c <= 8 && !C; c *= 2) {
            const int s4 = (((V + c - 1) / c) + 3) & ~3, s32 = (s4 + 31) & ~31;    // 128-byte slices when they still fit
            if ((size_t)(nin + 1) * s32 * sizeof(float) <= (size_t)K3_RESIDENT_SMEM) { C = c; S = s32; }
            else if ((size_t)(nin + 1) * s4 * sizeof(float) <= (size_t)K3_RESIDENT_SMEM) { C = c; S = s4; }
        }
    if (C) {
        if ((int64_t)n_groups * C > 0x7fffffffll) { set_error("var_to_factor: too many groups"); return MLBP_ERR_INVALID; }
#define MLBP_K3_RES(N)                                                                                             \
        case N:                                                                                                    \
            MLBP_CUDA(launch_resident<N>(n_groups, C, S, st, grp_u, grp_off, in_row, dest_off, dest, first_dest, second_dest, U, D, ldv, V, \
                                         (__half *)A_hi, (__half *)A_lo));                                         \
            break;
        switch (nin) {
            MLBP_K3_RES(1) MLBP_K3_RES(2) MLBP_K3_RES(3) MLBP_K3_RES(4) MLBP_K3_RES(5) MLBP_K3_RES(6) MLBP_K3_RES(7)
            MLBP_K3_RES(8) MLBP_K3_RES(9) MLBP_K3_RES(10) MLBP_K3_RES(11) MLBP_K3_RES(12) MLBP_K3_RES(13) MLBP_K3_RES(14)
            MLBP_K3_RES(15) MLBP_K3_RES(16) MLBP_K3_RES(17) MLBP_K3_RES(18) MLBP_K3_RES(19) MLBP_K3_RES(20)
            MLBP_K3_RES(21) MLBP_K3_RES(22) MLBP_K3_RES(23) MLBP_K3_RES(24)
        }
#undef MLBP_K3_RES
        MLBP_LAUNCH_CHECK();
        return MLBP_OK;
    }
    // up to 20 inputs the fp32 kernel is compiled for 3 CTAs per SM (80 registers): measured 1.28 ms vs 1.66 ms uncapped
#define MLBP_K3_LAUNCH(N)                                                                                        \
    do {                                                                                                         \
        if (fp32_ok && N <= 20)                                                                                  \
            var_to_factor_kernel<(N <= 20 ? N : 4), float, 3><<<n_groups, K3_THREADS, 0, st>>>(                  \
                grp_u, grp_off, in_row, dest_off, dest, first_dest, second_dest, U, D, ldv, V, (__half *)A_hi, (__half *)A_lo);           \
        else if (fp32_ok)                                                                                        \
            var_to_factor_kernel<N, float, 1><<<n_groups, K3_THREADS, 0, st>>>(                                  \
                grp_u, grp_off, in_row, dest_off, dest, first_dest, second_dest, U, D, ldv, V, (__half *)A_hi, (__half *)A_lo);           \
        else                                                                                                     \
            var_to_factor_kernel<N, double, 1><<<n_groups, K3_THREADS, 0, st>>>(                                 \
                grp_u, grp_off, in_row, dest_off, dest, first_dest, second_dest, U, D, ldv, V, (__half *)A_hi, (__half *)A_lo);           \
    } while (0)
    if (max_in <= 4) MLBP_K3_LAUNCH(4);
    else if (max_in <= 8) MLBP_K3_LAUNCH(8);
    else if (max_in <= 12) MLBP_K3_LAUNCH(12);
    else if (max_in <= 16) MLBP_K3_LAUNCH(16);
    else if (max_in <= 20) MLBP_K3_LAUNCH(20);
    else if (max_in <= 24) MLBP_K3_LAUNCH(24);
    else if (max_in <= 32) MLBP_K3_LAUNCH(32);
    else MLBP_K3_LAUNCH(48);
#undef MLBP_K3_LAUNCH
    MLBP_LAUNCH_CHECK();
    return MLBP_OK;
}

extern "C" int mlbp_topk_mask_rows(void *A_hi, void *A_lo, int ldv, int V, int64_t row0, int n_rows, int K, void *stream) {
    if (n_rows == 0 || K >= V) return MLBP_OK;
    MLBP_CHECK_ARG(A_hi && A_lo && n_rows > 0 && K > 0 && row0 >= 0 && ldv >= V, "topk_mask_rows: bad argument");
    topk_mask_rows_kernel<<<n_rows, 256, 0, as_stream(stream)>>>((__half *)A_hi, (__half *)A_lo, ldv, V, row0, K);
    MLBP_LAUNCH_CHECK();
    return MLBP_OK;
}

extern "C" int mlbp_marginals(int n_groups, const int32_t *grp_u, const int32_t *grp_off, const int32_t *in_row,
                              const int32_t *label, const float *U, const float *D, int ldv, int V, double *logp,
                              int32_t *top1, int32_t *rank, float *beliefs, float range_log2, int max_in, float tau,
                              float tau_label, double *aux, int32_t *cnts, int32_t *flags, int32_t *flagged,
                              int32_t *n_flagged, void *stream) {
    if (n_groups == 0) return MLBP_OK;
    MLBP_CHECK_ARG(n_groups > 0 && grp_u && grp_off && in_row && label && U && D && logp && top1 && rank,
                   "marginals: null pointer");
    if (max_in > 64) {                                            // the reference has no limit; this kernel's row table does
        set_error("marginals: a variable with %d incoming pairwise messages exceeds the supported 64", max_in);
        return MLBP_ERR_UNSUPPORTED;
    }
    MLBP_CHECK_ARG(!flags || (aux && cnts && flagged && n_flagged && tau >= 0.f && tau < 0.5f && tau_label >= 0.f && tau_label < 0.5f),
                   "marginals: near-tie detection needs aux, cnts, flagged, n_flagged and bands in [0, 0.5)");
    // 16-byte loads when every row starts 16-byte aligned (the engine's buffers do); else the element-wise variant
    const bool vec = (ldv % 4) == 0 && ((reinterpret_cast<uintptr_t>(U) | reinterpret_cast<uintptr_t>(D) |
                                         reinterpret_cast<uintptr_t>(beliefs)) % 16) == 0;
    const bool f32 = range_log2 >= 0.f && range_log2 < 100.f;
#define MLBP_K5(TT, VV)                                                                                                \
    marginals_kernel<TT, VV><<<n_groups, 256, 0, as_stream(stream)>>>(grp_u, grp_off, in_row, label, U, D, ldv, V, logp, top1, \
                                                                      rank, beliefs, tau, tau_label, aux, cnts, flags, flagged, n_flagged)
    if (f32 && vec) MLBP_K5(float, true);
    else if (f32) MLBP_K5(float, false);
    else if (vec) MLBP_K5(double, true);
    else MLBP_K5(double, false);
#undef MLBP_K5
    MLBP_LAUNCH_CHECK();
    return MLBP_OK;
}
