// K2: everything that depends on theta only.  The reference rebuilds exp(phi . theta) over the full
// (V,V,3) and (V,Vd,6) tensors for EVERY sentence (train.py:218-253); here it is one pass per SGD step that
// emits the tensor-core operand planes (fp16 hi/lo, both orientations) plus the small per-column /
// per-German-word statistics that make every unary factor O(1) in the gradient.
//
// Arithmetic: the planes keep 22 bits (fp16 hi + lo), so the exponentials are evaluated in fp32 -- but on an argument that is
// formed in double-float (a compensated fp32 pair): z = th_pmi * p + th_bias is split as z_hi + z_lo with |z_lo| ~ 2^-24 |z|,
// exp(z) = expf(z_hi) * (1 + z_lo).  Result: ~1 ulp of fp32 per table entry, no float64 instruction per element (the fp64
// pipe of this part issues only a few lanes per clock and SM: the float64 exp of round 1 ran at 0.27 of the HBM roofline).
// Column sums are accumulated as compensated fp32 pairs over the 8 rows a thread owns and in float64 above that, row sums in
// fp32 across the 64 columns of a tile and in float64 above; the rounding of the entries is random, so sums over V entries
// are good to ~1e-9 (columns) / ~1e-8 (rows) relative -- their consumers, the unary gradient and the constant messages, need 1e-6.
#include "common.cuh"

namespace mlbp {

constexpr int TS = 64;  // tile edge

struct ThetaEE { double pmi, w1, bias; };
struct ThetaED { double t[6]; };

// s += x for an unevaluated sum s = (hi, lo): two-sum, the rounding error of every addition is kept in lo
__device__ __forceinline__ void acc_f2(F2 &s, float x) {
    const float t = s.hi + x;
    const float bb = t - s.hi;
    s.lo += (s.hi - (t - bb)) + (x - bb);
    s.hi = t;
}
// hi half of a table entry by STOCHASTIC rounding: x is rounded down or up to fp16 with probabilities that make the expected
// value exact (13 pseudo-random bits, a hash of the cell, are added below the fp16 mantissa before truncation).  Why: feature
// planes are sparse (a PMI matrix is mostly zeros), so most entries of T = exp(theta . phi) are ONE constant, and round-to-
// nearest gives all of them the same error -- up to 2^-12 relative, in one direction.  The one-pass gradient rows (hi halves
// only) then see a normaliser Z = c'Tr that is off by that much while the numerator c'(T o PMI)r, whose entries under the
// zeros are exact zeros, is not: a systematic error of the expectation N/Z (measured 1.5e-4 relative on a sentence's
// gradient, tests/test_gpu_gates.py sparse_w1_negative).  With stochastic rounding the errors of equal entries are
// independent and average away like those of distinct entries; hi + lo still carries the full value.
__device__ __forceinline__ unsigned cell_hash(unsigned a, unsigned b) {
    unsigned h = a * 0x9E3779B1u + b * 0x85EBCA77u;
    h ^= h >> 15; h *= 0x2C1B3C6Du; h ^= h >> 12; h *= 0x297A2D39u; h ^= h >> 15;
    return h;
}
__device__ __forceinline__ __half half_stochastic(float x, unsigned r) {          // x >= 0
    const unsigned bits = (__float_as_uint(x) + (r & 0x1FFFu)) & 0xFFFFE000u;    // fp32 has 13 mantissa bits more than fp16
    return __float2half_rz(__uint_as_float(bits));
}
__device__ __forceinline__ __half half_stochastic_signed(float x, unsigned r) {  // magnitude rounded as above, sign kept
    const __half h = half_stochastic(fabsf(x), r);
    return x < 0.f ? __hneg(h) : h;
}

// One 64x64 tile of the (a, b) plane per CTA, 256 threads: thread (tx = tid % 32, ty = tid / 32) owns the column pair
// b0 + 2 tx, + 1 of rows ty, ty + 8, ...: 8-byte global loads and 4-byte (half2) plane stores, 128 bytes per warp and plane.
// The transposed planes go through shared memory and are written as half2 pairs along a.
__global__ void __launch_bounds__(256)
build_pairwise_tables_kernel(const float *__restrict__ pmi, const float *__restrict__ w1, int V, int ldf, F2 t_pmi, F2 t_w1,
                             F2 t_bias, float scale, __half *__restrict__ planes, int64_t ps, int ldv,
                             double *__restrict__ colsums, int with_grad, __half *__restrict__ r_planes, float tbar) {
    // hi / lo tiles of T, T1 (and G, G1, G1w with the gradient planes), indexed [a][b], for the transposed planes; the
    // column-sum partials reuse the storage once the tiles are written out.  Dynamic shared memory: 10 tiles = 84 KB.
    extern __shared__ __align__(16) unsigned char s_raw[];
    __half (*sT)[TS][TS + 2] = reinterpret_cast<__half (*)[TS][TS + 2]>(s_raw);
    double (*sSum)[8][TS] = reinterpret_cast<double (*)[8][TS]>(s_raw);
    static_assert(sizeof(double) * 5 * 8 * TS <= 4 * TS * (TS + 2) * sizeof(__half), "column-sum partials must fit the tile storage");
    const int n_tiles = with_grad ? 10 : 4;
    const int r_tile = n_tiles;                                   // two more tiles for the residual planes (r_planes != nullptr)
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int a0 = blockIdx.y * TS, b0 = blockIdx.x * TS;
    const int b = b0 + 2 * tx;
    F2 cs[5][2];                                                  // column sums over this thread's 8 rows, compensated
#pragma unroll
    for (int i = 0; i < 5; ++i) cs[i][0] = cs[i][1] = F2{0.f, 0.f};
    const F2 zero = {0.f, 0.f};
    for (int r = ty; r < TS; r += 8) {
        const int a = a0 + r;
        float rs_t = 0.f, rs_t1 = 0.f;
        __half2 h[10];
#pragma unroll
        for (int i = 0; i < 10; ++i) h[i] = __floats2half2_rn(0.f, 0.f);
        __half2 hr[2] = {h[0], h[0]};                             // residuals R = T - tbar, R1 = T1 - tbar (hi halves only)
        if (a < V && b < V) {                                     // ldf is even and >= V: the pair load stays inside the row
            const float2 p2 = *reinterpret_cast<const float2 *>(pmi + (size_t)a * ldf + b);
            const float2 w2 = *reinterpret_cast<const float2 *>(w1 + (size_t)a * ldf + b);
            const float pp[2] = {p2.x, p2.y}, ww[2] = {w2.x, w2.y};
            float v[5][2];
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                const bool in = b + q < V;
                const F2 z = axpb(t_pmi, pp[q], t_bias);
                const F2 zw = axpb(t_w1, ww[q], zero);
                const float t = in ? exp_f2(z) : 0.f;
                const float t1 = in ? t * exp_f2(zw) : 0.f;      // exp(z + th_w1 w) = exp(z) exp(th_w1 w)
                v[0][q] = t; v[1][q] = t1; v[2][q] = t * pp[q]; v[3][q] = t1 * pp[q]; v[4][q] = t1 * ww[q];
#pragma unroll
                for (int i = 0; i < 5; ++i) acc_f2(cs[i][q], v[i][q]);
            }
            rs_t = v[0][0] + v[0][1]; rs_t1 = v[1][0] + v[1][1];
            const unsigned r0 = cell_hash((unsigned)a, (unsigned)b), r1 = cell_hash((unsigned)a, (unsigned)b + 1u);
#pragma unroll
            for (int i = 0; i < 5; ++i) {
                const float2 x = make_float2(v[i][0] * scale, v[i][1] * scale);
                const __half2 hi = __halves2half2(half_stochastic(x.x, r0 >> (3 * i)), half_stochastic(x.y, r1 >> (3 * i)));
                const float2 back = __half22float2(hi);
                h[2 * i] = hi;
                h[2 * i + 1] = __floats2half2_rn(x.x - back.x, x.y - back.y);
            }
            const size_t o = (size_t)a * ldv + b;                 // even: 4-byte aligned
            if (r_planes) {
                // Residual planes for the ONE-pass message rows: T = tbar + R with tbar = T at phi = 0 (the value of every entry
                // under a zero of a sparse feature plane, and close to all entries once the pairwise weights are small): the
                // GEMM contracts the messages with fp16(R) and adds tbar * sum(message) -- a constant -- in its epilogue, so
                // the fp16 rounding is relative to |T - tbar|, not to T (exactly zero under the zeros).
                const unsigned q0 = cell_hash((unsigned)a ^ 0x5bd1e995u, (unsigned)b), q1 = cell_hash((unsigned)a ^ 0x5bd1e995u, (unsigned)b + 1u);
                const bool in1 = b + 1 < V;
                hr[0] = __halves2half2(half_stochastic_signed(v[0][0] * scale - tbar, q0), in1 ? half_stochastic_signed(v[0][1] * scale - tbar, q1) : __float2half_rn(0.f));
                hr[1] = __halves2half2(half_stochastic_signed(v[1][0] * scale - tbar, q0 >> 13), in1 ? half_stochastic_signed(v[1][1] * scale - tbar, q1 >> 13) : __float2half_rn(0.f));
                *reinterpret_cast<__half2 *>(r_planes + 0 * ps + o) = hr[0];
                *reinterpret_cast<__half2 *>(r_planes + 2 * ps + o) = hr[1];
            }
            auto st = [&](int plane, __half2 x) { *reinterpret_cast<__half2 *>(planes + plane * ps + o) = x; };
            st(0, h[0]); st(1, h[1]);                             // T
            st(4, h[2]); st(5, h[3]);                             // T1
            if (with_grad) {
                st(8, h[4]); st(9, h[5]);                         // G   = T  o PMI
                st(10, h[6]); st(11, h[7]);                       // G1  = T1 o PMI
                st(12, h[8]); st(13, h[9]);                       // G1w = T1 o PMI_w1
            }
        }
#pragma unroll
        for (int i = 0; i < 10; ++i)
            if (i < n_tiles) *reinterpret_cast<__half2 *>(&sT[i][r][2 * tx]) = h[i];
        if (r_planes) {
            *reinterpret_cast<__half2 *>(&sT[r_tile][r][2 * tx]) = hr[0];
            *reinterpret_cast<__half2 *>(&sT[r_tile + 1][r][2 * tx]) = hr[1];
        }
        // row sums of T and T1 (message of a pairwise factor whose input is still the uniform initial message)
        rs_t = warp_sum_f32(rs_t); rs_t1 = warp_sum_f32(rs_t1);
        if (tx == 0 && a < V) {
            atomicAdd(&colsums[(size_t)5 * V + a], (double)rs_t);
            atomicAdd(&colsums[(size_t)6 * V + a], (double)rs_t1);
        }
    }
    __syncthreads();
    // transposed planes: Tt[b][a] = T[a][b]; threads now run along a in pairs
    for (int r = ty; r < TS; r += 8) {
        const int bb = b0 + r, aa = a0 + 2 * tx;
        if (bb < V && aa < V) {                                   // aa + 1 < ldv: the padding column receives the zero of sT
            const size_t o = (size_t)bb * ldv + aa;
            // tiles 0..3 -> planes 2, 3 (Tt) and 6, 7 (T1t); tiles 4..9 -> planes 14..19 (Gt, G1t, G1wt: the spike compensation
            // of the gradient rows reads a COLUMN of T o PMI as a row of these)
#pragma unroll
            for (int i = 0; i < 10; ++i)
                if (i < n_tiles) {
                    const __half2 x = __halves2half2(sT[i][2 * tx][r], sT[i][2 * tx + 1][r]);
                    *reinterpret_cast<__half2 *>(planes + (i < 2 ? 2 + i : (i < 4 ? 4 + i : 10 + i)) * ps + o) = x;
                }
            if (r_planes) {                                       // Rt, R1t
                *reinterpret_cast<__half2 *>(r_planes + 1 * ps + o) = __halves2half2(sT[r_tile][2 * tx][r], sT[r_tile][2 * tx + 1][r]);
                *reinterpret_cast<__half2 *>(r_planes + 3 * ps + o) = __halves2half2(sT[r_tile + 1][2 * tx][r], sT[r_tile + 1][2 * tx + 1][r]);
            }
        }
    }
    __syncthreads();                                              // the tiles are dead: their storage takes the partial sums
#pragma unroll
    for (int i = 0; i < 5; ++i) {
        sSum[i][ty][2 * tx] = (double)cs[i][0].hi + (double)cs[i][0].lo;
        sSum[i][ty][2 * tx + 1] = (double)cs[i][1].hi + (double)cs[i][1].lo;
    }
    __syncthreads();
    if (threadIdx.x < TS && b0 + threadIdx.x < V) {
#pragma unroll
        for (int i = 0; i < 5; ++i) {
            double s = 0.0;
#pragma unroll
            for (int y = 0; y < 8; ++y) s += sSum[i][y][threadIdx.x];
            atomicAdd(&colsums[(size_t)i * V + b0 + threadIdx.x], s);
        }
    }
}

// one CTA per German word d: sum_e psi, sum_e psi*ed, sum_e psi*ped over the de-major rows
__global__ void __launch_bounds__(256)
build_unary_tables_kernel(const float *__restrict__ edT, const float *__restrict__ pedT, int V, int ldf, ThetaED th,
                          double *__restrict__ edstats) {
    __shared__ double red[32];
    const int d = blockIdx.x;
    const float *e = edT + (size_t)d * ldf, *p = pedT + (size_t)d * ldf;
    double s0 = 0, s1 = 0, s2 = 0;
    for (int i = threadIdx.x; i < V; i += blockDim.x) {
        const double x = e[i], y = p[i];
        const double psi = exp(th.t[0] * x + th.t[1] * y + th.t[5]);
        s0 += psi; s1 += psi * x; s2 += psi * y;
    }
    s0 = block_sum(s0, red); s1 = block_sum(s1, red); s2 = block_sum(s2, red);
    if (threadIdx.x == 0) {
        edstats[3 * d + 0] = s0; edstats[3 * d + 1] = s1; edstats[3 * d + 2] = s2;
    }
}

}  // namespace mlbp

using namespace mlbp;

extern "C" int mlbp_build_pairwise_tables(const float *pmi, const float *pmi_w1, int V, int ldf,
                                          const double *h_theta_ee, int scale_exp, void *planes,
                                          int64_t plane_stride, int ldv, double *colsums, int with_grad_planes,
                                          void *r_planes, float *h_tbar, void *stream) {
    MLBP_CHECK_ARG(pmi && pmi_w1 && planes && colsums && h_theta_ee, "build_pairwise_tables: null pointer");
    MLBP_CHECK_ARG(V > 0 && ldf >= V && (ldf % 2) == 0 && ldv >= V && (ldv % 64) == 0, "build_pairwise_tables: bad V/ld (%d,%d,%d)", V, ldf, ldv);
    MLBP_CHECK_ARG(plane_stride >= (int64_t)V * ldv && (plane_stride % 2) == 0, "build_pairwise_tables: plane_stride too small or odd");
    MLBP_CHECK_ARG(((reinterpret_cast<uintptr_t>(pmi) | reinterpret_cast<uintptr_t>(pmi_w1)) % 8) == 0 &&
                   (reinterpret_cast<uintptr_t>(planes) % 4) == 0, "build_pairwise_tables: misaligned buffer");
    MLBP_CHECK_ARG(scale_exp > -120 && scale_exp < 120, "build_pairwise_tables: scale_exp out of range");
    cudaStream_t st = as_stream(stream);
    MLBP_CUDA(cudaMemsetAsync(colsums, 0, sizeof(double) * MLBP_N_SUMS * (size_t)V, st));
    dim3 grid((V + TS - 1) / TS, (V + TS - 1) / TS);
    MLBP_CHECK_ARG(!r_planes || (reinterpret_cast<uintptr_t>(r_planes) % 4) == 0, "build_pairwise_tables: misaligned residual planes");
    const size_t smem = (size_t)((with_grad_planes ? 10 : 4) + (r_planes ? 2 : 0)) * TS * (TS + 2) * sizeof(__half);
    // tbar = T at phi = 0, scaled like the planes: what the one-pass message GEMM adds back as a constant (see the kernel)
    // (*h_tbar > 0 on entry: the caller's choice of the constant, already scaled; else the default, written back)
    const float tbar = (h_tbar && *h_tbar > 0.f) ? *h_tbar : (float)(exp(h_theta_ee[2]) * ldexp(1.0, scale_exp));
    if (h_tbar) *h_tbar = tbar;
    static bool attr_set_dev[MLBP_MAX_DEVICES] = {};
    if (!attr_set_dev[current_device()]) {
        MLBP_CUDA(cudaFuncSetAttribute(build_pairwise_tables_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       12 * TS * (TS + 2) * (int)sizeof(__half)));
        attr_set_dev[current_device()] = true;
    }
    build_pairwise_tables_kernel<<<grid, 256, smem, st>>>(pmi, pmi_w1, V, ldf, split_double(h_theta_ee[0]),
                                                       split_double(h_theta_ee[1]), split_double(h_theta_ee[2]),
                                                       ldexpf(1.0f, scale_exp), (__half *)planes, plane_stride, ldv, colsums,
                                                       with_grad_planes, (__half *)r_planes, tbar);
    MLBP_LAUNCH_CHECK();
    return MLBP_OK;
}

extern "C" int mlbp_build_unary_tables(const float *edT, const float *pedT, int V, int Vd, int ldf,
                                       const double *h_theta_ed, double *edstats, void *stream) {
    MLBP_CHECK_ARG(edT && pedT && edstats && h_theta_ed, "build_unary_tables: null pointer");
    MLBP_CHECK_ARG(V > 0 && Vd > 0 && ldf >= V, "build_unary_tables: bad shape");
    ThetaED th;
    for (int i = 0; i < 6; ++i) th.t[i] = h_theta_ed[i];
    build_unary_tables_kernel<<<Vd, 256, 0, as_stream(stream)>>>(edT, pedT, V, ldf, th, edstats);
    MLBP_LAUNCH_CHECK();
    return MLBP_OK;
}
