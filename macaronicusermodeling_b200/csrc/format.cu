// K7: the text of the .dist lines (FactorGraph.to_dist, LBP.py:125-143) ON THE DEVICE.
//
// For every belief row the reference writes  ' '.join('%0.6f' % x for x in np.log(row.astype(np.float64))).  On the host that
// is ~3 ms per predicted token at V = 10 000; here the bytes are made where the beliefs already are and copied back once.
//
// Two requirements make this more than a printf:
//   * log: the printed digits must be those of the correctly rounded float64 log of the float64 value of each float32 input
//     (CUDA's log() is documented at up to 1 ulp, and 1 ulp across a decimal rounding boundary changes a digit).  The log is
//     evaluated in double-double (~2^-100 relative) and rounded once to double.
//   * decimal: CPython '%0.6f' rounds the EXACT binary value half-to-even.  |log| < 2^7 and the float64 mantissa has 53 bits,
//     so y * 10^6 = M * 5^6 * 2^(E + 6) with M * 5^6 < 2^67: one 128-bit product and a shift with half-even rounding.
//
// Layout: one CTA per row.  Pass 1 writes every row's byte count to offsets[r + 1], pass 2 scans them (one CTA, integer sums:
// deterministic), pass 3 formats each tile of 256 numbers into shared memory at block-scanned positions and copies the tile
// out coalesced.  Passes 1 and 3 both evaluate the log: recomputing it is cheaper than a scratch buffer of lengths.
#include "common.cuh"

namespace mlbp {

constexpr int FMT_THREADS = 256;
constexpr int FMT_SCAN_THREADS = 1024;

// ---- double-double arithmetic (value = hi + lo, |lo| <= ulp(hi) / 2)
struct dd { double hi, lo; };

__device__ __forceinline__ dd two_sum(double a, double b) {
    const double s = a + b, bb = s - a;
    return {s, (a - (s - bb)) + (b - bb)};
}
__device__ __forceinline__ dd quick_two_sum(double a, double b) {
    const double s = a + b;
    return {s, b - (s - a)};
}
__device__ __forceinline__ dd dd_add(dd a, dd b) {
    dd s = two_sum(a.hi, b.hi);
    const dd t = two_sum(a.lo, b.lo);
    s.lo += t.hi;
    s = quick_two_sum(s.hi, s.lo);
    s.lo += t.lo;
    return quick_two_sum(s.hi, s.lo);
}
__device__ __forceinline__ dd dd_mul(dd a, dd b) {
    const double p = a.hi * b.hi;
    double e = fma(a.hi, b.hi, -p);
    e = fma(a.hi, b.lo, fma(a.lo, b.hi, e));
    return quick_two_sum(p, e);
}
// 1 / d as a double-double (d a small odd integer): the remainder fma(-q, d, 1) is exact
__device__ __forceinline__ dd dd_recip(double d) {
    const double q = 1.0 / d;
    return {q, fma(-q, d, 1.0) / d};
}

// Correctly rounded (up to the double-double error, ~2^-100 relative) float64 log of a positive finite float.
//   x = 2^k m, m in [sqrt(1/2), sqrt(2));  log x = k ln2 + 2 atanh(s),  s = (m - 1) / (m + 1),  |s| <= 0.1716,
//   atanh(s) = s (1 + z P(z)), z = s^2 <= 0.0295, P(z) = sum_n z^(n-1) / (2n + 1).
// Terms n >= 11 of P are below 2^-53 of the result and are summed in double; n = 1..10 in double-double.
__device__ double log_f32_cr(float xf) {
    unsigned bits = __float_as_uint(xf);
    int k;
    unsigned mant;
    if ((bits >> 23) == 0) {                                  // subnormal: normalise the 23-bit fraction
        const int lz = __clz(bits) - 8;                       // leading zeros inside the 24-bit field
        mant = (bits << lz) & 0x7fffffu;
        k = -126 - lz;
    } else {
        mant = bits & 0x7fffffu;
        k = (int)(bits >> 23) - 127;
    }
    double m = 1.0 + (double)mant * 0x1p-23;                  // exact, in [1, 2)
    if (m > 1.4142135623730951) { m *= 0.5; ++k; }            // exact
    const double num = m - 1.0, den = m + 1.0;                // both exact (m has 24 significant bits)
    dd s;
    s.hi = num / den;
    s.lo = fma(-s.hi, den, num) / den;
    const dd z = dd_mul(s, s);
    double t = 1.0 / 43.0;                                    // n = 21 .. 11 in double
#pragma unroll
    for (int n = 20; n >= 11; --n) t = fma(t, z.hi, 1.0 / (2 * n + 1));
    dd p = {t, 0.0};
#pragma unroll
    for (int n = 10; n >= 1; --n) p = dd_add(dd_mul(p, z), dd_recip((double)(2 * n + 1)));
    dd a = dd_add(dd_mul(z, p), dd{1.0, 0.0});                // atanh(s) / s
    a = dd_mul(a, s);
    a.hi *= 2.0; a.lo *= 2.0;                                 // log m
    const dd ln2 = {0x1.62e42fefa39efp-1, 0x1.abc9e3b39803fp-56};
    const dd kl = dd_mul(dd{(double)k, 0.0}, ln2);
    const dd r = dd_add(kl, a);
    return r.hi + r.lo;
}

// '%0.6f' % log(x) of one float into buf (at most 11 bytes: "-103.278930" is the longest); returns the byte count.
__device__ int format_log(float x, char *buf) {
    if (x != x || x < 0.f) { buf[0] = 'n'; buf[1] = 'a'; buf[2] = 'n'; return 3; }      // np.log: nan for x < 0
    if (x == 0.f) { buf[0] = '-'; buf[1] = 'i'; buf[2] = 'n'; buf[3] = 'f'; return 4; }
    if (isinf(x)) { buf[0] = 'i'; buf[1] = 'n'; buf[2] = 'f'; return 3; }
    int n = 0;
    unsigned long long q = 0;
    if (x != 1.f) {
        const double y = log_f32_cr(x);
        if (y < 0.0) buf[n++] = '-';                          // also when the value rounds to zero: "-0.000000"
        const unsigned long long b = __double_as_longlong(fabs(y));
        const unsigned long long M = (b & 0xfffffffffffffull) | 0x10000000000000ull;   // |y| >= 2^-25: normal
        const int sh = 1075 - (int)(b >> 52) - 6;             // |y| 10^6 = M 5^6 2^-sh, sh in [40, 72]
        const unsigned __int128 N = (unsigned __int128)M * 15625u;
        q = (unsigned long long)(N >> sh);
        const unsigned __int128 rem = N & (((unsigned __int128)1 << sh) - 1), half = (unsigned __int128)1 << (sh - 1);
        if (rem > half || (rem == half && (q & 1ull))) ++q;   // round half to even on the exact value
    }
    const unsigned ip = (unsigned)(q / 1000000ull), fp = (unsigned)(q % 1000000ull);
    if (ip >= 100) buf[n++] = '0' + ip / 100;
    if (ip >= 10) buf[n++] = '0' + (ip / 10) % 10;
    buf[n++] = '0' + ip % 10;
    buf[n++] = '.';
    unsigned f = fp;
#pragma unroll
    for (int i = 5; i >= 0; --i) { buf[n + i] = '0' + f % 10; f /= 10; }
    return n + 6;
}

__global__ void __launch_bounds__(FMT_THREADS)
format_len_kernel(const float *__restrict__ X, int ldx, int V, int64_t *__restrict__ offsets) {
    const float *x = X + (size_t)blockIdx.x * ldx;
    unsigned long long len = 0;
    char buf[12];
    for (int e = threadIdx.x; e < V; e += FMT_THREADS) len += format_log(__ldg(x + e), buf);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) len += __shfl_xor_sync(0xffffffffu, len, o);
    __shared__ unsigned long long red[FMT_THREADS / 32];
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = len;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long t = (unsigned long long)(V - 1);   // separators
        for (int w = 0; w < FMT_THREADS / 32; ++w) t += red[w];
        offsets[(size_t)blockIdx.x + 1] = (int64_t)t;
    }
}

// in-place inclusive scan of offsets[1 .. n], offsets[0] = 0 (one CTA)
__global__ void __launch_bounds__(FMT_SCAN_THREADS) format_scan_kernel(int64_t *offsets, int n) {
    __shared__ long long wsum[FMT_SCAN_THREADS / 32];
    __shared__ long long s_carry;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) { s_carry = 0; offsets[0] = 0; }
    __syncthreads();
    for (int base = 0; base < n; base += FMT_SCAN_THREADS) {
        const int i = base + threadIdx.x;
        long long v = i < n ? (long long)offsets[i + 1] : 0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long u = __shfl_up_sync(0xffffffffu, v, o);
            if (lane >= o) v += u;
        }
        if (lane == 31) wsum[warp] = v;
        __syncthreads();
        long long before = s_carry, total = 0;
        for (int w = 0; w < FMT_SCAN_THREADS / 32; ++w) {
            if (w < warp) before += wsum[w];
            total += wsum[w];
        }
        if (i < n) offsets[i + 1] = (int64_t)(before + v);
        __syncthreads();
        if (threadIdx.x == 0) s_carry += total;
        __syncthreads();
    }
}

__global__ void __launch_bounds__(FMT_THREADS)
format_write_kernel(const float *__restrict__ X, int ldx, int V, const int64_t *__restrict__ offsets, char *__restrict__ out) {
    __shared__ char tile[FMT_THREADS * 12];
    __shared__ int wsum[FMT_THREADS / 32];
    const float *x = X + (size_t)blockIdx.x * ldx;
    char *dst = out + offsets[blockIdx.x];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int e0 = 0; e0 < V; e0 += FMT_THREADS) {
        const int e = e0 + threadIdx.x;
        char buf[12];
        int len = 0;
        if (e < V) {
            len = format_log(__ldg(x + e), buf);
            if (e + 1 < V) buf[len++] = ' ';
        }
        int v = len;                                          // block exclusive scan of the byte counts
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int u = __shfl_up_sync(0xffffffffu, v, o);
            if (lane >= o) v += u;
        }
        if (lane == 31) wsum[warp] = v;
        __syncthreads();
        int before = v - len, total = 0;
        for (int w = 0; w < FMT_THREADS / 32; ++w) {
            if (w < warp) before += wsum[w];
            total += wsum[w];
        }
        for (int i = 0; i < len; ++i) tile[before + i] = buf[i];
        __syncthreads();
        for (int i = threadIdx.x; i < total; i += FMT_THREADS) dst[i] = tile[i];
        dst += total;
        __syncthreads();                                      // tile and wsum are reused by the next 256 numbers
    }
}

}  // namespace mlbp

using namespace mlbp;

extern "C" int mlbp_format_log_rows(const float *X, int ldx, int V, int n_rows, char *out, int64_t out_bytes, int64_t *offsets,
                                    void *stream) {
    MLBP_CHECK_ARG(offsets && n_rows >= 0 && V > 0 && V <= (1 << 26) && ldx >= V && out_bytes >= 0,
                   "format_log_rows: bad argument");
    MLBP_CHECK_ARG(n_rows == 0 || (X && out), "format_log_rows: null pointer");
    MLBP_CHECK_ARG(out_bytes / MLBP_FMT_MAX_BYTES / V >= n_rows,
                   "format_log_rows: the text buffer needs %d * V * n_rows = %lld bytes, got %lld", MLBP_FMT_MAX_BYTES,
                   (long long)MLBP_FMT_MAX_BYTES * V * n_rows, (long long)out_bytes);
    cudaStream_t s = as_stream(stream);
    if (n_rows == 0) {
        MLBP_CUDA(cudaMemsetAsync(offsets, 0, sizeof(int64_t), s));
        return MLBP_OK;
    }
    format_len_kernel<<<n_rows, FMT_THREADS, 0, s>>>(X, ldx, V, offsets);
    MLBP_LAUNCH_CHECK();
    format_scan_kernel<<<1, FMT_SCAN_THREADS, 0, s>>>(offsets, n_rows);
    MLBP_LAUNCH_CHECK();
    format_write_kernel<<<n_rows, FMT_THREADS, 0, s>>>(X, ldx, V, offsets, out);
    MLBP_LAUNCH_CHECK();
    return MLBP_OK;
}
