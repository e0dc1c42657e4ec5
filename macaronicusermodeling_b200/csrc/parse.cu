// K8: the np.loadtxt text of a feature matrix (train.py:589-603) parsed ON THE DEVICE into padded fp32 planes.
//
// The host streams a file in chunks that end on a line boundary; each chunk is parsed by three launches:
//   1. summary: every thread classifies 16 bytes (field starts, comment state, bytes the grammar does not allow) and each CTA
//      writes what its 4 096-byte tile does to the field count and to the "inside a # comment" state, for both entry states;
//   2. scan:    one CTA turns the tile summaries into each tile's absolute field index and entry state, starting from the
//               running field counter state[0], and advances the counter (successive chunks need no host synchronisation);
//   3. write:   every field is converted and stored at out[row * ld_out + col], (row, col) = divmod(field index, n_cols).
// Fields are converted to the correctly rounded float64 (Eisel-Lemire with a 128-bit table of powers of five: exact for any
// decimal significand below 2^64), then rounded once to fp32 -- what np.ascontiguousarray(a, dtype=np.float32) does to the
// float64 array np.loadtxt returns.  A field with more than 19 significant digits is converted from its first 19 digits w and
// from w + 1; when the two disagree it is listed in `hard` for the host to convert.  Everything but the order of the hard list
// is deterministic (the host sorts it).
#include "common.cuh"
#include "pow5.cuh"

namespace mlbp {

constexpr int PARSE_THREADS = 256;
constexpr int PARSE_SEG = 16;                                  // bytes per thread: one 16-byte load
static_assert(PARSE_THREADS * PARSE_SEG == MLBP_PARSE_TILE_BYTES, "tile size");
constexpr int PARSE_SCAN_THREADS = 1024;
constexpr uint64_t F64_INF = 0x7ff0000000000000ull, F64_QNAN = 0x7ff8000000000000ull, F64_SIGN = 1ull << 63;

enum { FIELD_OK = 0, FIELD_BAD = 1, FIELD_HARD = 2 };

[[maybe_unused]] static const uint64_t h_pow5[] = {MLBP_POW5_TABLE};
__device__ const uint64_t d_pow5[] = {MLBP_POW5_TABLE};

__host__ __device__ __forceinline__ uint64_t pow5_word(int i) {
#ifdef __CUDA_ARCH__
    return __ldg(reinterpret_cast<const unsigned long long *>(d_pow5) + i);
#else
    return h_pow5[i];
#endif
}

__host__ __device__ __forceinline__ int clz64(uint64_t x) {
#ifdef __CUDA_ARCH__
    return __clzll((long long)x);
#else
    return __builtin_clzll(x);
#endif
}

// Bits of the float64 nearest to w * 10^q (w > 0), ties to even: the Eisel-Lemire algorithm as in the fast_float library
// (Lemire, "Number parsing at a gigabyte per second", 2021; Mushtak & Lemire, "Fast number parsing without fallback", 2023:
// the 128-bit product decides every case, no fallback is needed).
__host__ __device__ inline uint64_t eisel_lemire(uint64_t w, int64_t q) {
    if (q < MLBP_POW5_MIN_Q) return 0;
    if (q > MLBP_POW5_MAX_Q) return F64_INF;
    const int lz = clz64(w);
    w <<= lz;
    const int idx = 2 * (int)(q - MLBP_POW5_MIN_Q);
    const unsigned __int128 p1 = (unsigned __int128)w * pow5_word(idx);
    uint64_t hi = (uint64_t)(p1 >> 64), lo = (uint64_t)p1;
    if ((hi & 0x1ff) == 0x1ff) {                               // the truncated table entry may matter: add its low word
        const uint64_t h2 = (uint64_t)(((unsigned __int128)w * pow5_word(idx + 1)) >> 64);
        lo += h2;
        if (h2 > lo) ++hi;
    }
    const int upper = (int)(hi >> 63), shift = upper + 9;
    uint64_t m = hi >> shift;
    int e2 = (int)(((217706 * (int)q) >> 16) + 63) + upper - lz + 1023;   // floor(q log2 10) + 63 + ...
    if (e2 <= 0) {                                             // subnormal (or zero) after rounding
        if (-e2 + 1 >= 64) return 0;
        m >>= -e2 + 1;
        m += m & 1;
        m >>= 1;
        return m;                                              // m == 2^52 is the smallest normal: the same bits
    }
    if (lo <= 1 && q >= -4 && q <= 23 && (m & 3) == 1 && (m << shift) == hi) m &= ~1ull;   // exact tie: to even
    m += m & 1;
    m >>= 1;
    if (m >= (2ull << 52)) { m = 1ull << 52; ++e2; }
    m &= ~(1ull << 52);
    if (e2 >= 0x7ff) return F64_INF;
    return ((uint64_t)e2 << 52) | m;
}

__host__ __device__ __forceinline__ bool is_sep(unsigned c) {
    return c == ' ' || c == '\t' || c == '\n' || c == '\v' || c == '\f' || c == '\r';
}
__host__ __device__ __forceinline__ bool ends_field(unsigned c) { return is_sep(c) || c == '#'; }
__host__ __device__ __forceinline__ bool is_digit(unsigned c) { return c - '0' < 10u; }

// case-insensitive comparison of [s, s + len) with the lower-case word w
__host__ __device__ __forceinline__ bool same_word(const unsigned char *s, int64_t len, const char *w) {
    int i = 0;
    for (; w[i]; ++i)
        if (i >= len || (s[i] | 0x20) != (unsigned char)w[i]) return false;
    return i == len;
}

struct Field { int status; uint64_t bits; };

// One field [s, e) (no separator, no '#') as PyOS_string_to_double reads it -- the float parser behind np.loadtxt:
// [+-] (digits [. digits] | . digits) [(e|E) [+-] digits]  or  [+-] (inf | infinity | nan), case-insensitive.
__host__ __device__ inline Field parse_field(const unsigned char *s, const unsigned char *e) {
    const unsigned char *p = s;
    uint64_t sign = 0;
    if (p < e && (*p == '+' || *p == '-')) { sign = (*p == '-') ? F64_SIGN : 0; ++p; }
    if (p == e) return {FIELD_BAD, 0};
    const unsigned c0 = *p | 0x20;
    if (c0 == 'i' || c0 == 'n') {
        if (same_word(p, e - p, "inf") || same_word(p, e - p, "infinity")) return {FIELD_OK, sign | F64_INF};
        if (same_word(p, e - p, "nan")) return {FIELD_OK, sign | F64_QNAN};
        return {FIELD_BAD, 0};
    }
    uint64_t w = 0;
    int nd = 0;                                               // significant digits kept in w (at most 19)
    int64_t e10 = 0;
    bool any = false, dropped = false;                        // a digit was seen; a non-zero digit did not fit in w
    for (; p < e && is_digit(*p); ++p) {
        const unsigned d = *p - '0';
        any = true;
        if (w == 0 && d == 0) continue;                       // leading zero
        if (nd < 19) { w = w * 10 + d; ++nd; } else { ++e10; dropped |= d != 0; }
    }
    if (p < e && *p == '.') {
        for (++p; p < e && is_digit(*p); ++p) {
            const unsigned d = *p - '0';
            any = true;
            if (w == 0 && d == 0) { --e10; continue; }
            if (nd < 19) { w = w * 10 + d; ++nd; --e10; } else { dropped |= d != 0; }
        }
    }
    if (!any) return {FIELD_BAD, 0};
    if (p < e && (*p | 0x20) == 'e') {
        ++p;
        bool neg = false;
        if (p < e && (*p == '+' || *p == '-')) { neg = *p == '-'; ++p; }
        if (p == e || !is_digit(*p)) return {FIELD_BAD, 0};
        int64_t x = 0;
        for (; p < e && is_digit(*p); ++p)
            if (x < 1000000000000000ll) x = x * 10 + (*p - '0');   // beyond 10^15 the value is 0 or inf either way
        e10 += neg ? -x : x;
    }
    if (p != e) return {FIELD_BAD, 0};
    if (w == 0) return {FIELD_OK, sign};
    const uint64_t b = eisel_lemire(w, e10);
    if (dropped && eisel_lemire(w + 1, e10) != b) return {FIELD_HARD, 0};
    return {FIELD_OK, sign | b};
}

// what 16 bytes [i0, i0 + 16) of a chunk hold: bit j of
//   start  byte j begins a token (it is not a separator or '#', the byte before it is, or it is the first byte of the chunk)
//   com0   byte j lies inside a comment if the segment is entered outside one; com1 the same if entered inside one
//   bad    byte j is not in the grammar: >= 0x80, a control byte other than \t \n \v \f, or \r not followed by \n
struct SegBits { unsigned start, com0, com1, bad; bool out0, out1; };

__device__ __forceinline__ unsigned byte_of(uint4 v, int j) {
    const unsigned w = j < 4 ? v.x : j < 8 ? v.y : j < 12 ? v.z : v.w;
    return (w >> (8 * (j & 3))) & 0xffu;
}

__device__ __forceinline__ SegBits classify(const unsigned char *__restrict__ t, int64_t n, int64_t i0) {
    const int cnt = n - i0 < PARSE_SEG ? (int)(n - i0) : PARSE_SEG;
    uint4 v = make_uint4(0, 0, 0, 0);
    if (cnt == PARSE_SEG) {
        v = __ldg(reinterpret_cast<const uint4 *>(t + i0));   // i0 is a multiple of 16, text is 16-byte aligned
    } else {
        unsigned wv[4] = {0, 0, 0, 0};
#pragma unroll
        for (int j = 0; j < PARSE_SEG; ++j)
            if (j < cnt) wv[j >> 2] |= (unsigned)__ldg(t + i0 + j) << (8 * (j & 3));
        v = make_uint4(wv[0], wv[1], wv[2], wv[3]);
    }
    const unsigned next = (i0 + PARSE_SEG < n) ? __ldg(t + i0 + PARSE_SEG) : 0u;
    bool prev_end = (i0 == 0) || ends_field(__ldg(t + i0 - 1));
    bool s0 = false, s1 = true;
    SegBits r = {0, 0, 0, 0, false, true};
#pragma unroll
    for (int j = 0; j < PARSE_SEG; ++j) {
        if (j < cnt) {
            const unsigned c = byte_of(v, j), nx = j + 1 < PARSE_SEG ? byte_of(v, j + 1) : next;
            if (c == '\n') { s0 = false; s1 = false; }
            else if (c == '#') { s0 = true; s1 = true; }
            const bool end = ends_field(c);
            if (!end && prev_end) r.start |= 1u << j;
            if (s0) r.com0 |= 1u << j;
            if (s1) r.com1 |= 1u << j;
            const bool ok = (c >= 0x20 && c < 0x7f) || c == '\t' || c == '\n' || c == '\v' || c == '\f' ||
                            (c == '\r' && nx == '\n');   // (bytes past the chunk's end read as 0)
            if (!ok) r.bad |= 1u << j;
            prev_end = end;
        }
    }
    r.out0 = s0;
    r.out1 = s1;
    return r;
}

// What a stretch of text does: fields counted (a0 entered outside a comment, a1 inside one) and the comment state it leaves
// (bit 0: entered outside, bit 1: entered inside).  compose(L, R) = L then R; the identity is {0, 0, 2}.
struct Seg { unsigned a0, a1, o; };

__device__ __forceinline__ Seg compose(Seg L, Seg R) {
    Seg r;
    r.a0 = L.a0 + ((L.o & 1) ? R.a1 : R.a0);
    r.a1 = L.a1 + ((L.o & 2) ? R.a1 : R.a0);
    const unsigned o0 = (L.o & 1) ? (R.o >> 1) & 1 : R.o & 1, o1 = (L.o & 2) ? (R.o >> 1) & 1 : R.o & 1;
    r.o = o0 | (o1 << 1);
    return r;
}

__device__ __forceinline__ Seg seg_of(const SegBits &b) {
    return {(unsigned)__popc(b.start & ~b.com0), (unsigned)__popc(b.start & ~b.com1), (b.out0 ? 1u : 0u) | (b.out1 ? 2u : 0u)};
}

__device__ __forceinline__ Seg shfl_up_seg(Seg s, int o) {
    return {__shfl_up_sync(0xffffffffu, s.a0, o), __shfl_up_sync(0xffffffffu, s.a1, o), __shfl_up_sync(0xffffffffu, s.o, o)};
}

// block-wide scan of Seg (blockDim.x = NT): returns the thread's EXCLUSIVE prefix; *total = the whole block
template <int NT>
__device__ __forceinline__ Seg block_scan(Seg s, Seg *total) {
    __shared__ Seg wsum[NT / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    Seg v = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const Seg u = shfl_up_seg(v, o);
        if (lane >= o) v = compose(u, v);
    }
    Seg ex = shfl_up_seg(v, 1);
    if (lane == 0) ex = {0, 0, 2};
    if (lane == 31) wsum[warp] = v;
    __syncthreads();
    Seg before = {0, 0, 2}, all = {0, 0, 2};
    for (int w = 0; w < NT / 32; ++w) {
        if (w < warp) before = compose(before, wsum[w]);
        all = compose(all, wsum[w]);
    }
    *total = all;
    return compose(before, ex);
}

__device__ __forceinline__ unsigned long long pack_seg(Seg s) {
    return (unsigned long long)s.a0 | ((unsigned long long)s.a1 << 24) | ((unsigned long long)s.o << 48);
}
__device__ __forceinline__ Seg unpack_seg(unsigned long long x) {
    return {(unsigned)(x & 0xffffffu), (unsigned)((x >> 24) & 0xffffffu), (unsigned)(x >> 48) & 3u};
}

__global__ void __launch_bounds__(PARSE_THREADS)
parse_summary_kernel(const unsigned char *__restrict__ t, int64_t n, unsigned long long *__restrict__ tile_ws) {
    const int64_t i0 = (int64_t)blockIdx.x * MLBP_PARSE_TILE_BYTES + (int64_t)threadIdx.x * PARSE_SEG;
    Seg s = {0, 0, 2};
    if (i0 < n) s = seg_of(classify(t, n, i0));
    Seg total;
    block_scan<PARSE_THREADS>(s, &total);
    if (threadIdx.x == 0) tile_ws[blockIdx.x] = pack_seg(total);
}

// tile summaries -> absolute field index of each tile's first field (bits 0..62) and its entry comment state (bit 63)
__global__ void __launch_bounds__(PARSE_SCAN_THREADS)
parse_scan_kernel(unsigned long long *__restrict__ tile_ws, int n_tiles, unsigned long long *__restrict__ state) {
    const unsigned long long base = state[MLBP_PARSE_FIELDS];
    const int per = (n_tiles + PARSE_SCAN_THREADS - 1) / PARSE_SCAN_THREADS;
    const int t0 = min(n_tiles, (int)threadIdx.x * per), t1 = min(n_tiles, t0 + per);
    Seg mine = {0, 0, 2};
    for (int t = t0; t < t1; ++t) mine = compose(mine, unpack_seg(tile_ws[t]));
    Seg total;
    const Seg ex = block_scan<PARSE_SCAN_THREADS>(mine, &total);
    unsigned long long k = base + ex.a0;                      // a chunk starts at a line start: outside a comment
    unsigned c = ex.o & 1;
    for (int t = t0; t < t1; ++t) {
        const Seg s = unpack_seg(tile_ws[t]);
        tile_ws[t] = k | ((unsigned long long)c << 63);
        k += c ? s.a1 : s.a0;
        c = c ? (s.o >> 1) & 1 : s.o & 1;
    }
    __syncthreads();                                          // every thread has read state[MLBP_PARSE_FIELDS]
    if (threadIdx.x == 0) state[MLBP_PARSE_FIELDS] = base + total.a0;
}

// order-preserving map of float64 bits to unsigned integers (-0 sorts below +0)
__device__ __forceinline__ unsigned long long order_key(uint64_t b) { return (b >> 63) ? ~b : (b | F64_SIGN); }

__device__ __forceinline__ void record_error(unsigned long long *state, int64_t offset, int kind) {
    atomicMax(state + MLBP_PARSE_ERROR, ~(((unsigned long long)offset << 3) | (unsigned long long)kind));
}

__global__ void __launch_bounds__(PARSE_THREADS)
parse_write_kernel(const unsigned char *__restrict__ t, int64_t n, int64_t file_offset, int n_cols, int64_t max_rows,
                   float *__restrict__ out, int64_t ld_out, unsigned long long *__restrict__ state, int64_t *__restrict__ hard,
                   int hard_cap, const unsigned long long *__restrict__ tile_ws) {
    const int64_t i0 = (int64_t)blockIdx.x * MLBP_PARSE_TILE_BYTES + (int64_t)threadIdx.x * PARSE_SEG;
    SegBits b = {0, 0, 0, 0, false, true};
    if (i0 < n) b = classify(t, n, i0);
    Seg total;
    const Seg ex = block_scan<PARSE_THREADS>(i0 < n ? seg_of(b) : Seg{0, 0, 2}, &total);
    const unsigned long long tp = tile_ws[blockIdx.x];
    const unsigned tc = (unsigned)(tp >> 63);
    unsigned long long k = (tp & ~F64_SIGN) + (tc ? ex.a1 : ex.a0);
    const unsigned com = tc ? (ex.o >> 1) & 1 : ex.o & 1;
    unsigned fields = b.start & ~(com ? b.com1 : b.com0);
    if (b.bad) record_error(state, file_offset + i0 + __ffs(b.bad) - 1, MLBP_PARSE_ERR_BYTE);
    unsigned long long kmin = ~0ull, kmax = 0ull, nan_bits = 0ull;
    while (fields) {
        const int j = __ffs(fields) - 1;
        fields &= fields - 1;
        const int64_t i = i0 + j;
        int64_t e = i + 1;
        while (e < n && !ends_field(__ldg(t + e))) ++e;
        bool first = true;                                    // the first field of its line: only separators before it
        for (int64_t q = i - 1; q >= 0; --q) {
            const unsigned c = __ldg(t + q);
            if (c == '\n') break;
            if (!is_sep(c)) { first = false; break; }
        }
        const unsigned long long row = k / (unsigned)n_cols, col = k % (unsigned)n_cols;
        if (first != (col == 0)) record_error(state, file_offset + i, MLBP_PARSE_ERR_COLS);
        if (row >= (unsigned long long)max_rows) {
            record_error(state, file_offset + i, MLBP_PARSE_ERR_ROWS);
        } else {
            const Field f = parse_field(t + i, t + e);
            if (f.status == FIELD_BAD) {
                record_error(state, file_offset + i, MLBP_PARSE_ERR_FIELD);
            } else if (f.status == FIELD_HARD) {
                const unsigned long long slot = atomicAdd(state + MLBP_PARSE_HARD, 1ull);
                if (slot < (unsigned long long)hard_cap) {
                    hard[2 * slot] = file_offset + i;
                    hard[2 * slot + 1] = (int64_t)k;
                }
            } else {
                float x;
                if ((f.bits & ~F64_SIGN) > F64_INF) {            // NaN: numpy's cast keeps the sign, payload of the default NaN
                    x = __uint_as_float((unsigned)(f.bits >> 32) & 0x80000000u | 0x7fc00000u);
                    nan_bits |= (f.bits >> 63) ? 2ull : 1ull;
                } else {
                    x = __double2float_rn(__longlong_as_double((long long)f.bits));
                    const unsigned long long key = order_key(f.bits);
                    kmin = min(kmin, key);
                    kmax = max(kmax, key);
                }
                out[row * ld_out + col] = x;
            }
        }
        ++k;
    }
    // block min / max / NaN flags, one atomic each per CTA
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        kmin = min(kmin, __shfl_xor_sync(0xffffffffu, kmin, o));
        kmax = max(kmax, __shfl_xor_sync(0xffffffffu, kmax, o));
        nan_bits |= __shfl_xor_sync(0xffffffffu, nan_bits, o);
    }
    __shared__ unsigned long long red[3][PARSE_THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) { red[0][warp] = kmin; red[1][warp] = kmax; red[2][warp] = nan_bits; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < PARSE_THREADS / 32; ++w) {
            kmin = min(kmin, red[0][w]);
            kmax = max(kmax, red[1][w]);
            nan_bits |= red[2][w];
        }
        if (kmin != ~0ull) atomicMax(state + MLBP_PARSE_MIN, ~kmin);
        if (kmax != 0ull) atomicMax(state + MLBP_PARSE_MAX, kmax);
        if (nan_bits) atomicOr(state + MLBP_PARSE_NAN, nan_bits);
    }
}

}  // namespace mlbp

using namespace mlbp;

extern "C" int mlbp_parse_float_text(const char *text, int64_t n_bytes, int64_t file_offset, int n_cols, int64_t max_rows,
                                     float *out, int64_t ld_out, uint64_t *state, int64_t *hard, int hard_cap,
                                     uint64_t *tile_ws, void *stream) {
    MLBP_CHECK_ARG(state && n_bytes >= 0 && n_bytes <= MLBP_PARSE_MAX_CHUNK && file_offset >= 0 &&
                   file_offset < ((int64_t)1 << 56) && n_cols >= 1 && ld_out >= n_cols && max_rows >= 0 && hard_cap >= 0 &&
                   (hard || hard_cap == 0), "parse_float_text: bad argument");
    if (n_bytes == 0) return MLBP_OK;
    MLBP_CHECK_ARG(text && tile_ws && (out || max_rows == 0), "parse_float_text: null pointer");
    MLBP_CHECK_ARG(((uintptr_t)text & 15) == 0, "parse_float_text: text must be 16-byte aligned");
    cudaStream_t s = as_stream(stream);
    const int n_tiles = (int)((n_bytes + MLBP_PARSE_TILE_BYTES - 1) / MLBP_PARSE_TILE_BYTES);
    const unsigned char *t = reinterpret_cast<const unsigned char *>(text);
    auto *ws = reinterpret_cast<unsigned long long *>(tile_ws);
    auto *st = reinterpret_cast<unsigned long long *>(state);
    parse_summary_kernel<<<n_tiles, PARSE_THREADS, 0, s>>>(t, n_bytes, ws);
    MLBP_LAUNCH_CHECK();
    parse_scan_kernel<<<1, PARSE_SCAN_THREADS, 0, s>>>(ws, n_tiles, st);
    MLBP_LAUNCH_CHECK();
    parse_write_kernel<<<n_tiles, PARSE_THREADS, 0, s>>>(t, n_bytes, file_offset, n_cols, max_rows, out, ld_out, st, hard,
                                                         hard_cap, ws);
    MLBP_LAUNCH_CHECK();
    return MLBP_OK;
}
