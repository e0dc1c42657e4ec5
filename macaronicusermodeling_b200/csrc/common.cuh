// Shared helpers for libmlbp.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>

#include "../../include/mlbp.h"

namespace mlbp {

void set_error(const char *fmt, ...);

#define MLBP_CHECK_ARG(cond, ...)                       \
    do {                                                \
        if (!(cond)) {                                  \
            ::mlbp::set_error(__VA_ARGS__);             \
            return MLBP_ERR_INVALID;                    \
        }                                               \
    } while (0)

#define MLBP_CUDA(call)                                                                        \
    do {                                                                                       \
        cudaError_t e_ = (call);                                                               \
        if (e_ != cudaSuccess) {                                                               \
            ::mlbp::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
            return MLBP_ERR_CUDA;                                                              \
        }                                                                                      \
    } while (0)

#define MLBP_LAUNCH_CHECK() MLBP_CUDA(cudaGetLastError())

static inline cudaStream_t as_stream(void *s) { return reinterpret_cast<cudaStream_t>(s); }

constexpr int MLBP_MAX_DEVICES = 64;   // per-device caches of function attributes / occupancy (one process may drive several GPUs)
static inline int current_device() {
    int d = 0;
    return (cudaGetDevice(&d) == cudaSuccess && d >= 0 && d < MLBP_MAX_DEVICES) ? d : 0;
}

// x (already scaled into fp16 range) -> hi + lo, both fp16; hi + lo == x to ~2^-22 relative.
__device__ __forceinline__ void split_f16(float x, __half &hi, __half &lo) {
    hi = __float2half_rn(x);
    lo = __float2half_rn(x - __half2float(hi));
}

// Compensated fp32 arithmetic of the table entries exp(theta . phi) (K2, K10): ~1 ulp of fp32 per entry without a float64
// instruction per element.
struct F2 { float hi, lo; };                                      // unevaluated sum hi + lo

__host__ __device__ __forceinline__ F2 split_double(double x) {
    F2 r;
    r.hi = (float)x;
    r.lo = (float)(x - (double)r.hi);
    return r;
}
// c * p + b with c = (c.hi + c.lo), b = (b.hi + b.lo), p an fp32 datum: result as hi + lo (error ~2^-46 relative)
__device__ __forceinline__ F2 axpb(F2 c, float p, F2 b) {
    const float ph = c.hi * p;
    const float pe = fmaf(c.hi, p, -ph);                          // exact product error
    const float s = ph + b.hi;
    const float bb = s - ph;
    const float se = (ph - (s - bb)) + (b.hi - bb);               // exact sum error (two-sum)
    F2 r;
    r.hi = s;
    r.lo = se + pe + fmaf(c.lo, p, b.lo);
    return r;
}
// exp(z.hi + z.lo), ~1 ulp: expf is IEEE-grade here (the library is built without fast-math)
__device__ __forceinline__ float exp_f2(F2 z) { return expf(z.hi) * (1.0f + z.lo); }

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ float warp_sum_f32(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_sum_t(float v) { return warp_sum_f32(v); }
__device__ __forceinline__ double warp_sum_t(double v) { return warp_sum(v); }

// Block-wide sum of one double per thread; result valid in every thread. `red` : >= 32 doubles of shared memory.
__device__ __forceinline__ double block_sum(double v, double *red) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    v = warp_sum(v);
    __syncthreads();
    if (lane == 0) red[warp] = v;
    __syncthreads();
    double t = (lane < nw) ? red[lane] : 0.0;
    t = warp_sum(t);
    return t;
}

}  // namespace mlbp
