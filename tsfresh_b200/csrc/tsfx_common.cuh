// tsfx_common.cuh -- shared device infrastructure for the per-series warp kernels (sm_100a).
//
// Execution model: ONE WARP PER SERIES.  The series (float32, as ingested) is staged once into shared
// memory; every calculator of a kernel group is then evaluated from that copy and from a small set of
// shared intermediates (moments, centred copy, sorted copy, spectrum ...).  All arithmetic is float64.
// Every lane of the warp executes every statement (descriptors are warp-uniform), so *_sync intrinsics
// always use the full mask.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>
#include "../../include/tsfx.h"

#define FULL 0xffffffffu
#define TSFX_WARP 32

namespace tsfx {

typedef tsfx_feature_desc Desc;

struct SeriesRef {              // how a kernel finds its series
    const float* values;
    const int64_t* begin;       // nullptr => dense: begin = s * dense_len
    const int32_t* len;         // nullptr => dense
    int32_t dense_len;
    int64_t n_series;
    const int64_t* times = nullptr;   // optional: timestamp (ns) of every row of `values` (linear_trend_timewise)
};

__device__ __forceinline__ double dnan() { return __longlong_as_double(0x7ff8000000000000LL); }
__device__ __forceinline__ double dinf() { return __longlong_as_double(0x7ff0000000000000LL); }

// ---------------------------------------------------------------- warp reductions (result in all lanes)
__device__ __forceinline__ double wsum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}
__device__ __forceinline__ double wmax(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(FULL, v, o));
    return v;
}
__device__ __forceinline__ double wmin(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(FULL, v, o));
    return v;
}
__device__ __forceinline__ float wmaxf(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(FULL, v, o));
    return v;
}
__device__ __forceinline__ float wminf(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(FULL, v, o));
    return v;
}
__device__ __forceinline__ int wsumi(int v) { return __reduce_add_sync(FULL, v); }
__device__ __forceinline__ int wmaxi(int v) { return __reduce_max_sync(FULL, v); }
__device__ __forceinline__ int wmini(int v) { return __reduce_min_sync(FULL, v); }

// count of lanes (x tiles) where pred holds; every lane must call with its own predicate
__device__ __forceinline__ int wcount(bool pred) { return __popc(__ballot_sync(FULL, pred)); }

// ---------------------------------------------------------------- per-warp working region
// Normally a slice of the CTA's dynamic shared memory.  Series too long for that (bytes_per_warp > 227 KB) run
// with the same carve-up in a global-memory scratch buffer (L2-resident; slower, but every length works).
// (compile-time switch: the shared-memory instantiation keeps pure shared-space addressing)
template <bool GLOBAL_SCRATCH>
__device__ __forceinline__ unsigned char* warp_region(unsigned char* smem_raw, unsigned char* gscratch, int bytes_per_warp,
                                                      int wpc, int warp) {
    if (GLOBAL_SCRATCH) return gscratch + ((size_t)blockIdx.x * wpc + warp) * (size_t)bytes_per_warp;
    return smem_raw + (size_t)warp * bytes_per_warp;
}

// ---------------------------------------------------------------- series staging
// Loads series s into shared memory xs[0..n) (coalesced; 128-bit loads when the start is 16B aligned).
__device__ __forceinline__ int load_series(const SeriesRef& R, int64_t s, float* xs, int lane) {
    int64_t b;
    int n;
    if (R.begin) { b = R.begin[s]; n = R.len[s]; } else { b = s * (int64_t)R.dense_len; n = R.dense_len; }
    const float* src = R.values + b;
    if (((((uintptr_t)src) | ((uintptr_t)xs)) & 15u) == 0) {
        const float4* s4 = reinterpret_cast<const float4*>(src);
        int n4 = n >> 2;
        for (int i = lane; i < n4; i += 32) {
            float4 v = __ldg(s4 + i);
            reinterpret_cast<float4*>(xs)[i] = v;
        }
        for (int i = (n4 << 2) + lane; i < n; i += 32) xs[i] = __ldg(src + i);
    } else {
        for (int i = lane; i < n; i += 32) xs[i] = __ldg(src + i);
    }
    __syncwarp();
    return n;
}

// ---------------------------------------------------------------- first/second moment block
struct Moments {
    int n;
    double sum, mean, sumsq, m2, var, sd;   // m2 = sum (x-mean)^2 ; var = m2/n (ddof 0)
    double vmin, vmax;
};

// Pass 1 + centred pass.  Optionally writes the centred copy xc[i] = x[i] - mean (float64).
__device__ __forceinline__ Moments moments(const float* xs, int n, double* xc, int lane) {
    Moments M;
    M.n = n;
    double s = 0.0, q = 0.0;
    float lo = INFINITY, hi = -INFINITY;
    for (int i = lane; i < n; i += 32) {
        float f = xs[i];
        double v = (double)f;
        s += v;
        q = fma(v, v, q);
        lo = fminf(lo, f);
        hi = fmaxf(hi, f);
    }
    M.sum = wsum(s);
    M.sumsq = wsum(q);
    M.vmin = (double)wminf(lo);
    M.vmax = (double)wmaxf(hi);
    M.mean = M.sum / (double)n;
    double a = 0.0;
    for (int i = lane; i < n; i += 32) {
        double d = (double)xs[i] - M.mean;
        if (xc) xc[i] = d;
        a = fma(d, d, a);
    }
    M.m2 = wsum(a);
    M.var = M.m2 / (double)n;
    M.sd = sqrt(M.var);
    if (xc) __syncwarp();
    return M;
}

}  // namespace tsfx
