// k_moments.cu -- reduction-only fast path of the BASIC group ("class M" rows of SURVEY.md section 8a):
// sum_values :371, mean :677, length :691, standard_deviation :705, variance :735, root_mean_square :783,
// maximum :2003, absolute_maximum :2017, minimum :2031, abs_energy :548, variation_coefficient :718,
// variance_larger_than_standard_deviation :239, large_standard_deviation :273, mean_change :624, skewness :749,
// kurtosis :766 (feature_calculators.py).
//
// When a plan's BASIC group holds nothing else (MinimalFCParameters: everything but the median), the descriptor
// interpreter of k_basic (shared-memory staging, lock-step walk, 250 KB of code) is replaced by this kernel: the
// series is streamed straight from HBM with 128-bit loads, EIGHT lanes per series (four series per warp, so a warp
// has 4 KB of loads in flight and the cross-lane reductions take 3 shuffle steps instead of 5), two passes (sums and
// extrema, then the centred moments -- the second pass hits L1), float64 accumulation.  The kernel is bound by HBM:
// algorithmic bytes per series = 4 n read + 8 per output column written.
#include <algorithm>

#include "tsfx_common.cuh"
#include "tsfx_kernels.h"

namespace tsfx {

bool moments_only_calc(int calc) {
    switch (calc) {
        case TSFX_VARIANCE_LARGER_THAN_STANDARD_DEVIATION: case TSFX_LARGE_STANDARD_DEVIATION: case TSFX_SUM_VALUES:
        case TSFX_ABS_ENERGY: case TSFX_MEAN: case TSFX_LENGTH: case TSFX_STANDARD_DEVIATION: case TSFX_VARIANCE:
        case TSFX_VARIATION_COEFFICIENT: case TSFX_ROOT_MEAN_SQUARE: case TSFX_MAXIMUM: case TSFX_MINIMUM:
        case TSFX_ABSOLUTE_MAXIMUM: case TSFX_MEAN_CHANGE: case TSFX_SKEWNESS: case TSFX_KURTOSIS:
        case TSFX_QUERY_SIMILARITY_COUNT: case TSFX_CONST_NAN:
            return true;
        default:
            return false;
    }
}

template <int SUB>
__device__ __forceinline__ double gsum(double v) {
#pragma unroll
    for (int o = SUB / 2; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}
template <int SUB>
__device__ __forceinline__ float gminf(float v) {
#pragma unroll
    for (int o = SUB / 2; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(FULL, v, o));
    return v;
}
template <int SUB>
__device__ __forceinline__ float gmaxf(float v) {
#pragma unroll
    for (int o = SUB / 2; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(FULL, v, o));
    return v;
}

struct MomStats { double n, sum, sumsq, mean, m2, m3, m4, var, sd, vmin, vmax, x0, xn1, rms, absmax, skew, kurt; };

// the square roots / divisions every column shares are formed ONCE per series by all lanes (uniform code); the
// per-descriptor pick below is then a couple of instructions per lane instead of a divergent walk through ten cases
__device__ __forceinline__ void moments_derive(MomStats& S, int need_high) {
    const double dn = S.n;
    S.var = S.m2 / dn;
    S.sd = sqrt(S.var);
    S.rms = sqrt(S.sumsq / dn);
    S.absmax = fmax(fabs(S.vmin), fabs(S.vmax));
    S.skew = dnan();
    S.kurt = dnan();
    if (need_high) {
        const int n = (int)dn;
        const double e1 = 2.220446049250313e-16 * S.absmax, e2 = e1 * e1;
        {   // pandas nanops.nanskew
            double m2 = S.m2, m3 = S.m3;
            if (fabs(m2) < e2 * dn) m2 = 0.0;
            if (fabs(m3) < e2 * e1 * dn) m3 = 0.0;
            if (n >= 3) S.skew = (m2 == 0.0) ? 0.0 : (dn * sqrt(dn - 1.0) / (dn - 2.0)) * (m3 / (m2 * sqrt(m2)));
        }
        {   // pandas nanops.nankurt
            double m2 = S.m2, m4 = S.m4;
            if (fabs(m2) < e2 * dn) m2 = 0.0;
            if (fabs(m4) < e2 * e2 * dn) m4 = 0.0;
            if (n >= 4) {
                const double adj = 3.0 * (dn - 1.0) * (dn - 1.0) / ((dn - 2.0) * (dn - 3.0));
                const double num = dn * (dn + 1.0) * (dn - 1.0) * m4;
                const double den = (dn - 2.0) * (dn - 3.0) * m2 * m2;
                S.kurt = (den == 0.0) ? 0.0 : num / den - adj;
            }
        }
    }
}

__device__ __forceinline__ double moments_value(const Desc& d, const MomStats& S) {
    const double dn = S.n;
    switch (d.calc) {
        case TSFX_VARIANCE_LARGER_THAN_STANDARD_DEVIATION: return (S.var > S.sd) ? 1.0 : 0.0;      // sd = sqrt(var)
        case TSFX_LARGE_STANDARD_DEVIATION: return (S.sd > d.p0 * (S.vmax - S.vmin)) ? 1.0 : 0.0;
        case TSFX_SUM_VALUES: return S.sum;
        case TSFX_ABS_ENERGY: return S.sumsq;
        case TSFX_MEAN: return S.mean;
        case TSFX_LENGTH: return dn;
        case TSFX_STANDARD_DEVIATION: return S.sd;
        case TSFX_VARIANCE: return S.var;
        case TSFX_VARIATION_COEFFICIENT: return (S.mean != 0.0) ? S.sd / S.mean : dnan();
        case TSFX_ROOT_MEAN_SQUARE: return S.rms;
        case TSFX_MAXIMUM: return S.vmax;
        case TSFX_MINIMUM: return S.vmin;
        case TSFX_ABSOLUTE_MAXIMUM: return S.absmax;
        case TSFX_MEAN_CHANGE: return dn > 1.0 ? (S.xn1 - S.x0) / (dn - 1.0) : dnan();
        case TSFX_SKEWNESS: return S.skew;
        case TSFX_KURTOSIS: return S.kurt;
        default: return dnan();       // query_similarity_count (default query=None), constant-NaN columns
    }
}

// REG = 8: series of up to 8 * SUB * 4 = 256 samples whose start is 16-byte aligned stay in registers between the two
// passes (one 128-bit load per chunk, issued back to back so a warp keeps 4 KB in flight); longer or unaligned series
// re-read the second pass from L1 / L2.
template <int SUB, int WPC, int REG>
__global__ void __launch_bounds__(WPC * 32, 3) k_moments(MomentsArgs A) {
    constexpr int SPW = 32 / SUB;                    // series per warp
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int sub = lane % SUB, slot = lane / SUB;
    const int64_t stride = (int64_t)gridDim.x * WPC * SPW;
    const int64_t first = ((int64_t)blockIdx.x * WPC + warp) * SPW;
    // every lane of a warp runs the same number of trips (shuffles below use the full mask)
    for (int64_t s0 = first; s0 < A.R.n_series; s0 += stride) {
        const int64_t s = s0 + slot;
        const bool live = s < A.R.n_series;
        int64_t b = 0;
        int n = 0;
        if (live) {
            if (A.R.begin) { b = A.R.begin[s]; n = A.R.len[s]; } else { b = s * (int64_t)A.R.dense_len; n = A.R.dense_len; }
        }
        const float* src = A.R.values + b;
        const bool vec = ((uintptr_t)src & 15u) == 0;
        const int n4 = vec ? (n >> 2) : 0;
        const float4* s4 = reinterpret_cast<const float4*>(src);
        const bool inreg = n4 <= REG * SUB;
        float4 v[REG];
        // ---- pass 1: sum, sum of squares, extrema
        double sm = 0.0, sq = 0.0;
        float lo = INFINITY, hi = -INFINITY;
        if (inreg) {
#pragma unroll
            for (int k = 0; k < REG; ++k) {
                const int c = sub + k * SUB;
                v[k] = (c < n4) ? __ldcs(s4 + c) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int k = 0; k < REG; ++k) {
                const int c = sub + k * SUB;
                if (c < n4) {
                    const double a = (double)v[k].x, bb = (double)v[k].y, cc = (double)v[k].z, dd = (double)v[k].w;
                    sm += (a + bb) + (cc + dd);
                    sq = fma(a, a, sq); sq = fma(bb, bb, sq); sq = fma(cc, cc, sq); sq = fma(dd, dd, sq);
                    lo = fminf(fminf(lo, v[k].x), fminf(v[k].y, fminf(v[k].z, v[k].w)));
                    hi = fmaxf(fmaxf(hi, v[k].x), fmaxf(v[k].y, fmaxf(v[k].z, v[k].w)));
                }
            }
        } else {
#pragma unroll 8
            for (int c = sub; c < n4; c += SUB) {
                const float4 w = __ldg(s4 + c);
                const double a = (double)w.x, bb = (double)w.y, cc = (double)w.z, dd = (double)w.w;
                sm += (a + bb) + (cc + dd);
                sq = fma(a, a, sq); sq = fma(bb, bb, sq); sq = fma(cc, cc, sq); sq = fma(dd, dd, sq);
                lo = fminf(fminf(lo, w.x), fminf(w.y, fminf(w.z, w.w)));
                hi = fmaxf(fmaxf(hi, w.x), fmaxf(w.y, fmaxf(w.z, w.w)));
            }
        }
        for (int i = (n4 << 2) + sub; i < n; i += SUB) {
            const float f = __ldg(src + i);
            const double a = (double)f;
            sm += a;
            sq = fma(a, a, sq);
            lo = fminf(lo, f);
            hi = fmaxf(hi, f);
        }
        MomStats S;
        S.n = (double)n;
        S.sum = gsum<SUB>(sm);
        S.sumsq = gsum<SUB>(sq);
        S.vmin = (double)gminf<SUB>(lo);
        S.vmax = (double)gmaxf<SUB>(hi);
        S.mean = S.sum / S.n;
        // ---- pass 2: centred moments
        double a2 = 0.0, a3 = 0.0, a4 = 0.0;
        const double mu = S.mean;
        auto centred = [&](const float4& w) {
            const double d0 = (double)w.x - mu, d1 = (double)w.y - mu, d2 = (double)w.z - mu, d3 = (double)w.w - mu;
            const double q0 = d0 * d0, q1 = d1 * d1, q2 = d2 * d2, q3 = d3 * d3;
            a2 += (q0 + q1) + (q2 + q3);
            if (A.need_high) {
                a3 = fma(q0, d0, a3); a3 = fma(q1, d1, a3); a3 = fma(q2, d2, a3); a3 = fma(q3, d3, a3);
                a4 = fma(q0, q0, a4); a4 = fma(q1, q1, a4); a4 = fma(q2, q2, a4); a4 = fma(q3, q3, a4);
            }
        };
        if (inreg) {
#pragma unroll
            for (int k = 0; k < REG; ++k)
                if (sub + k * SUB < n4) centred(v[k]);
        } else {
#pragma unroll 8
            for (int c = sub; c < n4; c += SUB) centred(__ldg(s4 + c));
        }
        for (int i = (n4 << 2) + sub; i < n; i += SUB) {
            const double d = (double)__ldg(src + i) - mu;
            const double q = d * d;
            a2 += q;
            a3 = fma(q, d, a3);
            a4 = fma(q, q, a4);
        }
        S.m2 = gsum<SUB>(a2);
        S.m3 = A.need_high ? gsum<SUB>(a3) : 0.0;
        S.m4 = A.need_high ? gsum<SUB>(a4) : 0.0;
        S.x0 = (live && n > 0) ? (double)__ldg(src) : 0.0;
        S.xn1 = (live && n > 0) ? (double)__ldg(src + n - 1) : 0.0;
        moments_derive(S, A.need_high);
        if (live) {
            double* orow = A.out + (size_t)s * A.ncols;
            for (int j = sub; j < A.nd; j += SUB) {
                const Desc d = A.descs[j];
                __stcs(orow + (A.colmap ? A.colmap[j] : d.col), moments_value(d, S));
            }
        }
    }
}

// Dense, 16-byte aligned series of at most REG * SUB * 4 samples (the BASELINE shapes): same arithmetic, but the loads of
// the NEXT series are issued before the current one is reduced (register double buffer), so every warp always has 4 KB
// of HBM reads in flight -- the kernel's only job is to keep the memory system busy.
template <int SUB, int WPC, int REG>
__global__ void __launch_bounds__(WPC * 32, 2) k_moments_dense(MomentsArgs A) {
    constexpr int SPW = 32 / SUB;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int sub = lane % SUB, slot = lane / SUB;
    const int64_t stride = (int64_t)gridDim.x * WPC * SPW;
    const int n = A.R.dense_len, n4 = n >> 2;
    float4 cur[REG], nxt[REG];
    auto fetch = [&](float4 (&dst)[REG], int64_t s) {
        const float4* s4 = reinterpret_cast<const float4*>(A.R.values + s * (int64_t)n);
#pragma unroll
        for (int k = 0; k < REG; ++k) {
            const int c = sub + k * SUB;
            dst[k] = (c < n4 && s < A.R.n_series) ? __ldcs(s4 + c) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    };
    int64_t s0 = ((int64_t)blockIdx.x * WPC + warp) * SPW;
    fetch(cur, s0 + slot);
    for (; s0 < A.R.n_series; s0 += stride) {
        const int64_t s = s0 + slot;
        const bool live = s < A.R.n_series;
        fetch(nxt, s + stride);                          // in flight while this series is reduced
        // four independent accumulators per sum: a single fma chain over the lane's 32 samples would be 32 dependent
        // FP64 operations (the kernel was bound by exactly that: stall "wait" 2.9 per issued instruction)
        double sm4[4] = {0.0, 0.0, 0.0, 0.0}, sq4[4] = {0.0, 0.0, 0.0, 0.0};
        float lo = INFINITY, hi = -INFINITY;
#pragma unroll
        for (int k = 0; k < REG; ++k) {
            if (sub + k * SUB < n4) {
                const double a = (double)cur[k].x, bb = (double)cur[k].y, cc = (double)cur[k].z, dd = (double)cur[k].w;
                sm4[0] += a; sm4[1] += bb; sm4[2] += cc; sm4[3] += dd;
                sq4[0] = fma(a, a, sq4[0]); sq4[1] = fma(bb, bb, sq4[1]); sq4[2] = fma(cc, cc, sq4[2]); sq4[3] = fma(dd, dd, sq4[3]);
                lo = fminf(fminf(lo, cur[k].x), fminf(cur[k].y, fminf(cur[k].z, cur[k].w)));
                hi = fmaxf(fmaxf(hi, cur[k].x), fmaxf(cur[k].y, fmaxf(cur[k].z, cur[k].w)));
            }
        }
        const double sm = (sm4[0] + sm4[1]) + (sm4[2] + sm4[3]), sq = (sq4[0] + sq4[1]) + (sq4[2] + sq4[3]);
        MomStats S;
        S.n = (double)n;
        S.sum = gsum<SUB>(sm);
        S.sumsq = gsum<SUB>(sq);
        S.vmin = (double)gminf<SUB>(lo);
        S.vmax = (double)gmaxf<SUB>(hi);
        S.mean = S.sum / S.n;
        const double mu = S.mean;
        double b2[4] = {0.0, 0.0, 0.0, 0.0}, b3[4] = {0.0, 0.0, 0.0, 0.0}, b4[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
        for (int k = 0; k < REG; ++k) {
            if (sub + k * SUB < n4) {
                const double d0 = (double)cur[k].x - mu, d1 = (double)cur[k].y - mu, d2 = (double)cur[k].z - mu, d3 = (double)cur[k].w - mu;
                const double q0 = d0 * d0, q1 = d1 * d1, q2 = d2 * d2, q3 = d3 * d3;
                b2[0] += q0; b2[1] += q1; b2[2] += q2; b2[3] += q3;
                if (A.need_high) {
                    b3[0] = fma(q0, d0, b3[0]); b3[1] = fma(q1, d1, b3[1]); b3[2] = fma(q2, d2, b3[2]); b3[3] = fma(q3, d3, b3[3]);
                    b4[0] = fma(q0, q0, b4[0]); b4[1] = fma(q1, q1, b4[1]); b4[2] = fma(q2, q2, b4[2]); b4[3] = fma(q3, q3, b4[3]);
                }
            }
        }
        const double a2 = (b2[0] + b2[1]) + (b2[2] + b2[3]), a3 = (b3[0] + b3[1]) + (b3[2] + b3[3]), a4 = (b4[0] + b4[1]) + (b4[2] + b4[3]);
        S.m2 = gsum<SUB>(a2);
        S.m3 = A.need_high ? gsum<SUB>(a3) : 0.0;
        S.m4 = A.need_high ? gsum<SUB>(a4) : 0.0;
        // first / last sample: lane `sub == 0` holds x[0] in its first chunk; x[n-1] sits in chunk n4 - 1
        const int lastc = n4 - 1, lk = lastc / SUB, lsub = lastc % SUB;
        float xl = 0.f;
#pragma unroll
        for (int k = 0; k < REG; ++k) if (k == lk) xl = cur[k].w;
        S.x0 = (double)__shfl_sync(FULL, cur[0].x, slot * SUB);
        S.xn1 = (double)__shfl_sync(FULL, xl, slot * SUB + lsub);
        moments_derive(S, A.need_high);
        if (live) {
            double* orow = A.out + (size_t)s * A.ncols;
            for (int j = sub; j < A.nd; j += SUB) {
                const Desc d = A.descs[j];
                __stcs(orow + (A.colmap ? A.colmap[j] : d.col), moments_value(d, S));
            }
        }
#pragma unroll
        for (int k = 0; k < REG; ++k) cur[k] = nxt[k];
    }
}

cudaError_t launch_moments(const MomentsArgs& A, cudaStream_t st, int sm_count) {
    constexpr int SUB = 8, WPC = 8;
    const int64_t per_cta = (int64_t)WPC * (32 / SUB);
    int64_t ctas = (A.R.n_series + per_cta - 1) / per_cta;
    const int64_t cap = (int64_t)sm_count * 8 * 8;
    if (ctas > cap) ctas = cap;
    if (ctas < 1) ctas = 1;
    const bool dense = A.R.begin == nullptr && (A.R.dense_len & 3) == 0 && A.R.dense_len >= 4 && A.R.dense_len <= 8 * SUB * 4 &&
                       ((uintptr_t)A.R.values & 15u) == 0;
    if (dense) {
        const int64_t cap2 = (int64_t)sm_count * 2;          // persistent: two CTAs per SM, prefetching
        int64_t c2 = (A.R.n_series + per_cta - 1) / per_cta;
        if (c2 > cap2) c2 = cap2;
        k_moments_dense<SUB, WPC, 8><<<(int)c2, WPC * 32, 0, st>>>(A);
        return cudaGetLastError();
    }
    k_moments<SUB, WPC, 8><<<(int)ctas, WPC * 32, 0, st>>>(A);
    return cudaGetLastError();
}

}  // namespace tsfx
