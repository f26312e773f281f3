// k_basic.cu -- kernel group BASIC: moments / extrema / counts / order-dependent streams.
//
// One warp per series.  Shared memory per warp: xs[npad] float32 (the series as ingested),
// xc[nxc] float64 (centred copy x - mean with a zero tail for the tiled lag products), scr[nscr] float64
// (scratch: chunk aggregates, histograms, cumulative masses, peak radii), lagS[nlag] float64 (lag products, pacf),
// ST[32] (shared statistics read by the lane-parallel finishers), altS[6 nalt] (regression sums per
// agg_linear_trend key); in front of the per-warp regions one CTA-wide copy of the descriptor table.  Two CTAs of 12
// warps per SM walk the descriptor list in lock step (instruction-cache sharing); the 41 lag products run on the FP64
// tensor cores (lag_products_dmma).  Calculators restated (feature_calculators.py line numbers in
// include/tsfx.h): every "class M" and "class O" row of SURVEY.md section 8a, plus linear_trend_timewise.
#include "tsfx_common.cuh"
#include "tsfx_math.cuh"
#include "tsfx_kernels.h"
#include <algorithm>

namespace tsfx {

struct Extra {
    double m3, m4;            // sum (x-mean)^3, ^4
    int cnt_above, cnt_below; // x > mean, x < mean
    int cnt_min, cnt_max, first_min, last_min, first_max, last_max;
    double sad, ssd;          // sum |dx|, sum dx^2
    int strike_above, strike_below;
};

struct Run { int len, pre, suf, best; };

__device__ __forceinline__ Run run_of_word(unsigned w, int bits) {
    // `bits` valid low bits (bits beyond are zero)
    Run r;
    r.len = bits;
    if (bits == 0) { r.pre = r.suf = r.best = 0; return r; }
    unsigned full = (bits == 32) ? 0xffffffffu : ((1u << bits) - 1u);
    if (w == full) { r.pre = r.suf = r.best = bits; return r; }
    r.pre = __ffs(~w) - 1;
    unsigned top = w << (32 - bits);                 // align the valid bits to the top
    r.suf = __clz(~top);
    int b = 0;
    unsigned t = w;
    while (t) { t &= (t << 1); ++b; }
    r.best = b;
    return r;
}
__device__ __forceinline__ Run run_combine(const Run& a, const Run& b) {
    Run r;
    r.len = a.len + b.len;
    r.pre = (a.pre == a.len) ? a.len + b.pre : a.pre;
    r.suf = (b.suf == b.len) ? b.len + a.suf : b.suf;
    r.best = max(max(a.best, b.best), a.suf + b.pre);
    return r;
}
// longest run of set bits over per-lane words (lane 0 first); result valid in all lanes
__device__ __forceinline__ Run run_warp(Run r) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        Run other;
        other.len = __shfl_down_sync(FULL, r.len, o);
        other.pre = __shfl_down_sync(FULL, r.pre, o);
        other.suf = __shfl_down_sync(FULL, r.suf, o);
        other.best = __shfl_down_sync(FULL, r.best, o);
        int lane = threadIdx.x & 31;
        if (lane + o < 32) r = run_combine(r, other);
    }
    Run out;
    out.len = __shfl_sync(FULL, r.len, 0);
    out.pre = __shfl_sync(FULL, r.pre, 0);
    out.suf = __shfl_sync(FULL, r.suf, 0);
    out.best = __shfl_sync(FULL, r.best, 0);
    return out;
}

__device__ __forceinline__ Extra extra_pass(const float* xs, const double* xc, int n, const Moments& M, int lane) {
    Extra E;
    double a3 = 0.0, a4 = 0.0, sad = 0.0, ssd = 0.0;
    int ca = 0, cb = 0, cmin = 0, cmax = 0;
    int fmin_i = 0x7fffffff, lmin_i = -1, fmax_i = 0x7fffffff, lmax_i = -1;
    const float fl = (float)M.vmin, fh = (float)M.vmax;
    Run ra = {0, 0, 0, 0}, rb = {0, 0, 0, 0};
    Run acc_a = {0, 0, 0, 0}, acc_b = {0, 0, 0, 0};
    unsigned wa = 0, wb = 0;
    int wbits = 0;
    int tile = 0;
    for (int base = 0; base < n; base += 32, ++tile) {
        int i = base + lane;
        bool ok = i < n;
        double d = ok ? xc[i] : 0.0;
        float f = ok ? xs[i] : 0.f;
        double d2 = d * d;
        a3 = fma(d2, d, a3);
        a4 = fma(d2, d2, a4);
        bool above = ok && d > 0.0, below = ok && d < 0.0;
        unsigned ma = __ballot_sync(FULL, above), mb = __ballot_sync(FULL, below);
        ca += __popc(ma);
        cb += __popc(mb);
        if ((tile & 31) == lane) { wa = ma; wb = mb; wbits = min(32, n - base); }
        if (ok && f == fl) { ++cmin; fmin_i = min(fmin_i, i); lmin_i = i; }
        if (ok && f == fh) { ++cmax; fmax_i = min(fmax_i, i); lmax_i = i; }
        if (i + 1 < n) {
            double dx = (double)xs[i + 1] - (double)f;
            sad += fabs(dx);
            ssd = fma(dx, dx, ssd);
        }
        if ((tile & 31) == 31 || base + 32 >= n) {      // flush a super-tile of up to 32 words
            ra = run_warp(run_of_word(wa, wbits));
            rb = run_warp(run_of_word(wb, wbits));
            acc_a = run_combine(acc_a, ra);
            acc_b = run_combine(acc_b, rb);
            wa = wb = 0; wbits = 0;
        }
    }
    E.m3 = wsum(a3);
    E.m4 = wsum(a4);
    E.sad = wsum(sad);
    E.ssd = wsum(ssd);
    E.cnt_above = ca;
    E.cnt_below = cb;
    E.cnt_min = wsumi(cmin);
    E.cnt_max = wsumi(cmax);
    E.first_min = wmini(fmin_i);
    E.last_min = wmaxi(lmin_i);
    E.first_max = wmini(fmax_i);
    E.last_max = wmaxi(lmax_i);
    E.strike_above = acc_a.best;
    E.strike_below = acc_b.best;
    return E;
}

// lagS[k] = sum_{t < n-k} xc[t] * xc[t+k], k = 0..kmax.  xc is zero beyond n (up to a whole 256-sample chunk plus the
// largest lag), so no bounds tests: each lane keeps 8 centred samples of a chunk in registers and every lag costs
// one load + one FMA per sample plus one warp sum.
__device__ __forceinline__ void lag_products(const double* xc, int n, int kmax, double* lagS, int lane) {
    for (int i0 = 0; i0 < n; i0 += 256) {
        double xr[8];
        const double* xb = xc + i0 + lane;
#pragma unroll
        for (int m = 0; m < 8; ++m) xr[m] = xb[32 * m];
        for (int k = 0; k <= kmax; ++k) {
            double a = 0.0;
#pragma unroll
            for (int m = 0; m < 8; ++m) a = fma(xr[m], xb[32 * m + k], a);
            a = wsum(a);
            if (lane == 0) lagS[k] = (i0 == 0) ? a : lagS[k] + a;
        }
    }
}

// The same lag products on the FP64 tensor cores (mma.sync m8n8k4, DMMA) -- the one GEMM-shaped piece of the path
// (BASELINE.json north_star).  With A[i][u] = xc[8 (b + u) + i] and B[u][j] = xc[8 (b + t + u) + j] (b = sample block,
// t = tile) the accumulator D_t[i][j] = sum_b,u A B collects x[s] x[s + 8 t + j - i] over all s = i mod 8: tile t
// holds lags 8 t - 7 .. 8 t + 7 on its diagonals, every (lag, residue) pair lands in exactly one tile, and
// lagS[k] = sum of the diagonal j - i = k - 8 t over the tiles.  Both fragments are the same strided view of xc
// (zero beyond n), so one shared-memory load feeds each MMA: per series ~8 loads + 6 MMAs per 32 samples and one
// diagonal fold per tile, instead of 41 x (8 loads + 8 FMAs + a warp sum) per 256 samples.
__device__ __forceinline__ void dmma_884(double& d0, double& d1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
                 : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}
#define TSFX_DMMA_MAX_TILES 8
__device__ __forceinline__ void lag_products_dmma(const double* xc, int n, int kmax, int ntiles, double* lagS, double* tile,
                                                  int lane) {
    double acc[TSFX_DMMA_MAX_TILES][2];
#pragma unroll
    for (int t = 0; t < TSFX_DMMA_MAX_TILES; ++t) { acc[t][0] = 0.0; acc[t][1] = 0.0; }
    const int li = lane >> 2, lu = lane & 3;
    const int G = (n + 31) >> 5;                          // groups of 4 sample blocks (32 samples)
    const double* xl = xc + 8 * lu + li;
    for (int g = 0; g < G; ++g) {
        const double a = xl[32 * g];
#pragma unroll
        for (int t = 0; t < TSFX_DMMA_MAX_TILES; ++t)
            if (t < ntiles) dmma_884(acc[t][0], acc[t][1], a, xl[32 * g + 8 * t]);
    }
    for (int k = lane; k <= kmax; k += 32) lagS[k] = 0.0;
    __syncwarp();
#pragma unroll
    for (int t = 0; t < TSFX_DMMA_MAX_TILES; ++t) {
        if (t < ntiles) {
            tile[li * 8 + 2 * lu] = acc[t][0];            // D[i][j]: i = lane / 4, j = 2 (lane % 4) + {0, 1}
            tile[li * 8 + 2 * lu + 1] = acc[t][1];
            __syncwarp();
            if (lane < 15) {
                const int d = lane - 7, k = 8 * t + d;    // diagonal j - i = d of tile t = lag k
                if (k >= 0 && k <= kmax) {
                    double sum = 0.0;
#pragma unroll
                    for (int i = 0; i < 8; ++i) { const int j = i + d; if (j >= 0 && j < 8) sum += tile[i * 8 + j]; }
                    lagS[k] += sum;
                }
            }
            __syncwarp();
        }
    }
}

// numpy histogram bin index for uniform bins (numpy/lib/_histograms_impl.py fast path)
__device__ __forceinline__ int hist_bin(double v, double first, double last, double denom, double step, int nb) {
    double f = __dmul_rn(__ddiv_rn(__dsub_rn(v, first), denom), (double)nb);
    int idx = (int)f;
    if (idx == nb) idx -= 1;
    // edge(i) = i*step + first, edge(nb) = last  (np.linspace)
    double e_lo = (idx == nb) ? last : __dadd_rn(__dmul_rn((double)idx, step), first);
    if (v < e_lo) idx -= 1;
    double e_hi = (idx + 1 == nb) ? last : __dadd_rn(__dmul_rn((double)(idx + 1), step), first);
    if (v >= e_hi && idx != nb - 1) idx += 1;
    return idx;
}

// -sum p ln p of an int histogram in shared memory (hist[0..nb)), total count n
__device__ __forceinline__ double hist_entropy(const int* hist, int nb, int n, int lane) {
    double a = 0.0;
    for (int b = lane; b < nb; b += 32) {
        int c = hist[b];
        if (c > 0) {
            double p = (double)c / (double)n;
            a += p * log(p);
        }
    }
    return -wsum(a);
}

// binned entropy of `cnt` values produced by f(i) (np.histogram(x, bins) -> -sum p ln p)
template <typename F>
__device__ __forceinline__ double binned_entropy_of(F val, int cnt, double vmin, double vmax, int nb,
                                                    int* hist, int lane) {
    double first = vmin, last = vmax;
    if (first == last) { first -= 0.5; last += 0.5; }
    double denom = __dsub_rn(last, first);
    double step = __ddiv_rn(denom, (double)nb);
    for (int b = lane; b < nb; b += 32) hist[b] = 0;
    __syncwarp();
    for (int i = lane; i < cnt; i += 32) {
        int idx = hist_bin(val(i), first, last, denom, step, nb);
        atomicAdd(&hist[idx], 1);
    }
    __syncwarp();
    double h = hist_entropy(hist, nb, cnt, lane);
    __syncwarp();
    return h;
}

__device__ __forceinline__ double agg_chunk(const float* xs, int lo, int hi, int f_agg) {
    // ndarray.max/min/mean/var/std/median over xs[lo:hi) by one lane (_aggregate_on_chunks :176-193)
    int c = hi - lo;
    if (f_agg == TSFX_AGG_MAX) { float m = xs[lo]; for (int i = lo + 1; i < hi; ++i) m = fmaxf(m, xs[i]); return (double)m; }
    if (f_agg == TSFX_AGG_MIN) { float m = xs[lo]; for (int i = lo + 1; i < hi; ++i) m = fminf(m, xs[i]); return (double)m; }
    double s = 0.0;
    for (int i = lo; i < hi; ++i) s += (double)xs[i];
    double mu = s / (double)c;
    if (f_agg == TSFX_AGG_MEAN) return mu;
    if (f_agg == TSFX_AGG_MEDIAN) {
        // rank selection without modifying the data (chunks are short)
        int k1 = (c - 1) / 2, k2 = c / 2;
        double v1 = 0.0, v2 = 0.0;
        for (int i = lo; i < hi; ++i) {
            float xi = xs[i];
            int r = 0;
            for (int j = lo; j < hi; ++j) r += (xs[j] < xi) || (xs[j] == xi && j < i);
            if (r == k1) v1 = (double)xi;
            if (r == k2) v2 = (double)xi;
        }
        return 0.5 * (v1 + v2);
    }
    double q = 0.0;
    for (int i = lo; i < hi; ++i) { double d = (double)xs[i] - mu; q = fma(d, d, q); }
    double v = q / (double)c;
    return f_agg == TSFX_AGG_STD ? sqrt(v) : v;
}

// the inputs of linregress(range(k), y[0..k)) with y in shared memory: k, mean(t), mean(y), ssxm, ssym, ssxym
struct LinSums { double k, tm, ym, sxx, syy, sxy; };
__device__ __forceinline__ LinSums linreg_sums(const double* y, int k, int lane) {
    double s = 0.0;
    for (int i = lane; i < k; i += 32) s += y[i];
    LinSums L;
    L.k = (double)k;
    L.ym = wsum(s) / (double)k;
    L.tm = 0.5 * (double)(k - 1);
    double sxx = 0.0, syy = 0.0, sxy = 0.0;
    for (int i = lane; i < k; i += 32) {
        double dt = (double)i - L.tm, dy = y[i] - L.ym;
        sxx = fma(dt, dt, sxx);
        syy = fma(dy, dy, syy);
        sxy = fma(dt, dy, sxy);
    }
    L.sxx = wsum(sxx) / (double)k;
    L.syy = wsum(syy) / (double)k;
    L.sxy = wsum(sxy) / (double)k;
    return L;
}

// leading decimal digit of |v| (shortest-repr digit == true digit for float32-origin values; 0 -> 0)
__device__ __forceinline__ int leading_digit(float f, const double* dec) {
    float a = fabsf(f);
    if (a == 0.f) return 0;
    double v = (double)a;
    int e = ilogb(v);
    int k = (int)floor((double)e * 0.30102999566398120);
    if (k < TSFX_DEC_MIN) k = TSFX_DEC_MIN;
    if (k + 1 <= TSFX_DEC_MAX && v >= dec[(k + 1 - TSFX_DEC_MIN) * 9]) ++k;
    if (k > TSFX_DEC_MIN && v < dec[(k - TSFX_DEC_MIN) * 9]) --k;
    const double* row = dec + (k - TSFX_DEC_MIN) * 9;
    int d = 1;
#pragma unroll
    for (int j = 1; j < 9; ++j) d += (v >= row[j]);
    return d;
}

// ---------------------------------------------------------------------------------------------------
// "Finisher" calculators are O(1) functions of the shared per-series statistics.  The statistics are parked
// in shared memory (ST) and the finishers are evaluated LANE-PARALLEL (lane l takes descriptors l, l+32, ...),
// so ~70 of the 178 BASIC columns cost a couple of warp instructions each instead of a full trip through
// the warp-uniform descriptor loop.
enum { ST_N = 0, ST_SUM, ST_MEAN, ST_SUMSQ, ST_M2, ST_VAR, ST_SD, ST_MIN, ST_MAX, ST_M3, ST_M4, ST_SAD, ST_SSD,
       ST_CNT_ABOVE, ST_CNT_BELOW, ST_CNT_MIN, ST_CNT_MAX, ST_FIRST_MIN, ST_LAST_MIN, ST_FIRST_MAX, ST_LAST_MAX,
       ST_STRIKE_ABOVE, ST_STRIKE_BELOW, ST_X0, ST_X1, ST_XN2, ST_XN1, ST_COUNT };

__host__ __device__ inline bool basic_is_finisher(int calc) {
    switch (calc) {
        case TSFX_VARIANCE_LARGER_THAN_STANDARD_DEVIATION: case TSFX_LARGE_STANDARD_DEVIATION:
        case TSFX_HAS_DUPLICATE_MAX: case TSFX_HAS_DUPLICATE_MIN: case TSFX_SUM_VALUES: case TSFX_ABS_ENERGY:
        case TSFX_MEAN: case TSFX_LENGTH: case TSFX_STANDARD_DEVIATION: case TSFX_VARIANCE:
        case TSFX_VARIATION_COEFFICIENT: case TSFX_ROOT_MEAN_SQUARE: case TSFX_MAXIMUM: case TSFX_MINIMUM:
        case TSFX_ABSOLUTE_MAXIMUM: case TSFX_MEAN_ABS_CHANGE: case TSFX_ABSOLUTE_SUM_OF_CHANGES:
        case TSFX_MEAN_CHANGE: case TSFX_MEAN_SECOND_DERIVATIVE_CENTRAL: case TSFX_SKEWNESS: case TSFX_KURTOSIS:
        case TSFX_LONGEST_STRIKE_BELOW_MEAN: case TSFX_LONGEST_STRIKE_ABOVE_MEAN: case TSFX_COUNT_ABOVE_MEAN:
        case TSFX_COUNT_BELOW_MEAN: case TSFX_LAST_LOCATION_OF_MAXIMUM: case TSFX_FIRST_LOCATION_OF_MAXIMUM:
        case TSFX_LAST_LOCATION_OF_MINIMUM: case TSFX_FIRST_LOCATION_OF_MINIMUM: case TSFX_CID_CE:
        case TSFX_AUTOCORRELATION: case TSFX_QUERY_SIMILARITY_COUNT: case TSFX_CONST_NAN:
            return true;
        default:
            return false;
    }
}

__device__ __noinline__ double basic_finisher(const Desc& d, const double* ST, const double* lagS) {
    const double dn = ST[ST_N];
    const int n = (int)dn;
    switch (d.calc) {
        case TSFX_VARIANCE_LARGER_THAN_STANDARD_DEVIATION: return (ST[ST_VAR] > sqrt(ST[ST_VAR])) ? 1.0 : 0.0;
        case TSFX_LARGE_STANDARD_DEVIATION: return (ST[ST_SD] > d.p0 * (ST[ST_MAX] - ST[ST_MIN])) ? 1.0 : 0.0;
        case TSFX_HAS_DUPLICATE_MAX: return ST[ST_CNT_MAX] >= 2.0 ? 1.0 : 0.0;
        case TSFX_HAS_DUPLICATE_MIN: return ST[ST_CNT_MIN] >= 2.0 ? 1.0 : 0.0;
        case TSFX_SUM_VALUES: return ST[ST_SUM];
        case TSFX_ABS_ENERGY: return ST[ST_SUMSQ];
        case TSFX_MEAN: return ST[ST_MEAN];
        case TSFX_LENGTH: return dn;
        case TSFX_STANDARD_DEVIATION: return ST[ST_SD];
        case TSFX_VARIANCE: return ST[ST_VAR];
        case TSFX_VARIATION_COEFFICIENT: return (ST[ST_MEAN] != 0.0) ? ST[ST_SD] / ST[ST_MEAN] : dnan();
        case TSFX_ROOT_MEAN_SQUARE: return sqrt(ST[ST_SUMSQ] / dn);
        case TSFX_MAXIMUM: return ST[ST_MAX];
        case TSFX_MINIMUM: return ST[ST_MIN];
        case TSFX_ABSOLUTE_MAXIMUM: return fmax(fabs(ST[ST_MIN]), fabs(ST[ST_MAX]));
        case TSFX_MEAN_ABS_CHANGE: return ST[ST_SAD] / (double)(n - 1);
        case TSFX_ABSOLUTE_SUM_OF_CHANGES: return ST[ST_SAD];
        case TSFX_MEAN_CHANGE: return n > 1 ? (ST[ST_XN1] - ST[ST_X0]) / (double)(n - 1) : dnan();
        case TSFX_MEAN_SECOND_DERIVATIVE_CENTRAL:
            return n > 2 ? (ST[ST_XN1] - ST[ST_XN2] - ST[ST_X1] + ST[ST_X0]) / (2.0 * (double)(n - 2)) : dnan();
        case TSFX_SKEWNESS: {   // pandas nanops.nanskew
            double amax = fmax(fabs(ST[ST_MIN]), fabs(ST[ST_MAX]));
            double e1 = 2.220446049250313e-16 * amax;
            double m2 = ST[ST_M2], m3 = ST[ST_M3];
            if (fabs(m2) < e1 * e1 * dn) m2 = 0.0;
            if (fabs(m3) < e1 * e1 * e1 * dn) m3 = 0.0;
            if (n < 3) return dnan();
            if (m2 == 0.0) return 0.0;
            return (dn * sqrt(dn - 1.0) / (dn - 2.0)) * (m3 / (m2 * sqrt(m2)));
        }
        case TSFX_KURTOSIS: {   // pandas nanops.nankurt
            double amax = fmax(fabs(ST[ST_MIN]), fabs(ST[ST_MAX]));
            double e1 = 2.220446049250313e-16 * amax, e2 = e1 * e1;
            double m2 = ST[ST_M2], m4 = ST[ST_M4];
            if (fabs(m2) < e2 * dn) m2 = 0.0;
            if (fabs(m4) < e2 * e2 * dn) m4 = 0.0;
            if (n < 4) return dnan();
            double adj = 3.0 * (dn - 1.0) * (dn - 1.0) / ((dn - 2.0) * (dn - 3.0));
            double num = dn * (dn + 1.0) * (dn - 1.0) * m4;
            double den = (dn - 2.0) * (dn - 3.0) * m2 * m2;
            return (den == 0.0) ? 0.0 : num / den - adj;
        }
        case TSFX_LONGEST_STRIKE_BELOW_MEAN: return ST[ST_STRIKE_BELOW];
        case TSFX_LONGEST_STRIKE_ABOVE_MEAN: return ST[ST_STRIKE_ABOVE];
        case TSFX_COUNT_ABOVE_MEAN: return ST[ST_CNT_ABOVE];
        case TSFX_COUNT_BELOW_MEAN: return ST[ST_CNT_BELOW];
        case TSFX_LAST_LOCATION_OF_MAXIMUM: return 1.0 - (double)(n - 1 - (int)ST[ST_LAST_MAX]) / dn;
        case TSFX_FIRST_LOCATION_OF_MAXIMUM: return ST[ST_FIRST_MAX] / dn;
        case TSFX_LAST_LOCATION_OF_MINIMUM: return 1.0 - (double)(n - 1 - (int)ST[ST_LAST_MIN]) / dn;
        case TSFX_FIRST_LOCATION_OF_MINIMUM: return ST[ST_FIRST_MIN] / dn;
        case TSFX_CID_CE:
            if (d.i0) return (ST[ST_SD] != 0.0) ? sqrt(ST[ST_SSD]) / ST[ST_SD] : 0.0;
            return sqrt(ST[ST_SSD]);
        case TSFX_AUTOCORRELATION: {
            const int lag = d.i0;
            if (n < lag || ST[ST_VAR] <= 1e-8) return dnan();      // np.isclose(v, 0) with v >= 0
            if (lag >= n) return dnan();                            // 0 / 0
            return lagS[lag] / ((double)(n - lag) * ST[ST_VAR]);
        }
        default: return dnan();
    }
}

template <int WPC, bool GS>
__global__ void __launch_bounds__(WPC * 32, (WPC == 8 ? 3 : (WPC == 12 ? 2 : 1))) k_basic(BasicArgs A) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // the descriptor table is walked by every warp on every trip: one copy per CTA in shared memory (the global-memory
    // fetch of the next descriptor right after the trip's barrier was the hottest line of the kernel)
    Desc* sdesc = reinterpret_cast<Desc*>(smem_raw);
    for (int i = threadIdx.x; i < A.nd * (int)(sizeof(Desc) / 8); i += WPC * 32)
        reinterpret_cast<double*>(sdesc)[i] = reinterpret_cast<const double*>(A.descs)[i];
    __syncthreads();
    unsigned char* base = warp_region<GS>(smem_raw + A.desc_bytes, A.gscratch, A.bytes_per_warp, WPC, warp);
    double* xc = reinterpret_cast<double*>(base);
    double* scr = xc + A.nxc;
    double* lagS = scr + A.nscr;
    double* ST = lagS + A.nlag;                     // ST_COUNT (padded to 32) shared statistics
    double* altS = ST + 32;                         // 6 regression sums per distinct agg_linear_trend key
    float* xs = reinterpret_cast<float*>(altS + 6 * A.nalt);
    const int64_t warps_total = (int64_t)gridDim.x * WPC;

    // The kernel body is ~250 KB of SASS; warps drifting through different calculators thrash the
    // instruction cache (ncu: stall_no_instruction dominated).  All warps of a CTA therefore walk the
    // descriptor list in lock step (one __syncthreads per descriptor): a CTA touches one calculator's code
    // at a time.  Rows past the end keep participating in the barriers with a duplicate of the last series.
    for (int64_t s0 = (int64_t)blockIdx.x * WPC; s0 < A.R.n_series; s0 += warps_total) {
        const bool live = (s0 + warp) < A.R.n_series;
        const int64_t s = live ? (s0 + warp) : (A.R.n_series - 1);
        const int n = load_series(A.R, s, xs, lane);
        const Moments M = moments(xs, n, xc, lane);
        const Extra E = extra_pass(xs, xc, n, M, lane);
        double* orow = A.out + (size_t)s * A.ncols;
        const double dn = (double)n;

        // zero tail of the centred copy (lag products read up to a whole chunk + the largest lag past n)
        for (int i = n + lane; i < A.nxc; i += 32) xc[i] = 0.0;
        __syncwarp();
        if (A.lag_needed > 0) {         // lag products 0..min(lag_needed, n-1)
            if (A.lag_tiles > 0) lag_products_dmma(xc, n, min(A.lag_needed, n - 1), A.lag_tiles, lagS, scr, lane);
            else lag_products(xc, n, min(A.lag_needed, n - 1), lagS, lane);
            __syncwarp();
        }
        if (lane == 0) {
            ST[ST_N] = dn; ST[ST_SUM] = M.sum; ST[ST_MEAN] = M.mean; ST[ST_SUMSQ] = M.sumsq; ST[ST_M2] = M.m2;
            ST[ST_VAR] = M.var; ST[ST_SD] = M.sd; ST[ST_MIN] = M.vmin; ST[ST_MAX] = M.vmax; ST[ST_M3] = E.m3;
            ST[ST_M4] = E.m4; ST[ST_SAD] = E.sad; ST[ST_SSD] = E.ssd; ST[ST_CNT_ABOVE] = (double)E.cnt_above;
            ST[ST_CNT_BELOW] = (double)E.cnt_below; ST[ST_CNT_MIN] = (double)E.cnt_min; ST[ST_CNT_MAX] = (double)E.cnt_max;
            ST[ST_FIRST_MIN] = (double)E.first_min; ST[ST_LAST_MIN] = (double)E.last_min;
            ST[ST_FIRST_MAX] = (double)E.first_max; ST[ST_LAST_MAX] = (double)E.last_max;
            ST[ST_STRIKE_ABOVE] = (double)E.strike_above; ST[ST_STRIKE_BELOW] = (double)E.strike_below;
            ST[ST_X0] = (double)xs[0]; ST[ST_X1] = (double)xs[n > 1 ? 1 : 0];
            ST[ST_XN2] = (double)xs[n > 1 ? n - 2 : 0]; ST[ST_XN1] = (double)xs[n - 1];
        }
        __syncwarp();
        // finishers (the first A.nfin descriptors of the group): one descriptor per lane
        if (live)
            for (int j = lane; j < A.nfin; j += 32) {
                const Desc d = sdesc[j];
                orow[d.col] = basic_finisher(d, ST, lagS);
            }
        // The remaining descriptors are sorted by calculator (tsfx_plan_create) and descriptor j writes column j of
        // the group's staging row.  One trip of the loop consumes a whole run of descriptors of one calculator
        // when they share a pass over the series (thresholds held in registers, results reduced with REDUX) or
        // when the per-descriptor work is O(1) after a shared preparation (then one descriptor per lane).
        for (int j = A.nfin; j < A.nd;) {
            if (WPC > 1) __syncthreads();
            const Desc d = sdesc[j];
            int run = 0;                    // descriptors j .. j+run-1 have the same calculator
            for (;;) {
                const int jj = j + run + lane;
                const unsigned same = __ballot_sync(FULL, jj < A.nd && sdesc[jj].calc == d.calc);
                if (same == FULL) { run += 32; continue; }
                run += __ffs(~same) - 1;
                break;
            }
            int used = 1;                   // descriptors consumed by this trip
            bool stored = false;            // the case wrote its own columns
            double r = dnan();
            switch (d.calc) {
                case TSFX_RATIO_BEYOND_R_SIGMA: {
                    constexpr int NB = 5;
                    used = min(run, NB);
                    stored = true;
                    double thr[NB];
                    int c[NB];
#pragma unroll
                    for (int t = 0; t < NB; ++t) { thr[t] = t < used ? sdesc[j + t].p0 * M.sd : dinf(); c[t] = 0; }
                    for (int i = lane; i < n; i += 32) {
                        const double v = fabs(xc[i]);
#pragma unroll
                        for (int t = 0; t < NB; ++t) c[t] += (v > thr[t]) ? 1 : 0;
                    }
#pragma unroll
                    for (int t = 0; t < NB; ++t) {
                        const int tot = wsumi(c[t]);
                        if (t < used && lane == 0 && live) orow[j + t] = (double)tot / dn;
                    }
                    break;
                }
                case TSFX_VALUE_COUNT: {
                    int c = 0;
                    for (int b0 = 0; b0 < n; b0 += 32) { int i = b0 + lane; c += wcount(i < n && (double)xs[i] == d.p0); }
                    r = (double)c;
                    break;
                }
                case TSFX_RANGE_COUNT: {
                    int c = 0;
                    for (int b0 = 0; b0 < n; b0 += 32) {
                        int i = b0 + lane;
                        double v = i < n ? (double)xs[i] : 0.0;
                        c += wcount(i < n && v >= d.p0 && v < d.p1);
                    }
                    r = (double)c;
                    break;
                }
                case TSFX_COUNT_ABOVE: {
                    int c = 0;
                    for (int b0 = 0; b0 < n; b0 += 32) { int i = b0 + lane; c += wcount(i < n && (double)xs[i] >= d.p0); }
                    r = (double)c / dn;
                    break;
                }
                case TSFX_COUNT_BELOW: {
                    int c = 0;
                    for (int b0 = 0; b0 < n; b0 += 32) { int i = b0 + lane; c += wcount(i < n && (double)xs[i] <= d.p0); }
                    r = (double)c / dn;
                    break;
                }
                case TSFX_NUMBER_CROSSING_M: {
                    int c = 0;
                    for (int b0 = 0; b0 + 1 < n; b0 += 32) {
                        int i = b0 + lane;
                        bool p = false;
                        if (i + 1 < n) p = ((double)xs[i] > d.p0) != ((double)xs[i + 1] > d.p0);
                        c += wcount(p);
                    }
                    r = (double)c;
                    break;
                }
                case TSFX_NUMBER_PEAKS: {
                    // support radius of every point (largest q with x[i] > x[i-k], x[i] > x[i+k] for all k <= q), formed
                    // once for the run; number_peaks(s) = #{radius >= s}.  Two phases keep the lanes busy: every
                    // point is walked up to radius CAP1, the few survivors (at least CAP1+1 apart) are then compacted
                    // and walked on side by side.
                    used = run;
                    stored = true;
                    constexpr int CAP1 = 12;
                    unsigned char* rad = reinterpret_cast<unsigned char*>(scr);
                    int* cand = reinterpret_cast<int*>(rad + ((n + 3) & ~3));
                    int supmax = 1;
                    for (int t = lane; t < run; t += 32) supmax = max(supmax, sdesc[j + t].i0);
                    supmax = min(wmaxi(supmax), 255);
                    int ncand = 0;
                    for (int b0 = 0; b0 < n; b0 += 32) {
                        const int i = b0 + lane;
                        bool more = false;
                        if (i < n) {
                            const float v = xs[i];
                            const int lim = min(min(i, n - 1 - i), supmax), l1 = min(lim, CAP1);
                            int q = 0;
                            while (q < l1 && v > xs[i - q - 1] && v > xs[i + q + 1]) ++q;
                            more = (q == CAP1) && (lim > CAP1);
                            rad[i] = (unsigned char)q;
                        }
                        const unsigned mm = __ballot_sync(FULL, more);
                        if (more) cand[ncand + __popc(mm & ((1u << lane) - 1u))] = i;
                        ncand += __popc(mm);
                    }
                    __syncwarp();
                    for (int c0 = 0; c0 < ncand; c0 += 32) {
                        if (c0 + lane < ncand) {
                            const int i = cand[c0 + lane];
                            const float v = xs[i];
                            const int lim = min(min(i, n - 1 - i), supmax);
                            int q = CAP1;
                            while (q < lim && v > xs[i - q - 1] && v > xs[i + q + 1]) ++q;
                            rad[i] = (unsigned char)q;
                        }
                    }
                    __syncwarp();
                    constexpr int NB = 5;
                    for (int t0 = 0; t0 < run; t0 += NB) {
                        int sup[NB], c[NB];
#pragma unroll
                        for (int t = 0; t < NB; ++t) { sup[t] = (t0 + t < run) ? sdesc[j + t0 + t].i0 : 0x7fffffff; c[t] = 0; }
                        for (int i = lane; i < n; i += 32) {
                            const int rv = rad[i];
#pragma unroll
                            for (int t = 0; t < NB; ++t) c[t] += (rv >= sup[t]) ? 1 : 0;
                        }
#pragma unroll
                        for (int t = 0; t < NB; ++t) {
                            int tot = wsumi(c[t]);
                            if (t0 + t < run && sup[t] > 255) {        // supports beyond the radius table: direct test
                                const int sp = sup[t];
                                tot = 0;
                                for (int b0 = sp; b0 < n - sp; b0 += 32) {
                                    const int i = b0 + lane;
                                    bool pk = i < n - sp;
                                    if (pk) {
                                        const float v = xs[i];
                                        for (int q = 1; q <= sp; ++q)
                                            if (!(v > xs[i - q] && v > xs[i + q])) { pk = false; break; }
                                    }
                                    tot += wcount(pk);
                                }
                            }
                            if (t0 + t < run && lane == 0 && live) orow[j + t0 + t] = (double)tot;
                        }
                    }
                    __syncwarp();
                    break;
                }
                case TSFX_AGG_AUTOCORRELATION: {
                    int cnt;
                    bool zero = (fabs(M.var) < 1e-10) || n == 1;
                    cnt = zero ? min(d.i0, n) : min(d.i0, n - 1);
                    if (cnt <= 0) { r = dnan(); break; }
                    if (zero) { r = 0.0; break; }
                    // a[k-1] = (S[k]/(n-k)) / (S[0]/n), k = 1..cnt ; staged in scr
                    double a0 = lagS[0] / dn;
                    for (int k = 1 + lane; k <= cnt; k += 32) scr[k - 1] = (lagS[k] / (double)(n - k)) / a0;
                    __syncwarp();
                    if (d.attr == TSFX_AGG_MEDIAN) {
                        int k1 = (cnt - 1) / 2, k2 = cnt / 2;
                        double v1 = 0.0, v2 = 0.0;
                        for (int i = lane; i < cnt; i += 32) {
                            double xi = scr[i];
                            int rk = 0;
                            for (int q = 0; q < cnt; ++q) { double xq = scr[q]; rk += (xq < xi) || (xq == xi && q < i); }
                            if (rk == k1) v1 = xi;
                            if (rk == k2) v2 = xi;
                        }
                        r = 0.5 * (wsum(v1) + wsum(v2));
                    } else {
                        double s1 = 0.0;
                        for (int i = lane; i < cnt; i += 32) s1 += scr[i];
                        double mu = wsum(s1) / (double)cnt;
                        if (d.attr == TSFX_AGG_MEAN) r = mu;
                        else {
                            double q2 = 0.0;
                            for (int i = lane; i < cnt; i += 32) { double dd = scr[i] - mu; q2 = fma(dd, dd, q2); }
                            double v = wsum(q2) / (double)cnt;
                            r = d.attr == TSFX_AGG_STD ? sqrt(v) : v;
                        }
                    }
                    __syncwarp();
                    break;
                }
                case TSFX_PARTIAL_AUTOCORRELATION: {
                    // pacf staged at lagS[pacf_off ..], computed once per series by lane 0; one column per lane
                    used = run;
                    stored = true;
                    double* pac = lagS + A.pacf_off;
                    const int want = d.i1;
                    if (lane == 0) {
                        int use = (want >= n / 2) ? n / 2 - 1 : want;
                        if (n <= 1 || use <= 0) { for (int k = 0; k <= want; ++k) pac[k] = dnan(); }
                        else {
                            double* acv = pac + (want + 1);
                            double* work = acv + (want + 1);
                            acv[0] = lagS[0] / dn;
                            for (int k = 1; k <= use; ++k) acv[k] = lagS[k] / (double)(n - k);
                            m_levinson_pacf(acv, use, pac, work);
                            for (int k = use + 1; k <= want; ++k) pac[k] = dnan();
                        }
                    }
                    __syncwarp();
                    if (live)
                        for (int t = lane; t < run; t += 32) orow[j + t] = pac[sdesc[j + t].i0];
                    break;
                }
                case TSFX_TIME_REVERSAL_ASYMMETRY_STATISTIC: {
                    int l = d.i0;
                    if (2 * l >= n) { r = 0.0; break; }
                    double a = 0.0;
                    for (int i = lane; i < n - 2 * l; i += 32) {
                        double x0 = xs[i], x1 = xs[i + l], x2 = xs[i + 2 * l];
                        a += x2 * x2 * x1 - x1 * x0 * x0;
                    }
                    r = wsum(a) / (double)(n - 2 * l);
                    break;
                }
                case TSFX_C3: {
                    int l = d.i0;
                    if (2 * l >= n) { r = 0.0; break; }
                    double a = 0.0;
                    for (int i = lane; i < n - 2 * l; i += 32) a += (double)xs[i + 2 * l] * (double)xs[i + l] * (double)xs[i];
                    r = wsum(a) / (double)(n - 2 * l);
                    break;
                }
                case TSFX_INDEX_MASS_QUANTILE: {
                    // cumulative mass fractions once (scr), then every quantile of the run is a count: the fractions
                    // are non-decreasing, so the first index with fraction >= q is the number of fractions < q
                    used = run;
                    stored = true;
                    double carry = 0.0;
                    for (int b0 = 0; b0 < n; b0 += 32) {
                        const int i = b0 + lane;
                        double v = i < n ? fabs((double)xs[i]) : 0.0;
#pragma unroll
                        for (int o = 1; o < 32; o <<= 1) {          // inclusive scan
                            double t = __shfl_up_sync(FULL, v, o);
                            if (lane >= o) v += t;
                        }
                        const double cum = carry + v;
                        if (i < n) scr[i] = cum;
                        carry = __shfl_sync(FULL, cum, 31);
                    }
                    const double tot = carry;
                    __syncwarp();
                    if (tot != 0.0)
                        for (int i = lane; i < n; i += 32) scr[i] = __ddiv_rn(scr[i], tot);
                    __syncwarp();
                    constexpr int NB = 4;
                    for (int t0 = 0; t0 < run; t0 += NB) {
                        double qv[NB];
                        int c[NB];
#pragma unroll
                        for (int t = 0; t < NB; ++t) { qv[t] = (t0 + t < run) ? sdesc[j + t0 + t].p0 : 0.0; c[t] = 0; }
                        for (int i = lane; i < n; i += 32) {
                            const double f = scr[i];
#pragma unroll
                            for (int t = 0; t < NB; ++t) c[t] += (f < qv[t]) ? 1 : 0;
                        }
#pragma unroll
                        for (int t = 0; t < NB; ++t) {
                            int found = wsumi(c[t]);
                            if (found >= n) found = 0;                  // np.argmax of all-False is 0
                            if (t0 + t < run && lane == 0 && live)
                                orow[j + t0 + t] = (tot == 0.0) ? dnan() : (double)(found + 1) / dn;
                        }
                    }
                    __syncwarp();
                    break;
                }
                case TSFX_ENERGY_RATIO_BY_CHUNKS: {
                    used = run;                                         // one segment per lane
                    stored = true;
                    for (int t = lane; t < run; t += 32) {
                        const Desc e = sdesc[j + t];
                        double rr = dnan();
                        if (M.sumsq != 0.0) {
                            const int ns = e.i0, fo = e.i1;
                            const int q = n / ns, rem = n % ns;
                            const int lo = fo * q + min(fo, rem), hi = lo + q + (fo < rem ? 1 : 0);
                            double a = 0.0;
                            for (int i = lo; i < hi; ++i) { const double v = xs[i]; a = fma(v, v, a); }
                            rr = a / M.sumsq;
                        }
                        if (live) orow[j + t] = rr;
                    }
                    break;
                }
                case TSFX_BINNED_ENTROPY: {
                    r = binned_entropy_of([&](int i) { return (double)xs[i]; }, n, M.vmin, M.vmax, d.i0,
                                          reinterpret_cast<int*>(scr), lane);
                    break;
                }
                case TSFX_LINEAR_TREND: {
                    used = run;                                         // one attribute per lane
                    stored = true;
                    const double tm = 0.5 * (double)(n - 1);
                    double sxx = 0.0, sxy = 0.0;
                    for (int i = lane; i < n; i += 32) {
                        double dt = (double)i - tm;
                        sxx = fma(dt, dt, sxx);
                        sxy = fma(dt, xc[i], sxy);
                    }
                    sxx = wsum(sxx) / dn;
                    sxy = wsum(sxy) / dn;
                    const LinReg fit = m_linregress(dn, tm, M.mean, sxx, M.var, sxy);
                    if (live)
                        for (int t = lane; t < run; t += 32) orow[j + t] = m_linreg_pick(fit, sdesc[j + t].attr);
                    break;
                }
                case TSFX_LINEAR_TREND_TIMEWISE: {
                    // linregress(hours since the first row, x) (:2296-2301): the regressor is
                    // (ix - ix[0]).total_seconds() / 3600 = ns / 1e9 / 3600, two correctly rounded divisions as pandas does
                    used = run;
                    stored = true;
                    LinReg fit;
                    bool have = A.R.times != nullptr;
                    if (have) {
                        const int64_t b0 = A.R.begin ? A.R.begin[s] : s * (int64_t)A.R.dense_len;
                        const int64_t* tp = A.R.times + b0;
                        const int64_t t0 = tp[0];
                        double st = 0.0;
                        for (int i = lane; i < n; i += 32) {
                            const double th = __ddiv_rn(__ddiv_rn((double)(tp[i] - t0), 1e9), 3600.0);
                            scr[i] = th;
                            st += th;
                        }
                        const double tm = wsum(st) / dn;
                        double sxx = 0.0, sxy = 0.0;
                        for (int i = lane; i < n; i += 32) {
                            const double dt = scr[i] - tm;
                            sxx = fma(dt, dt, sxx);
                            sxy = fma(dt, xc[i], sxy);
                        }
                        sxx = wsum(sxx) / dn;
                        sxy = wsum(sxy) / dn;
                        fit = m_linregress(dn, tm, M.mean, sxx, M.var, sxy);
                    }
                    if (live)
                        for (int t = lane; t < run; t += 32) orow[j + t] = have ? m_linreg_pick(fit, sdesc[j + t].attr) : dnan();
                    break;
                }
                case TSFX_AGG_LINEAR_TREND: {
                    // stage A, warp-uniform: the regression sums of every distinct (f_agg, chunk_len) of the run -> altS;
                    // stage B, one descriptor per lane: linregress of its key's sums and the attribute it asks for
                    used = run;
                    stored = true;
                    int slot = 0, key_prev = -1;
                    for (int t = 0; t < run; ++t) {
                        const int cl = sdesc[j + t].i0, fa = sdesc[j + t].i1;
                        const int key = (cl << 4) | fa;
                        if (key == key_prev) continue;
                        key_prev = key;
                        LinSums L;
                        L.k = -1.0;                                     // chunk_len >= n: NaN
                        L.tm = L.ym = L.sxx = L.syy = L.sxy = 0.0;
                        if (cl < n) {
                            const int k = (n + cl - 1) / cl;
                            for (int c = lane; c < k; c += 32) scr[c] = agg_chunk(xs, c * cl, min(n, (c + 1) * cl), fa);
                            __syncwarp();
                            L = linreg_sums(scr, k, lane);
                            __syncwarp();
                        }
                        if (lane == 0 && slot < A.nalt) {
                            double* S = altS + 6 * slot;
                            S[0] = L.k; S[1] = L.tm; S[2] = L.ym; S[3] = L.sxx; S[4] = L.syy; S[5] = L.sxy;
                        }
                        ++slot;
                    }
                    __syncwarp();
                    int base_slot = -1, last_key = -1;                  // slot of the descriptor before this batch of 32
                    for (int t0 = 0; t0 < run; t0 += 32) {
                        const int t = t0 + lane;
                        const bool ok = t < run;
                        const Desc e = sdesc[j + (ok ? t : 0)];
                        const int key = (e.i0 << 4) | e.i1;
                        int prev = __shfl_up_sync(FULL, key, 1);
                        if (lane == 0) prev = last_key;
                        const unsigned chg = __ballot_sync(FULL, ok && key != prev);
                        const int my_slot = base_slot + __popc(chg & (0xffffffffu >> (31 - lane)));
                        if (ok && live) {
                            const double* S = altS + 6 * my_slot;
                            double rr = dnan();
                            if (S[0] >= 0.0) rr = m_linreg_pick(m_linregress(S[0], S[1], S[2], S[3], S[4], S[5]), e.attr);
                            orow[j + t] = rr;
                        }
                        base_slot += __popc(chg);
                        last_key = __shfl_sync(FULL, key, 31);
                    }
                    __syncwarp();
                    break;
                }
                case TSFX_BENFORD_CORRELATION: {
                    int cnt[9];
#pragma unroll
                    for (int q = 0; q < 9; ++q) cnt[q] = 0;
                    for (int i = lane; i < n; i += 32) {
                        const int dg = leading_digit(xs[i], A.dec);
#pragma unroll
                        for (int q = 0; q < 9; ++q) cnt[q] += (dg == q + 1) ? 1 : 0;
                    }
                    // np.corrcoef(benford, observed)[0, 1];  benford[q] = log10(1 + 1/(q+1))
                    const double ben[9] = {0.30102999566398120, 0.17609125905568124, 0.12493873660829993,
                                           0.09691001300805642, 0.07918124604762482, 0.06694678963061322,
                                           0.05799194697768673, 0.05115252244738129, 0.04575749056067514};
                    double obs[9], mb = 0.0, mo = 0.0;
#pragma unroll
                    for (int q = 0; q < 9; ++q) { obs[q] = (double)wsumi(cnt[q]) / dn; mb += ben[q]; mo += obs[q]; }
                    mb /= 9.0; mo /= 9.0;
                    double sbb = 0.0, soo = 0.0, sbo = 0.0;
#pragma unroll
                    for (int q = 0; q < 9; ++q) { double a = ben[q] - mb, b = obs[q] - mo; sbb += a * a; soo += b * b; sbo += a * b; }
                    r = sbo / sqrt(sbb) / sqrt(soo);
                    if (r > 1.0) r = 1.0;
                    if (r < -1.0) r = -1.0;
                    break;
                }
                case TSFX_QUERY_SIMILARITY_COUNT:
                case TSFX_CONST_NAN:
                default: r = dnan(); break;
            }
            if (!stored && lane == 0 && live) orow[j] = r;
            j += used;
        }
        __syncwarp();
    }
}

bool basic_finisher_calc(int calc) { return basic_is_finisher(calc); }

// ------------------------------------------------------------------------------------------ launcher
cudaError_t launch_basic(const BasicArgs& A0, int max_len, cudaStream_t st, int sm_count) {
    BasicArgs A = A0;
    A.npad = (max_len + 3) & ~3;
    A.nxc = ((max_len + 255) / 256) * 256 + ((A.lag_needed + 1) & ~1);      // centred copy + zero tail for the lag products
    {
        // lag products on the FP64 tensor cores (DMMA) unless the largest lag needs more than TSFX_DMMA_MAX_TILES tiles
        // (then the FMA path); measured on B200 at 1 M x 256: 53.2 ms (FMA) -> 52.5 ms (DMMA) for the whole kernel
        const int tiles = A.lag_needed / 8 + 1 + ((A.lag_needed & 7) ? 1 : 0);
        A.lag_tiles = (A.lag_needed > 0 && tiles <= TSFX_DMMA_MAX_TILES) ? tiles : 0;
        if (A.lag_tiles > 0) {     // the strided fragment loads read up to 32 ceil(n / 32) + 8 tiles + 24 samples
            const int need = ((max_len + 31) / 32) * 32 + 8 * A.lag_tiles + 32;
            if (A.nxc < need) A.nxc = (need + 1) & ~1;
        }
    }
    size_t per = (size_t)A.nxc * 8 + (size_t)A.nscr * 8 + (size_t)A.nlag * 8 + 32 * 8 + (size_t)A.nalt * 48 + (size_t)A.npad * 4;
    per = (per + 15) & ~(size_t)15;
    A.bytes_per_warp = (int)per;
    A.desc_bytes = (int)(((size_t)A.nd * sizeof(Desc) + 15) & ~(size_t)15);
    Geometry G;
    const size_t budget = (size_t)100 * 1024 > (size_t)A.desc_bytes + per ? (size_t)100 * 1024 - A.desc_bytes : per;
    if (!plan_geometry(per, budget, 8, A.R.n_series, sm_count, A.gscratch, A.gscratch_bytes, &G)) return cudaErrorInvalidConfiguration;
    A.gscratch = G.gscratch;
    G.smem += A.desc_bytes;                       // CTA-wide descriptor table in front of the per-warp regions
    if (G.smem > 227 * 1024) return cudaErrorInvalidConfiguration;
    if (!G.gscratch && G.wpc == 8 && per * 12 + A.desc_bytes <= 227 * 1024) {
        // Two CTAs of 12 warps per SM instead of three of 8: all warps of a CTA walk the descriptor list in lock step,
        // so larger CTAs share more of the 250 KB instruction stream -- measured on B200 at 1 M x 256: 52.5 ms (3 x 8)
        // -> 42.9 ms (2 x 12), 43.9 ms (1 x 24); stall_no_instruction was the top stall reason
        const size_t smem = per * 12 + A.desc_bytes;
        const int64_t ctas = (A.R.n_series + 11) / 12;
        const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(ctas, (int64_t)sm_count * 4096));
        cudaError_t e = cudaFuncSetAttribute(k_basic<12, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        k_basic<12, false><<<grid, 12 * 32, smem, st>>>(A);
        return cudaGetLastError();
    }
    TSFX_DISPATCH(k_basic, G, st, A)
    return cudaGetLastError();
}

}  // namespace tsfx
