// k_sorted.cu -- kernel group SORTED: every calculator that needs an ordered copy of the series
// ("class S" rows of SURVEY.md section 8a): median, quantile, symmetry_looking, has_duplicate, the
// re-occurring-value family, mean_n_absolute_max, change_quantiles, friedrich_coefficients,
// max_langevin_fixed_point.
//
// One warp per series; one in-shared-memory bitonic sort (float32 keys, +inf padding) shared by all of
// them.  Shared memory per warp: xs[npad] (time order), srt[npow2] (ascending), scr[nscr] float64,
// cqS[5 ncq] (count / means / variances per change_quantiles corridor).
#include <algorithm>

#include "tsfx_common.cuh"
#include "tsfx_kernels.h"
#include "tsfx_math.cuh"

namespace tsfx {

__device__ __forceinline__ void warp_bitonic_sort(float* s, int m, int lane) {
    for (int k = 2; k <= m; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int t = lane; t < (m >> 1); t += 32) {
                int i = 2 * t - (t & (j - 1));
                int l = i + j;
                float a = s[i], b = s[l];
                bool up = (i & k) == 0;
                if ((a > b) == up) { s[i] = b; s[l] = a; }
            }
            __syncwarp();
        }
    }
}

struct Uniq { int n_unique, n_reocc_values, n_reocc_points; double sum_reocc_values, sum_reocc_points; bool any_dup; };

__device__ __forceinline__ Uniq unique_pass(const float* s, int n, int lane) {
    int nu = 0, nrv = 0, nrp = 0;
    double srv = 0.0, srp = 0.0;
    for (int i = lane; i < n; i += 32) {
        float v = s[i];
        bool eq_prev = i > 0 && s[i - 1] == v;
        bool eq_next = i + 1 < n && s[i + 1] == v;
        bool second = eq_prev && !(i > 1 && s[i - 2] == v);
        nu += !eq_prev;
        if (second) { ++nrv; srv += (double)v; }
        if (eq_prev || eq_next) { ++nrp; srp += (double)v; }
    }
    Uniq U;
    U.n_unique = wsumi(nu);
    U.n_reocc_values = wsumi(nrv);
    U.n_reocc_points = wsumi(nrp);
    U.sum_reocc_values = wsum(srv);
    U.sum_reocc_points = wsum(srp);
    U.any_dup = U.n_unique != n;
    return U;
}

// sorted copy of x[:-1] expressed as a view on the full sorted array with one instance of x[n-1] removed
struct DropLast {
    const float* s;
    int pos;
    __device__ __forceinline__ float operator[](int j) const { return s[j + (j >= pos ? 1 : 0)]; }
};

__device__ __forceinline__ double quantile_view(const DropLast& v, int n, double q) {
    double posf = q * (double)(n - 1);
    double fl = floor(posf);
    int lo = (int)fl;
    if (lo < 0) lo = 0;
    if (lo > n - 1) lo = n - 1;
    int hi = lo + 1 > n - 1 ? n - 1 : lo + 1;
    double t = posf - fl;
    double a = (double)v[lo], b = (double)v[hi];
    double d = b - a;
    if (t >= 0.5) return b - d * (1.0 - t);
    return a + d * t;
}

// np.polyfit(x, y, 3) for k >= 4 points held in shared memory, all lanes cooperating (points strided over
// lanes): column-scaled normal equations, 4x4 Cholesky done redundantly by every lane, two refinement steps
// with residuals formed from the data (same algebra as m_polyfit3, which stays for the k < 4 minimum-norm case).
__device__ __forceinline__ bool warp_polyfit3(const double* x, const double* y, int k, double* coef, int lane) {
    double sc[4] = {0, 0, 0, 0};
    for (int i = lane; i < k; i += 32) {
        const double v = x[i], v2 = v * v, v3 = v2 * v;
        sc[0] = fma(v3, v3, sc[0]); sc[1] = fma(v2, v2, sc[1]); sc[2] = fma(v, v, sc[2]); sc[3] += 1.0;
    }
#pragma unroll
    for (int a = 0; a < 4; ++a) sc[a] = sqrt(wsum(sc[a]));
    double G[16], rhs[4];
#pragma unroll
    for (int a = 0; a < 16; ++a) G[a] = 0.0;
#pragma unroll
    for (int a = 0; a < 4; ++a) rhs[a] = 0.0;
    for (int i = lane; i < k; i += 32) {
        const double v = x[i];
        const double col[4] = {v * v * v / sc[0], v * v / sc[1], v / sc[2], 1.0 / sc[3]};
#pragma unroll
        for (int a = 0; a < 4; ++a) {
            rhs[a] = fma(col[a], y[i], rhs[a]);
#pragma unroll
            for (int b = 0; b <= a; ++b) G[a * 4 + b] = fma(col[a], col[b], G[a * 4 + b]);
        }
    }
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        rhs[a] = wsum(rhs[a]);
#pragma unroll
        for (int b = 0; b <= a; ++b) G[a * 4 + b] = wsum(G[a * 4 + b]);
    }
    if (!m_cholesky(G, 4, 4)) return false;
    double sol[4] = {rhs[0], rhs[1], rhs[2], rhs[3]};
    m_forward(G, 4, 4, sol);
    m_backward(G, 4, 4, sol);
    for (int it = 0; it < 2; ++it) {
        double r4[4] = {0, 0, 0, 0};
        for (int i = lane; i < k; i += 32) {
            const double v = x[i];
            const double col[4] = {v * v * v / sc[0], v * v / sc[1], v / sc[2], 1.0 / sc[3]};
            const double e = y[i] - (col[0] * sol[0] + col[1] * sol[1] + col[2] * sol[2] + col[3] * sol[3]);
#pragma unroll
            for (int a = 0; a < 4; ++a) r4[a] = fma(col[a], e, r4[a]);
        }
#pragma unroll
        for (int a = 0; a < 4; ++a) r4[a] = wsum(r4[a]);
        m_forward(G, 4, 4, r4);
        m_backward(G, 4, 4, r4);
#pragma unroll
        for (int a = 0; a < 4; ++a) sol[a] += r4[a];
    }
    if (lane == 0) { coef[0] = sol[0] / sc[0]; coef[1] = sol[1] / sc[1]; coef[2] = sol[2] / sc[2]; coef[3] = sol[3] / sc[3]; }
    __syncwarp();
    return true;
}

// Estimates the Friedrich cubic (feature_calculators.py:131-173 with m = 3): returns in all lanes
// whether a coefficient vector exists; coefficients land in coef[0..3] (shared memory).
__device__ __forceinline__ bool friedrich_fit(const float* xs, const float* srt, int n, int r, double* scr, double* coef,
                                              int lane) {
    const int n1 = n - 1;                        // length of signal = x[:-1]
    if (n1 < 1) return false;
    double* edges = scr;                         // r + 1
    double* cnt = edges + (r + 1);               // r
    double* sx = cnt + r;                        // r
    double* sy = sx + r;                         // r
    // position of one instance of x[n-1] inside the sorted array
    const float last = xs[n - 1];
    int pos = 0x7fffffff;
    for (int b0 = 0; b0 < n && pos == 0x7fffffff; b0 += 32) {
        int i = b0 + lane;
        unsigned hit = __ballot_sync(FULL, i < n && srt[i] == last);
        if (hit) pos = b0 + __ffs(hit) - 1;
    }
    DropLast view{srt, pos};
    // quantile levels of pd.qcut(x, r): linspace(0, 1, r+1), bumped to the next double where r*q != i
    const double step = __ddiv_rn(1.0, (double)r);
    for (int i = lane; i <= r; i += 32) {
        double q = (i == r) ? 1.0 : __dmul_rn((double)i, step);
        if (__dmul_rn((double)r, q) != (double)i) q = nextafter(q, 1.0);
        edges[i] = quantile_view(view, n1, q);
    }
    for (int i = lane; i < r; i += 32) { cnt[i] = 0.0; sx[i] = 0.0; sy[i] = 0.0; }
    __syncwarp();
    bool dup = false;
    for (int i = lane; i < r; i += 32) dup |= (edges[i] == edges[i + 1]);
    if (__any_sync(FULL, dup) && r + 1 != 2) return false;      // "Bin edges must be unique" -> NaN
    for (int j = lane; j < n1; j += 32) {
        double v = (double)xs[j];
        double dl = (double)xs[j + 1] - v;
        // ids = searchsorted(edges, v, side="left") ; include_lowest: v == edges[0] -> 1
        int lo = 0, hi = r + 1;
        while (lo < hi) { int mid = (lo + hi) >> 1; if (edges[mid] < v) lo = mid + 1; else hi = mid; }
        int id = lo;
        if (v == edges[0]) id = 1;
        if (id >= 1 && id <= r) {
            atomicAdd(&cnt[id - 1], 1.0);
            atomicAdd(&sx[id - 1], v);
            atomicAdd(&sy[id - 1], dl);
        }
    }
    __syncwarp();
    // bin means of the non-empty bins, compacted in bin order (32 bins per round; a round only overwrites slots
    // at or below the bins it has already read)
    int k = 0;
    for (int b0 = 0; b0 < r; b0 += 32) {
        const int b = b0 + lane;
        const double c = b < r ? cnt[b] : 0.0;
        double mx = 0.0, my = 0.0;
        if (c > 0.0) { mx = sx[b] / c; my = sy[b] / c; }
        const unsigned full = __ballot_sync(FULL, c > 0.0);
        __syncwarp();
        if (c > 0.0) {
            const int dst = k + __popc(full & ((1u << lane) - 1u));
            sx[dst] = mx; sy[dst] = my;
        }
        k += __popc(full);
        __syncwarp();
    }
    int ok = 0;
    if (k >= 4) ok = warp_polyfit3(sx, sy, k, coef, lane) ? 1 : 0;
    else {
        if (lane == 0) {
            double c4[4];
            ok = (k > 0 && m_polyfit3(sx, sy, k, c4)) ? 1 : 0;
            if (ok) { coef[0] = c4[0]; coef[1] = c4[1]; coef[2] = c4[2]; coef[3] = c4[3]; }
        }
        ok = __shfl_sync(FULL, ok, 0);
    }
    __syncwarp();
    return ok != 0;
}

template <int WPC, bool GS>
__global__ void __launch_bounds__(WPC * 32, (WPC == 8 ? 3 : (WPC == 12 ? 2 : 1))) k_sorted(SortedArgs A) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned char* base = warp_region<GS>(smem_raw, A.gscratch, A.bytes_per_warp, WPC, warp);
    double* scr = reinterpret_cast<double*>(base);
    float* xs = reinterpret_cast<float*>(scr + A.nscr + 5 * A.ncq + (A.ncq & 1));
    float* srt = xs + A.npad;
    const int64_t warps_total = (int64_t)gridDim.x * WPC;

    // lock-step walk of the descriptor list per CTA (see k_basic.cu): keeps the instruction working set small
    for (int64_t s0 = (int64_t)blockIdx.x * WPC; s0 < A.R.n_series; s0 += warps_total) {
        const bool live = (s0 + warp) < A.R.n_series;
        const int64_t s = live ? (s0 + warp) : (A.R.n_series - 1);
        const int n = load_series(A.R, s, xs, lane);
        int m = 1;
        while (m < n) m <<= 1;
        double sum = 0.0;
        for (int i = lane; i < m; i += 32) {
            float v = i < n ? xs[i] : INFINITY;
            srt[i] = v;
            if (i < n) sum += (double)v;
        }
        sum = wsum(sum);
        __syncwarp();
        warp_bitonic_sort(srt, m, lane);
        const double dn = (double)n;
        const double mean = sum / dn;
        const double vmin = (double)srt[0], vmax = (double)srt[n - 1];
        const double med = (n & 1) ? (double)srt[n >> 1] : 0.5 * ((double)srt[(n >> 1) - 1] + (double)srt[n >> 1]);
        double* orow = A.out + (size_t)s * A.ncols;

        int fr_r = -1; bool fr_ok = false;          // friedrich cache
        double* coef = scr + (A.nscr - 8);
        double* cqS = scr + A.nscr;                 // 5 doubles per distinct change_quantiles corridor

        // O(1) "finishers" (the first A.nfin descriptors): order statistics and the unique-value counts, one
        // descriptor per lane
        if (A.nfin > 0) {
            const Uniq U = unique_pass(srt, n, lane);
            if (live)
                for (int j = lane; j < A.nfin; j += 32) {
                    const Desc d = A.descs[j];
                    double r = dnan();
                    switch (d.calc) {
                        case TSFX_MEDIAN: r = med; break;
                        case TSFX_QUANTILE: r = m_quantile_sorted(srt, n, d.p0); break;
                        case TSFX_SYMMETRY_LOOKING: r = (fabs(mean - med) < d.p0 * (vmax - vmin)) ? 1.0 : 0.0; break;
                        case TSFX_HAS_DUPLICATE: r = U.any_dup ? 1.0 : 0.0; break;
                        case TSFX_PERCENTAGE_OF_REOCCURRING_VALUES_TO_ALL_VALUES:
                            r = (double)U.n_reocc_values / (double)U.n_unique; break;
                        case TSFX_PERCENTAGE_OF_REOCCURRING_DATAPOINTS_TO_ALL_DATAPOINTS:
                            r = (double)U.n_reocc_points / dn; break;
                        case TSFX_SUM_OF_REOCCURRING_VALUES: r = U.sum_reocc_values; break;
                        case TSFX_SUM_OF_REOCCURRING_DATA_POINTS: r = U.sum_reocc_points; break;
                        case TSFX_RATIO_VALUE_NUMBER_TO_TIME_SERIES_LENGTH: r = (double)U.n_unique / dn; break;
                        default: break;
                    }
                    orow[j] = r;
                }
        }

        // remaining descriptors: sorted by calculator, descriptor j writes column j; one trip per run (see k_basic.cu)
        for (int j = A.nfin; j < A.nd;) {
            if (WPC > 1) __syncthreads();
            const Desc d = A.descs[j];
            int run = 0;
            for (;;) {
                const int jj = j + run + lane;
                const unsigned same = __ballot_sync(FULL, jj < A.nd && A.descs[jj].calc == d.calc);
                if (same == FULL) { run += 32; continue; }
                run += __ffs(~same) - 1;
                break;
            }
            int used = 1;
            bool stored = false;
            double r = dnan();
            switch (d.calc) {
                case TSFX_MEAN_N_ABSOLUTE_MAX: {
                    int k = d.i0;
                    if (n <= k) { r = dnan(); break; }
                    double acc = 0.0;
                    if (lane == 0) {
                        int a = 0, b = n - 1;
                        for (int q = 0; q < k; ++q) {
                            float fa = fabsf(srt[a]), fb = fabsf(srt[b]);
                            if (fa > fb) { acc += (double)fa; ++a; } else { acc += (double)fb; --b; }
                        }
                    }
                    r = __shfl_sync(FULL, acc, 0) / (double)k;
                    break;
                }
                case TSFX_CHANGE_QUANTILES: {
                    // stage A, warp-uniform: every distinct corridor (ql, qh) of the run -> count, mean and variance of
                    // the changes and of their magnitudes (two passes serve all four (isabs, f_agg) columns);
                    // stage B: one descriptor per lane picks its column
                    used = run;
                    stored = true;
                    int slot = 0;
                    double pl = -1.0, ph = -1.0;
                    for (int t = 0; t < run; ++t) {
                        const double ql = A.descs[j + t].p0, qh = A.descs[j + t].p1;
                        if (ql == pl && qh == ph) continue;
                        pl = ql; ph = qh;
                        int cnt = 0;
                        double mean0 = 0.0, mean1 = 0.0, var0 = 0.0, var1 = 0.0;
                        if (ql < qh) {
                            const double lo = m_quantile_sorted(srt, n, ql), hi = m_quantile_sorted(srt, n, qh);
                            int c = 0;
                            double s1 = 0.0, s1a = 0.0;
                            for (int i = lane; i + 1 < n; i += 32) {
                                const double a = (double)xs[i], b = (double)xs[i + 1];
                                if (a >= lo && a <= hi && b >= lo && b <= hi) { const double dx = b - a; s1 += dx; s1a += fabs(dx); ++c; }
                            }
                            cnt = wsumi(c);
                            mean0 = wsum(s1) / (double)cnt;
                            mean1 = wsum(s1a) / (double)cnt;
                            double q2 = 0.0, q2a = 0.0;
                            if (cnt > 0)
                                for (int i = lane; i + 1 < n; i += 32) {
                                    const double a = (double)xs[i], b = (double)xs[i + 1];
                                    if (a >= lo && a <= hi && b >= lo && b <= hi) {
                                        const double dx = b - a, e = dx - mean0, ea = fabs(dx) - mean1;
                                        q2 = fma(e, e, q2);
                                        q2a = fma(ea, ea, q2a);
                                    }
                                }
                            var0 = wsum(q2) / (double)cnt;
                            var1 = wsum(q2a) / (double)cnt;
                        }
                        if (lane == 0 && slot < A.ncq) {
                            double* S = cqS + 5 * slot;
                            S[0] = (double)cnt; S[1] = mean0; S[2] = mean1; S[3] = var0; S[4] = var1;
                        }
                        ++slot;
                    }
                    __syncwarp();
                    int base_slot = -1;
                    double last_l = -1.0, last_h = -1.0;
                    for (int t0 = 0; t0 < run; t0 += 32) {
                        const int t = t0 + lane;
                        const bool ok = t < run;
                        const Desc e = A.descs[j + (ok ? t : 0)];
                        double prev_l = __shfl_up_sync(FULL, e.p0, 1), prev_h = __shfl_up_sync(FULL, e.p1, 1);
                        if (lane == 0) { prev_l = last_l; prev_h = last_h; }
                        const unsigned chg = __ballot_sync(FULL, ok && !(e.p0 == prev_l && e.p1 == prev_h));
                        const int my_slot = base_slot + __popc(chg & (0xffffffffu >> (31 - lane)));
                        if (ok && live) {
                            const double* S = cqS + 5 * my_slot;
                            double rr = 0.0;                             // ql >= qh or an empty corridor: 0
                            if (S[0] > 0.0) {
                                const double mu = e.i0 ? S[2] : S[1], va = e.i0 ? S[4] : S[3];
                                rr = (e.attr == TSFX_AGG_MEAN) ? mu : (e.attr == TSFX_AGG_STD) ? sqrt(va) : va;
                            }
                            orow[j + t] = rr;
                        }
                        base_slot += __popc(chg);
                        last_l = __shfl_sync(FULL, e.p0, 31);
                        last_h = __shfl_sync(FULL, e.p1, 31);
                    }
                    __syncwarp();
                    break;
                }
                case TSFX_FRIEDRICH_COEFFICIENTS:
                case TSFX_MAX_LANGEVIN_FIXED_POINT: {
                    if (fr_r != d.i2) {
                        __syncwarp();
                        fr_ok = friedrich_fit(xs, srt, n, d.i2, scr, coef, lane);
                        fr_r = d.i2;
                    }
                    if (!fr_ok) { r = dnan(); break; }
                    if (d.calc == TSFX_FRIEDRICH_COEFFICIENTS) r = (d.i0 >= 0 && d.i0 <= 3) ? coef[d.i0] : dnan();
                    else r = m_poly3_max_real_root(coef[0], coef[1], coef[2], coef[3]);
                    break;
                }
                default: break;
            }
            if (!stored && lane == 0 && live) orow[j] = r;
            j += used;
        }
        __syncwarp();
    }
}

bool sorted_finisher_calc(int calc) {
    switch (calc) {
        case TSFX_MEDIAN: case TSFX_QUANTILE: case TSFX_SYMMETRY_LOOKING: case TSFX_HAS_DUPLICATE:
        case TSFX_PERCENTAGE_OF_REOCCURRING_VALUES_TO_ALL_VALUES:
        case TSFX_PERCENTAGE_OF_REOCCURRING_DATAPOINTS_TO_ALL_DATAPOINTS:
        case TSFX_SUM_OF_REOCCURRING_VALUES: case TSFX_SUM_OF_REOCCURRING_DATA_POINTS:
        case TSFX_RATIO_VALUE_NUMBER_TO_TIME_SERIES_LENGTH: return true;
        default: return false;
    }
}

cudaError_t launch_sorted(const SortedArgs& A0, int max_len, cudaStream_t st, int sm_count) {
    SortedArgs A = A0;
    A.npad = (max_len + 3) & ~3;
    int p2 = 1;
    while (p2 < max_len) p2 <<= 1;
    A.npow2 = std::max(p2, 4);
    A.nscr = (A.nscr + 1) & ~1;
    size_t per = (size_t)A.nscr * 8 + (size_t)(5 * A.ncq + (A.ncq & 1)) * 8 + (size_t)A.npad * 4 + (size_t)A.npow2 * 4;
    per = (per + 15) & ~(size_t)15;
    A.bytes_per_warp = (int)per;
    Geometry G;
    if (!plan_geometry(per, 100 * 1024, 8, A.R.n_series, sm_count, A.gscratch, A.gscratch_bytes, &G)) return cudaErrorInvalidConfiguration;
    A.gscratch = G.gscratch;
    // 8-warp CTAs: the 12-warp CTAs that help k_basic measured 23.7 -> 23.8 ms here on B200 at 1 M x 256 (no
    // instruction-cache pressure in this kernel; profiles/r2_notes.md)
    TSFX_DISPATCH(k_sorted, G, st, A)
    return cudaGetLastError();
}

}  // namespace tsfx
