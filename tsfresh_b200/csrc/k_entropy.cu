// k_entropy.cu -- kernel group ENTROPY: sample_entropy (feature_calculators.py:1701-1754) and
// approximate_entropy with m = 2 (feature_calculators.py:1759-1805) -- the O(n^2) "class Q" rows.
//
// Both need, for a tolerance tau and every template start i, the number of template starts j whose
// Chebyshev distance is <= tau, for templates of length 2 (i, j in [0, n-2]) and of length 3
// (i, j in [0, n-3]).  One warp per series; up to NT = 6 tolerances share one pass so the distances are formed
// once.  Differences are float64 of float32-origin values, i.e. the very same IEEE operations numpy performs,
// so the counts are bit-identical to the reference's.  Two formulations of the counting, chosen by the series length:
//   * rank space (k_entropy_rank; series of up to ~1100 samples): sort once, the matches of a sample are a contiguous
//     rank interval, bit rows come from a prefix-bit table -- no pair tests at all (see the comment there);
//   * bit tiles (all longer series, entropy_bittile): lane = row i, 32-column bit words per tolerance, counts by
//     popcount of three shifted rows -- ~17 warp instructions per 32 pair tests and 6 tolerances.
#include <algorithm>

#include "tsfx_common.cuh"
#include "tsfx_kernels.h"

namespace tsfx {

// |x| as one integer AND on the high word (keeps the half-rate FP64 pipe for the subtractions and compares)
__device__ __forceinline__ double abs_bits(double x) {
    return __hiloint2double(__double2hiint(x) & 0x7fffffff, __double2loint(x));
}

// ---------------------------------------------------------------------------------------------------
// Bit-tile formulation.  For a tolerance tau let R_i be the bit row R_i[j] = [ |x_i - x_j| <= tau ].
// The template counts are then pure bit operations on three consecutive rows:
//     c2(i) = popc( R_i & (R_{i+1} >> 1) )                      c3(i) = popc( R_i & (R_{i+1} >> 1) & (R_{i+2} >> 2) )
// (samples beyond n are NaN, whose comparisons are false, so the ranges j <= n-2 / j <= n-3 need no masks).
// Lane = row i; a 32-column tile of R_i is built with one float64 subtract per pair plus one DSETP + predicated OR
// per tolerance -- the same IEEE operations numpy performs, so the counts stay bit-identical -- and rows i+1, i+2
// come from the neighbouring lanes by shuffle, which is why a row block advances by 30 rows, not 32.  Per 32 pairs
// and 6 tolerances this issues ~17 warp instructions (7 of them FP64) against ~35 (17 FP64) for a sweep over j with
// one pair test per tolerance.
__device__ __forceinline__ void or_le(unsigned& w, double d, double tau, unsigned bit) {
    asm("{\n\t.reg .pred p;\n\tsetp.le.f64 p, %1, %2;\n\t@p or.b32 %0, %0, %3;\n\t}" : "+r"(w) : "d"(d), "d"(tau), "r"(bit));
}

template <int NT>
__device__ __forceinline__ void entropy_bittile(const double* xd, const double* lnk, int n, const double (&tau)[NT],
                                                double (&sum_ln2)[NT], double (&sum_ln3)[NT], double (&sumB)[NT],
                                                double (&sumA)[NT], int lane) {
#pragma unroll
    for (int q = 0; q < NT; ++q) { sum_ln2[q] = 0.0; sum_ln3[q] = 0.0; sumB[q] = 0.0; sumA[q] = 0.0; }
    const int n2 = n - 1, n3 = n - 2;          // number of length-2 / length-3 templates
    if (n2 <= 0) return;
    const int W = (n + 31) >> 5;
    int iB[NT], iA[NT];
#pragma unroll
    for (int q = 0; q < NT; ++q) { iB[q] = 0; iA[q] = 0; }
    for (int r0 = 0; r0 < n2; r0 += 30) {
        const int i = r0 + lane;
        const double a = xd[i];                 // NaN beyond n: an all-zero row
        unsigned wp[NT], s1p[NT], s2p[NT];      // previous tile of rows i, i+1, i+2
        int c2[NT], c3[NT];
#pragma unroll
        for (int q = 0; q < NT; ++q) { wp[q] = 0u; s1p[q] = 0u; s2p[q] = 0u; c2[q] = 0; c3[q] = 0; }
        for (int t = 0; t <= W; ++t) {
            unsigned wn[NT];
#pragma unroll
            for (int q = 0; q < NT; ++q) wn[q] = 0u;
            if (t < W) {
                const double* xt = xd + t * 32;
#pragma unroll
                for (int jj = 0; jj < 32; ++jj) {
                    const double d = abs_bits(a - xt[jj]);
#pragma unroll
                    for (int q = 0; q < NT; ++q) or_le(wn[q], d, tau[q], 1u << jj);
                }
            }
#pragma unroll
            for (int q = 0; q < NT; ++q) {      // finish tile t-1 now that the bit spilling over from tile t is known
                const unsigned s1n = __shfl_down_sync(FULL, wn[q], 1), s2n = __shfl_down_sync(FULL, wn[q], 2);
                const unsigned m2 = wp[q] & __funnelshift_r(s1p[q], s1n, 1);
                const unsigned m3 = m2 & __funnelshift_r(s2p[q], s2n, 2);
                c2[q] += __popc(m2);
                c3[q] += __popc(m3);
                wp[q] = wn[q]; s1p[q] = s1n; s2p[q] = s2n;
            }
        }
        const bool v2 = lane < 30 && i < n2, v3 = lane < 30 && i < n3;
#pragma unroll
        for (int q = 0; q < NT; ++q) {
            if (v2) { sum_ln2[q] += lnk[c2[q]]; iB[q] += c2[q] - 1; }
            if (v3) { sum_ln3[q] += lnk[c3[q]]; iA[q] += c3[q] - 1; }
        }
    }
    const double ln2 = log((double)n2), ln3 = n3 > 0 ? log((double)n3) : 0.0;
#pragma unroll
    for (int q = 0; q < NT; ++q) {              // sum_i log(c_i / N) = sum_i log(c_i) - N log(N)
        sum_ln2[q] = wsum(sum_ln2[q]) - (double)n2 * ln2;
        sum_ln3[q] = wsum(sum_ln3[q]) - (double)n3 * ln3;
        sumB[q] = wsum((double)iB[q]);
        sumA[q] = wsum((double)iA[q]);
    }
}

template <int NT>
__device__ __forceinline__ void entropy_batch(const Desc* descs, int j0, int cnt, const double* xd, int n, double sd,
                                              double* orow, int lane, const double* lnk) {
    double tau[NT], l2[NT], l3[NT], sB[NT], sA[NT];
#pragma unroll
    for (int t = 0; t < NT; ++t) {
        if (t < cnt) {
            const Desc d = descs[j0 + t];
            tau[t] = (d.calc == TSFX_SAMPLE_ENTROPY) ? 0.2 * sd : d.p0 * sd;
        } else tau[t] = -1.0;
    }
    entropy_bittile<NT>(xd, lnk, n, tau, l2, l3, sB, sA, lane);
#pragma unroll
    for (int t = 0; t < NT; ++t) {
        if (t < cnt) {
            const Desc d = descs[j0 + t];
            double r;
            if (d.calc == TSFX_SAMPLE_ENTROPY) r = -log(sA[t] / sB[t]);
            else if (n <= 3) r = 0.0;                                  // N <= m + 1
            else r = fabs(l2[t] / (double)(n - 1) - l3[t] / (double)(n - 2));
            if (lane == 0) orow[d.col] = r;
        }
    }
}

template <int WPC, bool GS>
__global__ void __launch_bounds__(WPC * 32, (WPC == 4 ? 3 : 1)) k_entropy(EntropyArgs A) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned char* base = warp_region<GS>(smem_raw, A.gscratch, A.bytes_per_warp, WPC, warp);
    double* xd = reinterpret_cast<double*>(base);                         // xpad doubles (NaN beyond n)
    double* lnk = xd + A.xpad;                                             // log(k), k = 0..npad
    float* xs = reinterpret_cast<float*>(lnk + A.npad + 4);
    const int64_t warps_total = (int64_t)gridDim.x * WPC;

    for (int64_t s = (int64_t)blockIdx.x * WPC + warp; s < A.R.n_series; s += warps_total) {
        const int n = load_series(A.R, s, xs, lane);
        const Moments M = moments(xs, n, nullptr, lane);
        for (int i = lane; i < A.xpad; i += 32) xd[i] = i < n ? (double)xs[i] : dnan();      // NaN padding: comparisons false
        for (int k = lane; k <= n; k += 32) lnk[k] = log((double)k);
        __syncwarp();
        double* orow = A.out + (size_t)s * A.ncols;
        int j = 0;
        while (j < A.nd) {
            int left = A.nd - j;
            if (left >= 6) { entropy_batch<6>(A.descs, j, 6, xd, n, M.sd, orow, lane, lnk); j += 6; }
            else if (left > 3) { entropy_batch<6>(A.descs, j, left, xd, n, M.sd, orow, lane, lnk); j += left; }
            else if (left == 3) { entropy_batch<3>(A.descs, j, 3, xd, n, M.sd, orow, lane, lnk); j += 3; }
            else if (left == 2) { entropy_batch<2>(A.descs, j, 2, xd, n, M.sd, orow, lane, lnk); j += 2; }
            else { entropy_batch<1>(A.descs, j, 1, xd, n, M.sd, orow, lane, lnk); j += 1; }
        }
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------------------
// Rank-space formulation (series whose prefix table fits in shared memory).
// Sort the series once (rank a <-> time index pi(a)).  For a tolerance tau the set { j : |x_i - x_j| <= tau } is a
// CONTIGUOUS rank interval [lo, hi] around rank(i) (float64 subtraction of float32-origin values is monotone), so
// the bit row of the bit-tile formulation needs no pair tests at all:
//     R_i = T[hi + 1] & ~T[lo],      T[k] = { j : rank(j) < k }   (prefix bit vectors in TIME order, built once)
// and the template counts stay popc(R_i & R_{i+1} >> 1 [& R_{i+2} >> 2]).  The interval ends come from two binary
// searches per (row, tolerance) with exactly the predicate numpy evaluates ( fl64(x_a - x_b) <= tau ), so the counts
// are bit-identical to the pair-test formulation above.  O(n^2 / 32) word operations + O(n log n) searches per
// tolerance instead of O(n^2) float64 compares.
// G warps work on one series (G = 1: warp per series; G > 1: the CTA is one series and shares the table).
template <int G>
__device__ __forceinline__ void gsync() { if (G == 1) __syncwarp(); else __syncthreads(); }

__device__ __forceinline__ unsigned f32_key(float f) {      // order-preserving; -0.0 and +0.0 share one key
    unsigned u = __float_as_uint(f);
    if (u == 0x80000000u) u = 0u;
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key_f32(unsigned k) {
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

struct RankLayout {            // byte offsets inside one series' working region
    int t_off, s_off, pi_off, rk_off, lh_off, cnt_off, red_off, bytes;
    int lh_stride;             // words between the two interval tables
    int rs;                    // row stride of T in 32-bit words (multiple of 4; an odd multiple of 16 bytes when G > 1)
};
// Rows are padded when several warps share one series: an unpadded 128-byte row stride puts every row on the same
// banks.  With one warp per series they are not: measured on B200 at 1 M x 256, 39.1 ms unpadded (16 warps/SM) vs
// 39.2 ms padded (12 warps/SM).
__host__ __device__ inline RankLayout rank_layout(int nmax, int G) {
    RankLayout L;
    const bool pad = G > 1;
    int n2 = 32;
    while (n2 < nmax) n2 <<= 1;
    const int W = (nmax + 31) >> 5;
    int rs4 = (W + 3) >> 2;
    if (pad && (rs4 & 1) == 0) rs4 += 1;
    L.rs = rs4 * 4;
    int tb = (nmax + 1) * L.rs * 4;
    if (tb < n2 * 8) tb = n2 * 8;                  // the sort keys alias the table
    int o = 0;
    L.t_off = o; o += (tb + 15) & ~15;
    L.s_off = o; o += (n2 * 4 + 15) & ~15;                     // sorted keys (uint32), 0xffffffff beyond n
    L.pi_off = o; o += (n2 * 2 + 15) & ~15;
    L.rk_off = o; o += ((nmax + 2) * 2 + 15) & ~15;
    L.lh_stride = (nmax + 3) & ~3;
    L.lh_off = o; o += 2 * ((L.lh_stride * 4 + 15) & ~15);    // two tables of lo | (hi+1) << 16 per rank; the first aliases the float32 staging copy
    L.lh_stride = ((L.lh_stride * 4 + 15) & ~15) / 4;
    L.cnt_off = o; o += ((nmax + 2) * 4 + 15) & ~15;           // histogram of the interval starts
    L.red_off = o; o += (G > 1) ? G * 4 * 8 : 0;
    L.bytes = (o + 15) & ~15;
    return L;
}

template <int G, int SPC>
__global__ void __launch_bounds__(G * SPC * 32, (G == 1 ? 4 : (G == 4 ? 4 : 1))) k_entropy_rank(EntropyArgs A) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int NTHR = G * 32;
    const int lane = threadIdx.x & 31;
    const int grp = threadIdx.x / NTHR;                 // series slot inside the CTA
    const int tid = threadIdx.x - grp * NTHR;           // thread inside the series group
    const int gw = tid >> 5;                            // warp inside the series group
    const RankLayout L = rank_layout(A.npad, G);
    double* lnk = reinterpret_cast<double*>(smem_raw);                              // log(k), k = 0..npad (CTA-wide)
    unsigned char* base = smem_raw + (((A.npad + 1) * 8 + 15) & ~15) + (size_t)grp * L.bytes;
    unsigned* T = reinterpret_cast<unsigned*>(base + L.t_off);
    unsigned long long* keys = reinterpret_cast<unsigned long long*>(base + L.t_off);
    unsigned* sk = reinterpret_cast<unsigned*>(base + L.s_off);
    unsigned short* pi = reinterpret_cast<unsigned short*>(base + L.pi_off);
    unsigned short* rk = reinterpret_cast<unsigned short*>(base + L.rk_off);
    unsigned* lohi = reinterpret_cast<unsigned*>(base + L.lh_off);
    unsigned* cnt = reinterpret_cast<unsigned*>(base + L.cnt_off);
    float* xs = reinterpret_cast<float*>(base + L.lh_off);
    double* red = reinterpret_cast<double*>(base + L.red_off);
    const int RS = L.rs;

    for (int k = threadIdx.x; k <= A.npad; k += blockDim.x) lnk[k] = log((double)k);
    __syncthreads();

    const int64_t groups_total = (int64_t)gridDim.x * SPC;
    int64_t s0 = (int64_t)blockIdx.x * SPC + grp;
    // every group of a CTA runs the same number of trips when G > 1 (SPC == 1 there), so __syncthreads is safe
    for (int64_t s = s0; s < A.R.n_series; s += groups_total) {
        // ---- stage the series (every warp of the group keeps its own registers; xs is written once)
        int64_t b; int n;
        if (A.R.begin) { b = A.R.begin[s]; n = A.R.len[s]; } else { b = s * (int64_t)A.R.dense_len; n = A.R.dense_len; }
        const float* src = A.R.values + b;
        for (int i = tid; i < n; i += NTHR) xs[i] = __ldg(src + i);
        gsync<G>();
        const Moments M = moments(xs, n, nullptr, lane);          // identical in every warp of the group
        int N2 = 32;
        while (N2 < n) N2 <<= 1;
        for (int i = tid; i < N2; i += NTHR)
            keys[i] = i < n ? (((unsigned long long)f32_key(xs[i]) << 32) | (unsigned)i) : ~0ull;
        gsync<G>();
        // ---- bitonic sort by value (payload: time index)
        for (int k = 2; k <= N2; k <<= 1) {
            for (int j = k >> 1; j > 0; j >>= 1) {
                for (int t = tid; t < (N2 >> 1); t += NTHR) {
                    const int i = 2 * t - (t & (j - 1));
                    const int l = i + j;
                    const unsigned long long a = keys[i], c = keys[l];
                    const bool up = (i & k) == 0;
                    if ((a > c) == up) { keys[i] = c; keys[l] = a; }
                }
                gsync<G>();
            }
        }
        // sorted keys (for the searches), rank <-> time maps.  keys alias T: read everything before T is built
        const int per = (N2 + NTHR - 1) / NTHR;
        for (int q = 0; q < per; ++q) {
            const int a = tid + q * NTHR;
            if (a < N2) {
                const unsigned long long kv = keys[a];
                sk[a] = (unsigned)(kv >> 32);              // 0xffffffff beyond n
                if (a < n) {
                    const unsigned idx = (unsigned)kv;
                    pi[a] = (unsigned short)idx;
                    rk[idx] = (unsigned short)a;
                }
            }
        }
        gsync<G>();
        // ---- prefix table T[k][w], k = 0..n: bit j of T[k] = [rank(j) < k]
        const int W = (n + 31) >> 5;
        const int Wr = ((W + 3) >> 2) << 2;                 // the main loop reads whole 16-byte chunks
        {
            int NC = NTHR / Wr;                              // k-chunks per word column
            if (NC < 1) NC = 1;
            const int CH = (n + NC - 1) / NC;                // rows per chunk (the last chunk also writes row n)
            const int items = NC * Wr;
            for (int it0 = (tid & ~31); it0 < items; it0 += NTHR) {      // warp-uniform trip count
                unsigned init = 0u;
                for (int u = 0; u < 32; ++u) {               // starting words by ballot: 32 items per warp pass
                    const int item = it0 + u;
                    if (item >= items) break;
                    const int w = item % Wr, c = item / Wr;
                    const int j = 32 * w + lane;
                    const bool below = j < n && (int)rk[j] < c * CH;
                    const unsigned v = __ballot_sync(FULL, below);
                    if (lane == u) init = v;
                }
                const int item = it0 + lane;
                if (item < items) {
                    const int w = item % Wr, c = item / Wr;
                    const int k0 = c * CH;
                    int k1 = k0 + CH;
                    if (k1 > n) k1 = n;
                    unsigned cur = init;
                    unsigned* col = T + w;
                    for (int k = k0; k < k1; ++k) {
                        col[(size_t)k * RS] = cur;
                        const unsigned p = pi[k];
                        if ((int)(p >> 5) == w) cur |= 1u << (p & 31);
                    }
                    if (k1 == n) col[(size_t)n * RS] = cur;      // row n (every rank below n): written by the chunk(s) ending there
                }
            }
        }
        gsync<G>();
        double* orow = A.out + (size_t)s * A.ncols;
        const int n2 = n - 1, n3 = n - 2;
        // tolerances are processed two at a time: the two interval tables are built one after the other, then ONE sweep
        // over the row blocks counts both (two independent dependency chains per lane hide the shuffle / load latency)
        for (int dj = 0; dj < A.nd; dj += 2) {
            const int nq = min(2, A.nd - dj);
            double tauq[2];
            for (int q = 0; q < 2; ++q) {
                const Desc d = A.descs[dj + (q < nq ? q : 0)];
                tauq[q] = (d.calc == TSFX_SAMPLE_ENTROPY) ? 0.2 * M.sd : d.p0 * M.sd;
            }
            // ---- phase A: rank interval [lo, hi] of every rank r, per tolerance.
            // lo(r) = #{ a : x_(a) < L_r } where L_r is the smallest float32 y with fl64(x_(r) - y) <= tau (the predicate is
            // monotone in y, so the interval is exact): L_r = round-up of x_(r) - tau, corrected by at most one float32
            // step with the exact predicate, then ONE binary search over the sorted keys.  hi needs no second search:
            // the relation is symmetric (a <= hi(r) <=> lo(a) <= r), so hi(r) + 1 = #{ a : lo(a) <= r } = the inclusive
            // prefix sum of the histogram of lo.
            // both tolerances of the pair are searched together (2 x U independent chains per lane); their histograms
            // share one array (tolerance 0 in the low, tolerance 1 in the high 16 bits of each counter: counts are <= n)
            const bool sane0 = tauq[0] >= 0.0, sane1 = nq > 1 && tauq[1] >= 0.0;      // NaN / negative: every comparison is false
            unsigned* lhq[2] = {lohi, lohi + L.lh_stride};
            for (int r = tid; r <= n; r += NTHR) cnt[r] = 0u;
            gsync<G>();
            {
                constexpr int U = 4;                                 // ranks per lane and tolerance in flight
                for (int r0 = tid; r0 < n; r0 += U * NTHR) {
                    unsigned kL[2][U];
                    int pos[2][U];
#pragma unroll
                    for (int u = 0; u < U; ++u) {
                        const int r = r0 + u * NTHR;
                        const double sr = (double)key_f32(sk[r < n ? r : 0]);
#pragma unroll
                        for (int q = 0; q < 2; ++q) {
                            const double tau = tauq[q];
                            float Lf = __double2float_ru(sr - tau);
                            if (!((sr - (double)Lf) <= tau)) Lf = key_f32(f32_key(Lf) + 1u);       // one float32 step up
                            else {
                                const float Lp = key_f32(f32_key(Lf) - 1u);                          // one step down still inside?
                                if ((sr - (double)Lp) <= tau) Lf = Lp;
                            }
                            kL[q][u] = f32_key(Lf);
                            pos[q][u] = 0;
                        }
                    }
                    for (int st = N2 >> 1; st > 0; st >>= 1) {
#pragma unroll
                        for (int u = 0; u < U; ++u) {
#pragma unroll
                            for (int q = 0; q < 2; ++q)
                                if (sk[pos[q][u] + st - 1] < kL[q][u]) pos[q][u] += st;
                        }
                    }
#pragma unroll
                    for (int u = 0; u < U; ++u) {
                        const int r = r0 + u * NTHR;
                        if (r < n) {
                            // (N2 a power of two >= n: the search above covers [0, N2 - 1]; a count of N2 - 1 can only
                            // be short by the last element, checked here)
                            int lo0 = pos[0][u], lo1 = pos[1][u];
                            if (lo0 == N2 - 1 && sk[N2 - 1] < kL[0][u]) lo0 = N2;
                            if (lo1 == N2 - 1 && sk[N2 - 1] < kL[1][u]) lo1 = N2;
                            if (sane0) { lhq[0][r] = (unsigned)lo0; atomicAdd(&cnt[lo0], 1u); }
                            if (sane1) { lhq[1][r] = (unsigned)lo1; atomicAdd(&cnt[lo1], 0x10000u); }
                        }
                    }
                }
            }
            gsync<G>();
            {   // inclusive scan of the histograms by the whole group: thread t owns a contiguous run of ranks, warp scans by
                // shuffle, warp totals through shared memory (with one warp per series the last step disappears)
                const int run = (n + NTHR - 1) / NTHR;
                const int b0 = tid * run;
                unsigned v[8];
                unsigned tot = 0u;
                if (run <= 8) {         // the run lives in registers: one dependent shared-memory round trip, not one per rank
#pragma unroll
                    for (int k = 0; k < 8; ++k) { const int r = b0 + k; v[k] = (k < run && r < n) ? cnt[r] : 0u; }
#pragma unroll
                    for (int k = 0; k < 8; ++k) { tot += v[k]; v[k] = tot; }
                } else {
                    for (int k = 0; k < run; ++k) { const int r = b0 + k; if (r < n) tot += cnt[r]; }
                }
                unsigned inc = tot;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) { const unsigned w = __shfl_up_sync(FULL, inc, o); if (lane >= o) inc += w; }
                unsigned off = inc - tot;
                if (G > 1) {
                    unsigned* wtot = reinterpret_cast<unsigned*>(red);
                    if (lane == 31) wtot[gw] = inc;
                    __syncthreads();
                    for (int w = 0; w < gw; ++w) off += wtot[w];
                }
                if (run <= 8) {
#pragma unroll
                    for (int k = 0; k < 8; ++k) {
                        const int r = b0 + k;
                        if (k < run && r < n) {
                            const unsigned acc = off + v[k];
                            lhq[0][r] = sane0 ? (lhq[0][r] | (acc << 16)) : 0x00010001u;       // lo | (hi + 1) << 16; empty: T[1] & ~T[1]
                            if (nq > 1) lhq[1][r] = sane1 ? (lhq[1][r] | (acc & 0xffff0000u)) : 0x00010001u;
                        }
                    }
                } else {
                    unsigned acc = off;
                    for (int k = 0; k < run; ++k) {
                        const int r = b0 + k;
                        if (r < n) {
                            acc += cnt[r];
                            lhq[0][r] = sane0 ? (lhq[0][r] | (acc << 16)) : 0x00010001u;
                            if (nq > 1) lhq[1][r] = sane1 ? (lhq[1][r] | (acc & 0xffff0000u)) : 0x00010001u;
                        }
                    }
                }
            }
            gsync<G>();
            // ---- phase B: template counts, lane = row (30 rows per block: rows i+1, i+2 come from the next lanes)
            double l2[2] = {0.0, 0.0}, l3[2] = {0.0, 0.0};
            int iB[2] = {0, 0}, iA[2] = {0, 0};
            const double ln_n2 = n2 > 0 ? lnk[n2] : 0.0, ln_n3 = n3 > 0 ? lnk[n3] : 0.0;
            const unsigned* lh1 = lohi + (nq > 1 ? L.lh_stride : 0);
#define TSFX_RANK_STEP(Q, WN)                                                                  \
            {                                                                                  \
                const unsigned wn_ = (WN);                                                     \
                const unsigned s1n = __shfl_down_sync(FULL, wn_, 1), s2n = __shfl_down_sync(FULL, wn_, 2); \
                const unsigned m2 = wp[Q] & __funnelshift_r(s1p[Q], s1n, 1);                   \
                const unsigned m3 = m2 & __funnelshift_r(s2p[Q], s2n, 2);                      \
                c2[Q] += __popc(m2);                                                           \
                c3[Q] += __popc(m3);                                                           \
                wp[Q] = wn_; s1p[Q] = s1n; s2p[Q] = s2n;                                       \
            }
            auto sweep = [&](auto nc_tag) {
                constexpr int NC = decltype(nc_tag)::value;          // 16-byte chunks per row, 0 = run-time count
                const int nchunks = NC > 0 ? NC : (Wr >> 2);
                for (int r0 = gw * 30; r0 < n2; r0 += G * 30) {
                    const int i = r0 + lane;
                    const int ri = i < n ? (int)rk[i] : 0;
                    const unsigned lhA = i < n ? lohi[ri] : 0x00010001u;
                    const unsigned lhB = i < n ? lh1[ri] : 0x00010001u;
                    const uint4* ThiA = reinterpret_cast<const uint4*>(T + (size_t)(lhA >> 16) * RS);
                    const uint4* TloA = reinterpret_cast<const uint4*>(T + (size_t)(lhA & 0xffffu) * RS);
                    const uint4* ThiB = reinterpret_cast<const uint4*>(T + (size_t)(lhB >> 16) * RS);
                    const uint4* TloB = reinterpret_cast<const uint4*>(T + (size_t)(lhB & 0xffffu) * RS);
                    unsigned wp[2] = {0u, 0u}, s1p[2] = {0u, 0u}, s2p[2] = {0u, 0u};
                    int c2[2] = {0, 0}, c3[2] = {0, 0};
                    if (NC > 0) {
                        uint4 hA[NC > 0 ? NC : 1], lA[NC > 0 ? NC : 1], hB[NC > 0 ? NC : 1], lB[NC > 0 ? NC : 1];
#pragma unroll
                        for (int c = 0; c < NC; ++c) { hA[c] = ThiA[c]; lA[c] = TloA[c]; hB[c] = ThiB[c]; lB[c] = TloB[c]; }
#pragma unroll
                        for (int c = 0; c < NC; ++c) {
                            TSFX_RANK_STEP(0, hA[c].x & ~lA[c].x) TSFX_RANK_STEP(1, hB[c].x & ~lB[c].x)
                            TSFX_RANK_STEP(0, hA[c].y & ~lA[c].y) TSFX_RANK_STEP(1, hB[c].y & ~lB[c].y)
                            TSFX_RANK_STEP(0, hA[c].z & ~lA[c].z) TSFX_RANK_STEP(1, hB[c].z & ~lB[c].z)
                            TSFX_RANK_STEP(0, hA[c].w & ~lA[c].w) TSFX_RANK_STEP(1, hB[c].w & ~lB[c].w)
                        }
                    } else {
                        for (int c = 0; c < nchunks; ++c) {
                            const uint4 hA = ThiA[c], lA = TloA[c], hB = ThiB[c], lB = TloB[c];
                            TSFX_RANK_STEP(0, hA.x & ~lA.x) TSFX_RANK_STEP(1, hB.x & ~lB.x)
                            TSFX_RANK_STEP(0, hA.y & ~lA.y) TSFX_RANK_STEP(1, hB.y & ~lB.y)
                            TSFX_RANK_STEP(0, hA.z & ~lA.z) TSFX_RANK_STEP(1, hB.z & ~lB.z)
                            TSFX_RANK_STEP(0, hA.w & ~lA.w) TSFX_RANK_STEP(1, hB.w & ~lB.w)
                        }
                    }
                    TSFX_RANK_STEP(0, 0u) TSFX_RANK_STEP(1, 0u)
#pragma unroll
                    for (int q = 0; q < 2; ++q) {      // log(c / N) as log c - log N per row: exactly 0 when every template matches
                        if (lane < 30 && i < n2) { l2[q] += lnk[c2[q]] - ln_n2; iB[q] += c2[q] - 1; }
                        if (lane < 30 && i < n3) { l3[q] += lnk[c3[q]] - ln_n3; iA[q] += c3[q] - 1; }
                    }
                }
            };
            if (Wr == 8) sweep(std::integral_constant<int, 2>());
            else if (Wr == 4) sweep(std::integral_constant<int, 1>());
            else if (Wr == 12) sweep(std::integral_constant<int, 3>());
            else sweep(std::integral_constant<int, 0>());
#undef TSFX_RANK_STEP
            for (int q = 0; q < nq; ++q) {
                double t2 = wsum(l2[q]), t3 = wsum(l3[q]);
                double sB = (double)wsumi(iB[q]), sA = (double)wsumi(iA[q]);
                if (G > 1) {
                    if (lane == 0) { red[gw * 4 + 0] = t2; red[gw * 4 + 1] = t3; red[gw * 4 + 2] = sB; red[gw * 4 + 3] = sA; }
                    __syncthreads();
                    t2 = 0.0; t3 = 0.0; sB = 0.0; sA = 0.0;
                    for (int w = 0; w < G; ++w) { t2 += red[w * 4 + 0]; t3 += red[w * 4 + 1]; sB += red[w * 4 + 2]; sA += red[w * 4 + 3]; }
                    __syncthreads();
                }
                const Desc d = A.descs[dj + q];
                double r;
                if (d.calc == TSFX_SAMPLE_ENTROPY) r = -log(sA / sB);
                else if (n <= 3) r = 0.0;                          // N <= m + 1
                else r = fabs(t2 / (double)(n - 1) - t3 / (double)(n - 2));
                if (tid == 0) orow[d.col] = r;
            }
            gsync<G>();                                            // the interval tables are rewritten by the next pair
        }
    }
}

template <int G, int SPC>
static cudaError_t launch_rank(const EntropyArgs& A, size_t smem, int ctas_per_sm, cudaStream_t st, int sm_count) {
    cudaError_t e = cudaFuncSetAttribute(k_entropy_rank<G, SPC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int64_t ctas = (A.R.n_series + SPC - 1) / SPC;
    const int64_t cap = (int64_t)sm_count * ctas_per_sm * 16;
    if (ctas > cap) ctas = cap;
    if (ctas < 1) ctas = 1;
    k_entropy_rank<G, SPC><<<(int)ctas, G * SPC * 32, smem, st>>>(A);
    return cudaGetLastError();
}

cudaError_t launch_entropy(const EntropyArgs& A0, int max_len, cudaStream_t st, int sm_count) {
    EntropyArgs A = A0;
    A.npad = (max_len + 3) & ~3;
    A.xpad = ((A.npad + 2 + 31) / 32) * 32 + 32;          // NaN padding up to a whole 32-sample tile / 32-row block
    if (max_len < 65000) {
        // rank-space kernel: warp per series while four working regions fit three CTAs per SM, then 4 / 16 warps per
        // series with the CTA sharing one prefix table; beyond that (n > ~1100) the pair-test tiles below take over
        const size_t lnk = (((size_t)A.npad + 1) * 8 + 15) & ~(size_t)15;
        const size_t s1 = lnk + 4 * (size_t)rank_layout(A.npad, 1).bytes;
        const size_t s4 = lnk + (size_t)rank_layout(A.npad, 4).bytes;
        const size_t s16 = lnk + (size_t)rank_layout(A.npad, 16).bytes;
        const size_t sm_bytes = 227 * 1024;
        if (s1 <= 75 * 1024) return launch_rank<1, 4>(A, s1, (int)std::min<size_t>(4, sm_bytes / (s1 + 1024)), st, sm_count);
        if (s4 <= 55 * 1024) return launch_rank<4, 1>(A, s4, 4, st, sm_count);
        if (s16 <= 226 * 1024) return launch_rank<16, 1>(A, s16, 1, st, sm_count);
    }
    size_t per = (size_t)A.xpad * 8 + (size_t)(A.npad + 4) * 8 + (size_t)A.npad * 4;
    per = (per + 15) & ~(size_t)15;
    A.bytes_per_warp = (int)per;
    Geometry G;
    if (!plan_geometry(per, 64 * 1024, 4, A.R.n_series, sm_count, A.gscratch, A.gscratch_bytes, &G)) return cudaErrorInvalidConfiguration;
    A.gscratch = G.gscratch;
    TSFX_DISPATCH(k_entropy, G, st, A)
    return cudaGetLastError();
}

}  // namespace tsfx
