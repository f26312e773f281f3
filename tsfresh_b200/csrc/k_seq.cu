// k_seq.cu -- kernel group SEQ: the inherently sequential / dictionary calculators
//   lempel_ziv_complexity (feature_calculators.py:1825-1862)   lane-per-parameter trie parse
//   permutation_entropy   (feature_calculators.py:1866-1915)   rank codes -> bitonic sort -> run lengths
//   number_cwt_peaks      (feature_calculators.py:1320-1339; scipy.signal.find_peaks_cwt with _ricker :1307)
//
// One warp per series.  k_seq (lempel_ziv + permutation_entropy): general layout = uint32 codes[npow2], one uint32
// open-addressing key table per Lempel-Ziv parameter, uint16 symbols, float xs[npad] (17.8 KB per warp at 256 samples,
// run from the global working region); compact layout k_seq_small (series <= 256, alphabets <= 127) = packed 16-bit
// histogram counters, 16-bit keys in 256-slot tables, byte symbols (6.5 KB per warp, shared memory, 32 warps per SM).
// k_peaks (number_cwt_peaks): row0[npad], tmp[npad] (cwt rows, float64), noise[npad], hw[TSFX_MAXW_PTS] (wavelet taps),
// float32 copies of the wider rows, a zero-padded float64 copy of the series in the working region; the ridge-line
// tables (5 int16 + 3 int32 per line), the column map and the local-maximum bit masks in shared memory.
#include <algorithm>

#include "tsfx_common.cuh"
#include "tsfx_kernels.h"

namespace tsfx {

#define TSFX_CWT_MAXN 16
#define TSFX_MAXW_PTS 160
#define LZ_LANES 8

struct SeqLayout {
    int hot_bytes, hot_lines, hot_map, hot_bits;     // k_peaks from the global working region: the small, latency-critical
                                                     // tables (ridge lines, column map, maxima bits) stay in shared memory
    int hist_cap;                                    // permutation-histogram bins the `codes` area can hold
    int npad, npow2, nwords, lz_lanes, cwt_n, lz_hash, lz_stride, nxd;
    int off_rowsf, off_noise, off_hw, off_codes, off_trie, off_sym, off_bits, off_lines, off_map, off_xs, off_xd;   // byte offsets
};

// ---------------------------------------------------------------------------- Lempel-Ziv
// symbol = np.searchsorted(np.linspace(min, max, bins+1)[1:], x, side="left")
__device__ __forceinline__ int lz_symbol(double v, double vmin, double vmax, double step, int bins) {
    int c = (int)__ddiv_rn(__dsub_rn(v, vmin), step);      // NaN (step == 0) converts to 0
    if (c < 0) c = 0;
    if (c > bins) c = bins;
    // edge(i) = i*step + vmin for i < bins, edge(bins) = vmax ; count edges i in 1..bins with edge(i) < v
    while (c < bins) {
        double e = (c + 1 == bins) ? vmax : __dadd_rn(__dmul_rn((double)(c + 1), step), vmin);
        if (e < v) ++c; else break;
    }
    while (c > 0) {
        double e = (c == bins) ? vmax : __dadd_rn(__dmul_rn((double)c, step), vmin);
        if (!(e < v)) --c; else break;
    }
    return c;
}

// ---------------------------------------------------------------------------- bitonic sort on uint32
__device__ __forceinline__ void warp_bitonic_sort_u32(unsigned* s, int m, int lane) {
    for (int k = 2; k <= m; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int t = lane; t < (m >> 1); t += 32) {
                int i = 2 * t - (t & (j - 1));
                int l = i + j;
                unsigned a = s[i], b = s[l];
                bool up = (i & k) == 0;
                if ((a > b) == up) { s[i] = b; s[l] = a; }
            }
            __syncwarp();
        }
    }
}

// ---------------------------------------------------------------------------- find_peaks_cwt pieces
// cwt row of width w: dst[i] = convolve(x, ricker(npts, w), mode="same")[i] = sum_u h[u] x[i + c0 - u], c0 = (npts-1)/2.
// xd is the series as float64 with TSFX_MAXW_PTS zeros in front and zeros up to a whole 256-sample chunk (+ the
// same margin) behind, so no tap needs a bounds test.  Each lane forms 8 outputs (i = lane + 32 m) at once: one
// broadcast load of the tap serves all of them, i.e. ~2.4 instructions per output tap instead of ~5.5.
__device__ __forceinline__ void cwt_row(const double* xd, int n, const double* hw, int npts, double* dst, int lane) {
    const int c0 = (npts - 1) / 2;
    for (int i0 = 0; i0 < n; i0 += 256) {
        double acc[8];
#pragma unroll
        for (int m = 0; m < 8; ++m) acc[m] = 0.0;
        const double* xb = xd + TSFX_MAXW_PTS + i0 + lane + c0;
        for (int u = 0; u < npts; ++u) {
            const double h = hw[u];
#pragma unroll
            for (int m = 0; m < 8; ++m) acc[m] = fma(xb[32 * m - u], h, acc[m]);
        }
#pragma unroll
        for (int m = 0; m < 8; ++m) {
            const int i = i0 + lane + 32 * m;
            if (i < n) dst[i] = acc[m];
        }
    }
}

__device__ __forceinline__ void ricker_fill(double* hw, int npts, int w, int lane) {
    // _ricker(points, a) (:1307-1316)
    const double a = (double)w;
    const double A = 2.0 / (sqrt(3.0 * a) * pow(3.14159265358979323846, 0.25));
    const double wsq = a * a;
    for (int v = lane; v < npts; v += 32) {
        double vec = (double)v - ((double)npts - 1.0) / 2.0;
        double xsq = vec * vec;
        double mod = 1.0 - xsq / wsq;
        double gauss = exp(-xsq / (2.0 * wsq));
        hw[v] = A * mod * gauss;
    }
    __syncwarp();
}

// scipy.stats.scoreatpercentile(win[0..wlen), 10): the order statistics i = floor(0.1 (wlen-1)) and i+1 are
// found by successive minima over (value, index) pairs -- no scratch, read-only window, O(wlen * (i+2)).
__device__ __forceinline__ double percentile10(const double* win, int wlen) {
    const double idx = 10.0 / 100.0 * (double)(wlen - 1);
    const int i = (int)idx;
    double pv = 0.0, v0 = 0.0, v1 = 0.0;
    int pi = -1;
    if (i <= 1) {                       // windows of up to 20 samples: the three smallest in one pass
        double m0 = dinf(), m1 = dinf(), m2 = dinf();
        for (int a = 0; a < wlen; ++a) {
            const double va = win[a];
            if (va < m0) { m2 = m1; m1 = m0; m0 = va; }
            else if (va < m1) { m2 = m1; m1 = va; }
            else if (va < m2) m2 = va;
        }
        v0 = i == 0 ? m0 : m1;
        v1 = i == 0 ? m1 : m2;
    } else
    for (int r = 0; r <= i + 1 && r < wlen; ++r) {
        double bv = 0.0;
        int bi = -1;
        for (int a = 0; a < wlen; ++a) {
            const double va = win[a];
            const bool after = (pi < 0) || (va > pv) || (va == pv && a > pi);
            if (after && (bi < 0 || va < bv)) { bv = va; bi = a; }
        }
        pv = bv; pi = bi;
        if (r == i) v0 = bv;
        if (r == i + 1) v1 = bv;
    }
    if ((double)i == idx) return v0;
    const double w0 = (double)(i + 1) - idx, w1 = idx - (double)i;
    return (v0 * w0 + v1 * w1) / (w0 + w1);
}

// ---------------------------------------------------------------------------- permutation patterns
// A window's rank pattern is fixed by its pairwise order bits b(p,q) = [w_q < w_p], p < q (ties: the earlier
// sample counts as smaller = stable ranks).  With the bits laid out q-major (bit q(q-1)/2 + p) the pattern of
// the first D samples is the low D(D-1)/2 bits, so ONE pass over a window serves every dimension.  The dense
// index used for counting is the Lehmer code: digit p = popcount(bits & PE_MASK[D][p]).
struct PeMasks { unsigned m[9][8]; };
__host__ __device__ constexpr PeMasks make_pe_masks() {
    PeMasks M = {};
    for (int D = 2; D <= 8; ++D)
        for (int p = 0; p < D - 1; ++p) {
            unsigned v = 0;
            for (int q = p + 1; q < D; ++q) v |= 1u << (q * (q - 1) / 2 + p);
            M.m[D][p] = v;
        }
    return M;
}
__constant__ PeMasks PE_MASKS = make_pe_masks();

__device__ __forceinline__ unsigned pe_order_bits(const float* w, int m) {      // m = samples available (<= 8)
    float v[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) v[q] = q < m ? w[q] : 0.f;
    unsigned bits = 0;
#pragma unroll
    for (int q = 1; q < 8; ++q)
#pragma unroll
        for (int p = 0; p < q; ++p)
            if (q < m) bits |= (v[q] < v[p]) ? (1u << (q * (q - 1) / 2 + p)) : 0u;
    return bits;
}
__device__ __forceinline__ unsigned pe_lehmer(unsigned bits, int D) {
    unsigned code = 0;
    for (int p = 0; p < D - 1; ++p) code = code * (unsigned)(D - p) + (unsigned)__popc(bits & PE_MASKS.m[D][p]);
    return code;            // digit D-1 is always 0 (radix 1)
}

// SMALL = compact shared-memory working set for series of at most 256 samples and alphabets of at most 127 symbols (the
// BASELINE shapes): byte symbols, 16-bit trie keys (node << 7 | symbol, 256 slots per parse) and permutation histograms
// with two 16-bit counters per word -- 6.5 KB per warp, so 32 warps per SM run entirely from shared memory.  The general
// layout (uint32 keys, uint16 symbols, uint32 counters) needs 17.8 KB per warp and runs from the global working region,
// where every probe of the sequential parse and every histogram update is an L2 round trip (ncu: long_scoreboard 5.2
// stalls per issued instruction).
template <int WPC, bool GS, bool SMALL>
__device__ __forceinline__ void seq_body(const SeqArgs& A, const SeqLayout& Y) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ double clogc_small[64];            // c ln c for small counts (permutation histograms are mostly tiny)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x < 64) clogc_small[threadIdx.x] = threadIdx.x > 1 ? (double)threadIdx.x * log((double)threadIdx.x) : 0.0;
    if (WPC * 32 < 64 && threadIdx.x < 32) clogc_small[32 + threadIdx.x] = (double)(32 + threadIdx.x) * log((double)(32 + threadIdx.x));
    __syncthreads();
    unsigned char* base = warp_region<GS>(smem_raw, A.gscratch, A.bytes_per_warp, WPC, warp);
    unsigned* codes = reinterpret_cast<unsigned*>(base + Y.off_codes);
    unsigned short* trie = reinterpret_cast<unsigned short*>(base + Y.off_trie);
    unsigned short* symbuf = reinterpret_cast<unsigned short*>(base + Y.off_sym);
    unsigned char* symbuf8 = base + Y.off_sym;
    float* xs = reinterpret_cast<float*>(base + Y.off_xs);
    const int64_t warps_total = (int64_t)gridDim.x * WPC;

    for (int64_t s = (int64_t)blockIdx.x * WPC + warp; s < A.R.n_series; s += warps_total) {
        const int n = load_series(A.R, s, xs, lane);
        double* orow = A.out + (size_t)s * A.ncols;
        float lo = INFINITY, hi = -INFINITY;
        for (int i = lane; i < n; i += 32) { lo = fminf(lo, xs[i]); hi = fmaxf(hi, xs[i]); }
        const double vmin = (double)wminf(lo), vmax = (double)wmaxf(hi);

        int j = 0;
        while (j < A.nd) {
            const Desc d0 = A.descs[j];
            if (d0.calc == TSFX_LEMPEL_ZIV_COMPLEXITY) {
                // up to lz_lanes consecutive LZ descriptors, one per lane
                int cnt = 0;
                while (j + cnt < A.nd && cnt < Y.lz_lanes && A.descs[j + cnt].calc == TSFX_LEMPEL_ZIV_COMPLEXITY) ++cnt;
                for (int q = 0; q < cnt; ++q) {                      // symbols of every position, all lanes
                    const int bins = A.descs[j + q].i0;
                    const double step = __ddiv_rn(__dsub_rn(vmax, vmin), (double)bins);
                    if (SMALL) {
                        unsigned char* sb = symbuf8 + (size_t)q * Y.npad;
                        for (int pos = lane; pos < n; pos += 32) sb[pos] = (unsigned char)lz_symbol((double)xs[pos], vmin, vmax, step, bins);
                    } else {
                        unsigned short* sb = symbuf + (size_t)q * Y.npad;
                        for (int pos = lane; pos < n; pos += 32) sb[pos] = (unsigned short)lz_symbol((double)xs[pos], vmin, vmax, step, bins);
                    }
                }
                __syncwarp();
                // phrase dictionary = prefix-closed trie stored as ONE open-addressing table of keys
                // (parent slot << 16 | symbol); a node's id is the slot its key lives in, the root is 0xffff
                {
                    unsigned* tab = reinterpret_cast<unsigned*>(trie);       // SMALL: two 16-bit keys per word
                    const int words = SMALL ? (cnt * Y.lz_hash) >> 1 : cnt * Y.lz_hash;
                    for (int q = lane; q < words; q += 32) tab[q] = 0xffffffffu;
                }
                __syncwarp();
                if (lane < cnt) {
                    const Desc d = A.descs[j + lane];
                    int phrases = 0;
                    if (SMALL) {
                        const unsigned char* sb = symbuf8 + (size_t)lane * Y.npad;
                        unsigned short* hkey = trie + (size_t)lane * Y.lz_hash;
                        const unsigned mask = (unsigned)Y.lz_hash - 1u;          // 256 slots: node ids fit 8 bits, the root is 256
                        unsigned node = 256u;
                        for (int pos = 0; pos < n; ++pos) {
                            const unsigned key = (node << 7) | (unsigned)sb[pos];
                            unsigned h = ((key * 0x9E3779B1u) >> 20) & mask;
                            unsigned k;
                            while ((k = hkey[h]) != key && k != 0xffffu) h = (h + 1u) & mask;
                            if (k == key) node = h;
                            else { hkey[h] = (unsigned short)key; ++phrases; node = 256u; }
                        }
                    } else {
                        const unsigned short* sb = symbuf + (size_t)lane * Y.npad;
                        unsigned* hkey = reinterpret_cast<unsigned*>(trie) + (size_t)lane * Y.lz_hash;
                        const unsigned mask = (unsigned)Y.lz_hash - 1u;
                        unsigned node = 0xffffu;
                        for (int pos = 0; pos < n; ++pos) {
                            const unsigned key = (node << 16) | (unsigned)sb[pos];
                            unsigned h = (key * 0x9E3779B1u) >> 15;
                            h &= mask;
                            unsigned k;
                            while ((k = hkey[h]) != key && k != 0xffffffffu) h = (h + 1u) & mask;
                            if (k == key) node = h;                      // phrase seen: extend it
                            else { hkey[h] = key; ++phrases; node = 0xffffu; }
                        }
                    }
                    orow[d.col] = (double)phrases / (double)n;
                }
                __syncwarp();
                j += cnt;
            } else if (d0.calc == TSFX_PERMUTATION_ENTROPY) {
                // run of permutation_entropy descriptors sharing tau: one pass over the windows serves all of
                // them (dimensions <= 6 through shared-memory histograms over the D! Lehmer indices)
                const int tau = d0.i0;
                int cnt = 0, bins_total = 0, Dh = 0;
                while (j + cnt < A.nd && A.descs[j + cnt].calc == TSFX_PERMUTATION_ENTROPY && A.descs[j + cnt].i0 == tau) {
                    const int D = A.descs[j + cnt].i1;
                    if (D <= 6) {
                        int f = 1;
                        for (int q = 2; q <= D; ++q) f *= q;
                        if (bins_total + f > Y.hist_cap) break;
                        bins_total += f;
                        Dh = max(Dh, D);
                    }
                    ++cnt;
                }
                if (cnt == 0) {             // a histogram that does not fit the `codes` area at all: cannot happen for
                    if (lane == 0) orow[d0.col] = dnan();      // dimensions <= 6 (720 bins <= hist_cap); never loop in place
                    ++j;
                    continue;
                }
                if (Dh > 0) {
                    for (int b = lane; b < (SMALL ? (bins_total + 1) >> 1 : bins_total); b += 32) codes[b] = 0u;
                    __syncwarp();
                    const int Wmax = (n >= 2) ? (n - 2) / tau + 1 : 0;          // windows of the smallest dimension
                    for (int k = lane; k < Wmax; k += 32) {
                        const int st = k * tau;
                        const unsigned bits = pe_order_bits(xs + st, min(8, n - st));
                        int off = 0;
                        for (int t = 0; t < cnt; ++t) {
                            const int D = A.descs[j + t].i1;
                            if (D > 6) continue;
                            int f = 1;
                            for (int q = 2; q <= D; ++q) f *= q;
                            if (st + D <= n) {
                                const unsigned bin = off + pe_lehmer(bits, D);
                                if (SMALL) atomicAdd(&codes[bin >> 1], (bin & 1u) ? 0x10000u : 1u);
                                else atomicAdd(&codes[bin], 1u);
                            }
                            off += f;
                        }
                    }
                    __syncwarp();
                    int off = 0;
                    for (int t = 0; t < cnt; ++t) {
                        const Desc d = A.descs[j + t];
                        const int D = d.i1;
                        if (D > 6) continue;
                        int f = 1;
                        for (int q = 2; q <= D; ++q) f *= q;
                        double r = dnan();
                        if (n >= D) {
                            const int W = (n - D) / tau + 1;
                            // -sum p ln p = ln W - (1/W) sum c ln c  (bins with c = 1 contribute nothing)
                            double acc = 0.0;
                            for (int b = lane; b < f; b += 32) {
                                const unsigned c = SMALL ? (codes[(off + b) >> 1] >> (16 * ((off + b) & 1))) & 0xffffu : codes[off + b];
                                if (c > 1u) acc += c < 64u ? clogc_small[c] : (double)c * log((double)c);
                            }
                            r = log((double)W) - wsum(acc) / (double)W;
                        }
                        if (lane == 0) orow[d.col] = r;
                        off += f;
                    }
                    __syncwarp();
                }
                for (int t = 0; t < cnt; ++t) {             // dimensions 7, 8: sort the indices, count run lengths
                    const Desc d = A.descs[j + t];
                    const int D = d.i1;
                    if (D <= 6) continue;
                    double r = dnan();
                    if (n >= D) {
                        const int W = (n - D) / tau + 1;
                        int m = 2;
                        while (m < W) m <<= 1;
                        for (int k = lane; k < m; k += 32)
                            codes[k] = (k < W) ? pe_lehmer(pe_order_bits(xs + k * tau, D), D) : 0xffffffffu;
                        __syncwarp();
                        warp_bitonic_sort_u32(codes, m, lane);
                        double acc = 0.0;
                        for (int k = lane; k < W; k += 32) {
                            const unsigned c = codes[k];
                            if ((k == 0 || codes[k - 1] != c) && k + 1 < W && codes[k + 1] == c) {
                                int len = 2;
                                while (k + len < W && codes[k + len] == c) ++len;
                                acc += len < 64 ? clogc_small[len] : (double)len * log((double)len);
                            }
                        }
                        r = log((double)W) - wsum(acc) / (double)W;
                        __syncwarp();
                    }
                    if (lane == 0) orow[d.col] = r;
                }
                j += cnt;
            } else {
                if (lane == 0) orow[d0.col] = dnan();
                ++j;
            }
        }
        __syncwarp();
    }
}

template <int WPC, bool GS>
__global__ void __launch_bounds__(WPC * 32) k_seq(SeqArgs A, SeqLayout Y) { seq_body<WPC, GS, false>(A, Y); }

template <int WPC, bool GS>
__global__ void __launch_bounds__(WPC * 32, (WPC == 4 ? 8 : 1)) k_seq_small(SeqArgs A, SeqLayout Y) { seq_body<WPC, GS, true>(A, Y); }

template <int WPC, bool GS>
__global__ void __launch_bounds__(WPC * 32) k_peaks(SeqArgs A, SeqLayout Y) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned char* base = warp_region<GS>(smem_raw, A.gscratch, A.bytes_per_warp, WPC, warp);
    double* row0 = reinterpret_cast<double*>(base);                       // npad : width-1 row (float64)
    double* tmp = row0 + Y.npad;                                           // npad : the row being formed
    double* noise = reinterpret_cast<double*>(base + Y.off_noise);         // npad : memoised noise floor (NaN = not yet)
    float* rowsf = reinterpret_cast<float*>(base + Y.off_rowsf);           // (cwt_n - 1) x npad : wider rows, float32 copies
    double* hw = reinterpret_cast<double*>(base + Y.off_hw);
    // ridge-line bookkeeping is a chain of dependent small-table lookups: from the global region every one of them is
    // an L2 round trip (the hottest stalls of the kernel), so these tables get their own shared-memory slice
    unsigned char* hot = (GS && Y.hot_bytes > 0) ? smem_raw + (size_t)warp * Y.hot_bytes : nullptr;
    unsigned* maxbits = hot ? reinterpret_cast<unsigned*>(hot + Y.hot_bits) : reinterpret_cast<unsigned*>(base + Y.off_bits);
    short* lines = hot ? reinterpret_cast<short*>(hot + Y.hot_lines) : reinterpret_cast<short*>(base + Y.off_lines);
    int* colmap = hot ? reinterpret_cast<int*>(hot + Y.hot_map) : reinterpret_cast<int*>(base + Y.off_map);
    float* xs = reinterpret_cast<float*>(base + Y.off_xs);
    double* xd = reinterpret_cast<double*>(base + Y.off_xd);               // zero-padded float64 copy for the convolutions
    const int64_t warps_total = (int64_t)gridDim.x * WPC;
    const int LCAP = Y.npad + Y.npad / 2 + 32;   // alive (<= maxima of the two previous rows <= n) + new in this row (<= n/2)

    for (int64_t s = (int64_t)blockIdx.x * WPC + warp; s < A.R.n_series; s += warps_total) {
        const int n = load_series(A.R, s, xs, lane);
        double* orow = A.out + (size_t)s * A.ncols;
        bool cwt_ready = false;

        int j = 0;
        while (j < A.nd) {
            const Desc d0 = A.descs[j];
            if (d0.calc == TSFX_NUMBER_CWT_PEAKS) {
                if (!cwt_ready) {
                    for (int p = lane; p < Y.nxd; p += 32) {
                        const int t = p - TSFX_MAXW_PTS;
                        xd[p] = (t >= 0 && t < n) ? (double)xs[t] : 0.0;
                    }
                    __syncwarp();
                    // all rows 1..cwt_n once (kept in shared memory) + local-maximum bit masks per row
                    for (int w = 1; w <= Y.cwt_n; ++w) {
                        const int npts = min(10 * w, n);
                        ricker_fill(hw, npts, w, lane);
                        double* dst = (w == 1) ? row0 : tmp;
                        cwt_row(xd, n, hw, npts, dst, lane);
                        __syncwarp();
                        unsigned* bits = maxbits + (size_t)(w - 1) * Y.nwords;
                        for (int b0 = 0; b0 < n; b0 += 32) {
                            int i = b0 + lane;
                            bool mx = false;
                            if (i < n) {
                                double v = dst[i];
                                double pl = dst[min(i + 1, n - 1)], mi = dst[max(i - 1, 0)];
                                mx = (v > pl) && (v > mi);
                                if (w > 1) rowsf[(size_t)(w - 2) * Y.npad + i] = (float)v;   // only read for the SNR test
                            }
                            unsigned word = __ballot_sync(FULL, mx);
                            if (lane == 0) bits[b0 >> 5] = word;
                        }
                        __syncwarp();
                    }
                    for (int c = lane; c < n; c += 32) noise[c] = dnan();
                    __syncwarp();
                    cwt_ready = true;
                }
                const int nrows = d0.i0;
                // ---- ridge lines (scipy _identify_ridge_lines + _filter_ridge_lines), warp-parallel ----
                // line table (list order = creation order, as in scipy's Python list)
                short* l_last = lines;                 // last attached column
                short* l_gap = lines + LCAP;
                short* l_len = lines + 2 * LCAP;
                short* l_minrow = lines + 3 * LCAP;    // smallest row so far
                short* l_mincol = lines + 4 * LCAP;    // first column attached at that row
                int* t_max = reinterpret_cast<int*>(lines + 5 * LCAP);   // per-row attachment summaries
                int* t_min = t_max + LCAP;
                int* t_cnt = t_min + LCAP;
                const int min_length = (nrows + 3) / 4;                       // ceil(nrows / 4)
                const unsigned lt = (1u << lane) - 1u;
                const int NONE = 0x7fffffff;
                int result = 0, nl = 0, start = -1;
                for (int r = nrows - 1; r >= 0 && start < 0; --r) {             // largest row with any maximum
                    const unsigned* bits = maxbits + (size_t)r * Y.nwords;
                    unsigned any = 0;
                    for (int wd = lane; wd * 32 < n; wd += 32) any |= bits[wd];
                    if (__any_sync(FULL, any != 0)) start = r;
                }
                if (start >= 0) {
                    const unsigned* bits = maxbits + (size_t)start * Y.nwords;
                    for (int b0 = 0; b0 < n; b0 += 32) {
                        const unsigned word = bits[b0 >> 5];
                        const int idx = nl + __popc(word & lt);
                        if (((word >> lane) & 1u) && idx < LCAP) {
                            const int c = b0 + lane;
                            l_last[idx] = (short)c; l_gap[idx] = 0; l_len[idx] = 1; l_minrow[idx] = (short)start; l_mincol[idx] = (short)c;
                        }
                        nl = min(nl + __popc(word), LCAP);
                    }
                }
                __syncwarp();
                // filter of _filter_ridge_lines for one finished line
                const int window = (n + 19) / 20, hf = window / 2, odd = window & 1;
                auto accept = [&](int len, int rr, int cc) -> bool {
                    if (len < min_length) return false;
                    double nz = noise[cc];
                    if (nz != nz) {                 // 10th percentile of row 0 around cc, formed on first use
                        const int ws = max(cc - hf, 0), we = min(cc + hf + odd, n);
                        nz = percentile10(row0 + ws, we - ws);
                        noise[cc] = nz;
                    }
                    const double val = (rr == 0) ? row0[cc] : (double)rowsf[(size_t)(rr - 1) * Y.npad + cc];
                    const double snr = fabs(val / nz);
                    return !(snr < 1.0);
                };
                for (int r = start - 1; r >= 0; --r) {
                    const unsigned* bits = maxbits + (size_t)r * Y.nwords;
                    const int maxd = (r + 1) / 4;                  // floor(widths[r] / 4); distances are integers
                    for (int c = lane; c < n; c += 32) colmap[c] = NONE;
                    for (int li = lane; li < nl; li += 32) { t_max[li] = -1; t_min[li] = NONE; t_cnt[li] = 0; l_gap[li] += 1; }
                    __syncwarp();
                    // snapshot: column -> first line (list order) whose last column is that column
                    for (int li = lane; li < nl; li += 32) atomicMin(&colmap[l_last[li]], li);
                    __syncwarp();
                    const int nl_snapshot = nl;
                    for (int b0 = 0; b0 < n; b0 += 32) {
                        const unsigned word = bits[b0 >> 5];
                        const bool mine = (word >> lane) & 1u;
                        const int c = b0 + lane;
                        int best = -1;
                        if (mine && nl_snapshot > 0) {
                            // np.argmin(|c - prev|): smallest distance, first in list order on ties; attach only
                            // when that distance is <= max_distances[row]
                            for (int dd = 0; dd <= maxd && best < 0; ++dd) {
                                const int a = (c - dd >= 0) ? colmap[c - dd] : NONE;
                                const int b = (dd > 0 && c + dd < n) ? colmap[c + dd] : NONE;
                                const int m = min(a, b);
                                if (m != NONE) best = m;
                            }
                        }
                        if (mine && best >= 0) { atomicMax(&t_max[best], c); atomicMin(&t_min[best], c); atomicAdd(&t_cnt[best], 1); }
                        const unsigned newm = __ballot_sync(FULL, mine && best < 0);
                        if (mine && best < 0) {
                            const int idx = nl + __popc(newm & lt);
                            if (idx < LCAP) { l_last[idx] = (short)c; l_gap[idx] = 0; l_len[idx] = 1; l_minrow[idx] = (short)r; l_mincol[idx] = (short)c; }
                        }
                        nl = min(nl + __popc(newm), LCAP);
                    }
                    __syncwarp();
                    for (int li = lane; li < nl_snapshot; li += 32) {
                        const int cnt = t_cnt[li];
                        if (cnt > 0) {      // points are appended in ascending column order within a row
                            l_last[li] = (short)t_max[li]; l_gap[li] = 0; l_len[li] = (short)(l_len[li] + cnt);
                            l_minrow[li] = (short)r; l_mincol[li] = (short)t_min[li];
                        }
                    }
                    __syncwarp();
                    // retire lines whose gap exceeds gap_thresh = ceil(widths[0]) = 1; survivors keep their order
                    int keep = 0;
                    for (int b0 = 0; b0 < nl; b0 += 32) {
                        const int li = b0 + lane;
                        const bool valid = li < nl;
                        short f_last = 0, f_gap = 0, f_len = 0, f_row = 0, f_col = 0;
                        if (valid) { f_last = l_last[li]; f_gap = l_gap[li]; f_len = l_len[li]; f_row = l_minrow[li]; f_col = l_mincol[li]; }
                        const bool retire = valid && f_gap > 1;
                        const bool ok = retire && accept(f_len, f_row, f_col);
                        result += __popc(__ballot_sync(FULL, ok));
                        const unsigned keepm = __ballot_sync(FULL, valid && !retire);
                        __syncwarp();
                        if (valid && !retire) {
                            const int dst = keep + __popc(keepm & lt);
                            l_last[dst] = f_last; l_gap[dst] = f_gap; l_len[dst] = f_len; l_minrow[dst] = f_row; l_mincol[dst] = f_col;
                        }
                        keep += __popc(keepm);
                        __syncwarp();
                    }
                    nl = keep;
                }
                for (int b0 = 0; b0 < nl; b0 += 32) {
                    const int li = b0 + lane;
                    const bool ok = li < nl && accept(l_len[li], l_minrow[li], l_mincol[li]);
                    result += __popc(__ballot_sync(FULL, ok));
                }
                if (lane == 0) orow[d0.col] = (double)result;
                __syncwarp();
                ++j;
            } else {
                if (lane == 0) orow[d0.col] = dnan();
                ++j;
            }
        }
        __syncwarp();
    }
}

// lempel_ziv_complexity + permutation_entropy
cudaError_t launch_seq(const SeqArgs& A0, int max_len, cudaStream_t st, int sm_count) {
    SeqArgs A = A0;
    A.npad = (max_len + 3) & ~3;
    if (max_len > 21000) return cudaErrorInvalidConfiguration;      // LZ node ids are 15-bit slot indices
    SeqLayout Y = {};
    Y.npad = A.npad;
    int p2 = 2;
    while (p2 < max_len) p2 <<= 1;
    Y.npow2 = std::max(p2, 1024);                 // >= 6! = 720 so dimensions up to 6 use the histogram path
    Y.hist_cap = Y.npow2;
    const bool need_lz = (A.nscr & 1) != 0, need_perm = (A.nscr & 2) != 0;
    Y.lz_lanes = need_lz ? std::min(LZ_LANES, std::max(1, (A.nscr >> 16) & 0xff)) : 0;
    Y.lz_hash = 4;
    while (Y.lz_hash < A.npad + A.npad / 2 + 2) Y.lz_hash <<= 1;      // load factor <= 2/3 in the worst case
    Y.lz_stride = 2 * Y.lz_hash;                  // uint16 units: one uint32 key per slot
    {
        // compact shared-memory layout (k_seq_small) where it fits: measured on B200 at 1 M x 256, 35.3 -> 26.8 ms
        // against the general kernel below (profiles/r2_notes.md)
        const int max_bins = (A.nscr >> 24) & 0xff;
        if (max_len <= 256 && max_bins <= 127) {
            Y.lz_hash = 256;
            Y.npow2 = 256;                                   // sort path of dimensions 7, 8: <= 256 windows
            Y.hist_cap = 896;                                // 1792 bytes of packed 16-bit counters
            size_t o = 0;
            Y.off_codes = (int)o; o += need_perm ? (size_t)1792 : 0;     // 870 packed 16-bit bins (dimensions 3..6), or 256 sort keys
            Y.off_trie = (int)o;  o += (size_t)Y.lz_lanes * Y.lz_hash * 2;
            Y.off_sym = (int)o;   o += (size_t)Y.lz_lanes * A.npad;
            o = (o + 15) & ~(size_t)15;
            Y.off_xs = (int)o;    o += (size_t)A.npad * 4;
            const size_t per = (o + 15) & ~(size_t)15;
            A.bytes_per_warp = (int)per;
            Geometry G;
            G.wpc = 4; G.smem = per * 4; G.gscratch = nullptr;
            const int64_t ctas = (A.R.n_series + 3) / 4;
            const int64_t cap = (int64_t)sm_count * 4096;
            G.grid = (int)std::max<int64_t>(1, std::min(ctas, cap));
            A.gscratch = nullptr;
            cudaError_t e = cudaFuncSetAttribute(k_seq_small<4, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)G.smem);
            if (e != cudaSuccess) return e;
            k_seq_small<4, false><<<G.grid, 4 * 32, G.smem, st>>>(A, Y);
            return cudaGetLastError();
        }
    }
    size_t off = 0;
    Y.off_codes = (int)off; off += need_perm ? (size_t)Y.npow2 * 4 : 0;
    Y.off_trie = (int)off;  off += (size_t)Y.lz_lanes * Y.lz_stride * 2;
    off = (off + 3) & ~(size_t)3;
    Y.off_sym = (int)off;   off += (size_t)Y.lz_lanes * A.npad * 2;
    off = (off + 15) & ~(size_t)15;
    Y.off_xs = (int)off;    off += (size_t)A.npad * 4;
    size_t per = (off + 15) & ~(size_t)15;
    A.bytes_per_warp = (int)per;
    Geometry G;
    if (!plan_geometry(per, 72 * 1024, 8, A.R.n_series, sm_count, A.gscratch, A.gscratch_bytes, &G, 16 * 1024, 8)) return cudaErrorInvalidConfiguration;
    A.gscratch = G.gscratch;
    TSFX_DISPATCH(k_seq, G, st, A, Y)
    return cudaGetLastError();
}

// number_cwt_peaks
cudaError_t launch_peaks(const SeqArgs& A0, int max_len, cudaStream_t st, int sm_count) {
    SeqArgs A = A0;
    A.npad = (max_len + 3) & ~3;
    if (max_len > 32000) return cudaErrorInvalidConfiguration;      // int16 line tables
    SeqLayout Y = {};
    Y.npad = A.npad;
    Y.nwords = (A.npad + 31) / 32 + 1;
    Y.cwt_n = (A.nscr >> 8) & 0xff;
    size_t off = 0;
    off += (size_t)2 * A.npad * 8;                          // row0 + tmp (float64)
    Y.off_noise = (int)off; off += (size_t)A.npad * 8;
    Y.off_hw = (int)off;    off += (size_t)TSFX_MAXW_PTS * 8;
    Y.off_bits = (int)off;  off += (size_t)Y.cwt_n * Y.nwords * 4;
    off = (off + 3) & ~(size_t)3;
    Y.off_rowsf = (int)off; off += (size_t)std::max(Y.cwt_n - 1, 0) * A.npad * 4;
    Y.off_lines = (int)off; off += (size_t)(A.npad + A.npad / 2 + 32) * (5 * 2 + 3 * 4);    // 5 int16 + 3 int32 tables of LCAP lines
    Y.off_map = (int)off;   off += (size_t)A.npad * 4;
    off = (off + 15) & ~(size_t)15;
    Y.off_xs = (int)off;    off += (size_t)A.npad * 4;
    off = (off + 15) & ~(size_t)15;
    Y.nxd = ((max_len + 255) / 256) * 256 + 2 * TSFX_MAXW_PTS;
    Y.off_xd = (int)off;    off += (size_t)Y.nxd * 8;
    size_t per = (off + 15) & ~(size_t)15;
    A.bytes_per_warp = (int)per;
    Geometry G;
    if (!plan_geometry(per, 72 * 1024, 8, A.R.n_series, sm_count, A.gscratch, A.gscratch_bytes, &G, 16 * 1024)) return cudaErrorInvalidConfiguration;
    A.gscratch = G.gscratch;
    if (G.gscratch) {
        // hybrid placement: bulk rows in the global (L2-resident) region, hot tables in shared memory when four CTAs
        // per SM still fit
        const size_t lines_b = (size_t)(A.npad + A.npad / 2 + 32) * (5 * 2 + 3 * 4);
        const size_t map_b = (size_t)A.npad * 4, bits_b = (size_t)Y.cwt_n * Y.nwords * 4;
        size_t hot = ((lines_b + 15) & ~(size_t)15) + ((map_b + 15) & ~(size_t)15) + ((bits_b + 15) & ~(size_t)15);
        if (hot * G.wpc <= 54 * 1024) {
            Y.hot_lines = 0;
            Y.hot_map = (int)((lines_b + 15) & ~(size_t)15);
            Y.hot_bits = Y.hot_map + (int)((map_b + 15) & ~(size_t)15);
            Y.hot_bytes = (int)hot;
            G.smem = hot * G.wpc;
        }
    }
    TSFX_DISPATCH(k_peaks, G, st, A, Y)
    return cudaGetLastError();
}

}  // namespace tsfx
