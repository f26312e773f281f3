// tsfx_kernels.h -- argument blocks and launchers of the kernel groups (internal to libtsfx.so).
#pragma once
#include <cuda_runtime.h>
#include "tsfx_common.cuh"

#define TSFX_DEC_MIN (-46)
#define TSFX_DEC_MAX 39

namespace tsfx {

struct Geometry { int wpc; size_t smem; int grid; unsigned char* gscratch; };

// Chooses warps per CTA / grid for a warp-per-series kernel needing `per` bytes per warp.  Shared memory when it
// fits (budget = target bytes per CTA so several CTAs stay resident), else the global scratch buffer.
inline bool plan_geometry(size_t per, size_t budget, int maxw, int64_t n_series, int sm_count, unsigned char* gs,
                          size_t gs_bytes, Geometry* G, size_t prefer_global_above = 227 * 1024,
                          int global_ctas = 0) {
    // Working sets above `prefer_global_above` bytes per warp run from the global (L2-resident) region even though
    // they would fit in shared memory: measured on B200, the latency-bound PEAKS / SEQ kernels are up to 5x faster
    // that way at 1024 samples because shared memory would limit them to 2-4 warps per SM (profiles/r1_notes.md).
    if (per <= prefer_global_above && per <= 227 * 1024) {
        size_t w = budget / per;
        int wpc = w >= 8 ? 8 : w >= 4 ? 4 : w >= 2 ? 2 : 1;
        while (wpc > maxw) wpc >>= 1;
        G->wpc = wpc;
        G->smem = per * wpc;
        int64_t cap = (int64_t)sm_count * 4096;      // CTAs per SM: each CTA loops over its share of the series
        int64_t ctas = (n_series + wpc - 1) / wpc;
        G->grid = (int)(ctas < cap ? (ctas < 1 ? 1 : ctas) : cap);
        G->gscratch = nullptr;
        return true;
    }
    int wpc = maxw >= 4 ? 4 : 1;
    size_t max_ctas = gs ? gs_bytes / (per * wpc) : 0;
    if (max_ctas < 1) { wpc = 1; max_ctas = gs ? gs_bytes / per : 0; }
    if (max_ctas < 1) return false;
    int64_t ctas = (n_series + wpc - 1) / wpc;
    // CTAs per SM in global-region mode: the kernel's own choice, else 4
    int64_t cap = (int64_t)sm_count * (global_ctas > 0 ? global_ctas : 4);
    if ((int64_t)max_ctas < cap) cap = (int64_t)max_ctas;
    G->wpc = wpc;
    G->smem = 0;
    G->grid = (int)(ctas < cap ? (ctas < 1 ? 1 : ctas) : cap);
    G->gscratch = gs;
    return true;
}

#define TSFX_LAUNCH_GEOM(KERNEL, W, GS, G, st, ...)                                                               \
    {                                                                                                             \
        if ((G).smem) {                                                                                           \
            cudaError_t e__ = cudaFuncSetAttribute(KERNEL<W, GS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(G).smem); \
            if (e__ != cudaSuccess) return e__;                                                                   \
        }                                                                                                         \
        KERNEL<W, GS><<<(G).grid, W * 32, (G).smem, st>>>(__VA_ARGS__);                                           \
    }
// shared-memory instantiations for 8/4/2/1 warps per CTA, global-scratch instantiations for 4/1
#define TSFX_DISPATCH(KERNEL, G, st, ...)                                                   \
    if ((G).gscratch) {                                                                     \
        if ((G).wpc == 4) TSFX_LAUNCH_GEOM(KERNEL, 4, true, G, st, __VA_ARGS__)             \
        else TSFX_LAUNCH_GEOM(KERNEL, 1, true, G, st, __VA_ARGS__)                          \
    } else switch ((G).wpc) {                                                               \
        case 8: TSFX_LAUNCH_GEOM(KERNEL, 8, false, G, st, __VA_ARGS__) break;               \
        case 4: TSFX_LAUNCH_GEOM(KERNEL, 4, false, G, st, __VA_ARGS__) break;               \
        case 2: TSFX_LAUNCH_GEOM(KERNEL, 2, false, G, st, __VA_ARGS__) break;               \
        default: TSFX_LAUNCH_GEOM(KERNEL, 1, false, G, st, __VA_ARGS__) break;              \
    }

enum Group { G_BASIC = 0, G_SORTED, G_SPECTRAL, G_LA, G_ENTROPY, G_SEQ, G_PEAKS, G_COUNT };
#define G_EVENTS (G_COUNT + 1)      // + the assemble pass

// Result assembly: every kernel group writes its own dense [n_series x ncols_g] staging matrix (so each
// 32-byte sector is completed by the warp that owns the row, while it is still in L2); this pass
// scatters the staging rows into the final row-major [n_series x ncols] matrix in column order.
struct AssembleArgs {
    const double* stage;          // group g starts at stage + n_series * cum[g]
    double* out;
    int64_t n_series;
    int ncols;                    // columns of this plan
    int ld;                       // row stride of `out` (>= ncols: several kinds share one matrix, each its own column block)
    int n_groups;
    int cum[G_COUNT + 1];         // columns before group g (cum[n_groups] = total staged columns)
    const int32_t* final_col;     // device: final column of staged column (cum[g] + j)
    // multi-GPU result placement (tsfx_set_peer_outputs): the finished row is ALSO stored at the same offset of
    // every peer's mapped result matrix (plain P2P stores over NVLink), or -- when the result matrix has a multicast
    // mapping -- stored once through it (the NVSwitch replicates the store to every GPU, including this one)
    int n_extra;
    double* extra[7];
    double* out_mc;               // non-null: store through the multicast mapping instead of `out`
};
cudaError_t launch_assemble(const AssembleArgs& A, cudaStream_t st, int sm_count);

struct BasicArgs {
    SeriesRef R;
    unsigned char* gscratch;     // global scratch (API) -> set to nullptr by the launcher when shared memory is used
    size_t gscratch_bytes;
    const Desc* descs;   // device, this group's descriptors
    int nd;
    double* out;
    int ncols;
    int npad, nscr, nlag, bytes_per_warp;   // shared-memory carve-up (doubles / doubles / doubles / bytes)
    int lag_tiles;       // > 0: lag products by DMMA (mma.sync m8n8k4 f64) with this many 8 x 8 tiles; 0: FMA path
    int desc_bytes;      // CTA-wide copy of the descriptor table in front of the per-warp regions (set by the launcher)
    int nxc, nalt;       // doubles of the centred copy incl. its zero tail; distinct agg_linear_trend (f_agg, chunk_len) keys
    int nfin;            // the first nfin descriptors are O(1) "finishers" (see k_basic.cu)
    int lag_needed;      // largest lag product any descriptor reads (0 = none)
    int pacf_off;        // offset (doubles) of the pacf staging area inside lagS
    const double* dec;   // device table d*10^k, k = TSFX_DEC_MIN..TSFX_DEC_MAX, 9 per decade
};
cudaError_t launch_basic(const BasicArgs& A, int max_len, cudaStream_t st, int sm_count);
bool basic_finisher_calc(int calc);
bool sorted_finisher_calc(int calc);    // same for the SORTED group     // host: is this calculator evaluated by the lane-parallel finisher stage?

// reduction-only fast path of the BASIC group (k_moments.cu)
struct MomentsArgs {
    SeriesRef R;
    const Desc* descs;   // device, the BASIC group's descriptors (all moments_only_calc)
    int nd;
    double* out;         // staging matrix (colmap == nullptr: column = descriptor index) or the final matrix
    int ncols;           // row stride of `out`
    const int32_t* colmap;   // device: final column of descriptor j (direct write, no assemble pass), or nullptr
    int need_high;       // third / fourth centred moments are needed (skewness, kurtosis)
};
cudaError_t launch_moments(const MomentsArgs& A, cudaStream_t st, int sm_count);
bool moments_only_calc(int calc);       // host: can the reduction-only kernel evaluate this calculator?

struct SortedArgs {
    SeriesRef R;
    unsigned char* gscratch;     // global scratch (API) -> set to nullptr by the launcher when shared memory is used
    size_t gscratch_bytes;
    const Desc* descs;
    int nd;
    double* out;
    int ncols;
    int npad, npow2, nscr, bytes_per_warp;
    int nfin, ncq;       // leading O(1) descriptors (lane-parallel); distinct change_quantiles corridors
};
cudaError_t launch_sorted(const SortedArgs& A, int max_len, cudaStream_t st, int sm_count);

struct SpectralArgs {
    SeriesRef R;
    unsigned char* gscratch;     // global scratch (API) -> set to nullptr by the launcher when shared memory is used
    size_t gscratch_bytes;
    const Desc* descs;
    int nd;
    double* out;
    int ncols;
    int npad, nspec, bytes_per_warp;
    const double2* twiddle;    // device: exp(-2 pi i k / tw_n), k = 0 .. tw_n/2
    int tw_n;                  // power of two >= largest power-of-two FFT length in use
    const double* tables;      // cwt tables (device)
    const int64_t* table_off;
    const int32_t* table_half;
    int need_fft, need_welch;
    int max_hist;
    int nfft;                  // the first nfft descriptors are fft_coefficient (lane-parallel stage)
};
cudaError_t launch_spectral(const SpectralArgs& A, int max_len, cudaStream_t st, int sm_count);

struct LaArgs {
    SeriesRef R;
    unsigned char* gscratch;     // global scratch (API) -> set to nullptr by the launcher when shared memory is used
    size_t gscratch_bytes;
    const Desc* descs;
    int nd;
    double* out;
    int ncols;
    int npad, nscr, bytes_per_warp;
};
cudaError_t launch_la(const LaArgs& A, int max_len, cudaStream_t st, int sm_count);

struct EntropyArgs {
    int xpad;                  // padded sample count of the bit-tile kernel
    SeriesRef R;
    unsigned char* gscratch;     // global scratch (API) -> set to nullptr by the launcher when shared memory is used
    size_t gscratch_bytes;
    const Desc* descs;
    int nd;
    double* out;
    int ncols;
    int npad, bytes_per_warp;
};
cudaError_t launch_entropy(const EntropyArgs& A, int max_len, cudaStream_t st, int sm_count);

struct SeqArgs {
    SeriesRef R;
    unsigned char* gscratch;     // global scratch (API) -> set to nullptr by the launcher when shared memory is used
    size_t gscratch_bytes;
    const Desc* descs;
    int nd;
    double* out;
    int ncols;
    int npad, nscr, bytes_per_warp;
};
cudaError_t launch_seq(const SeqArgs& A, int max_len, cudaStream_t st, int sm_count);
cudaError_t launch_peaks(const SeqArgs& A, int max_len, cudaStream_t st, int sm_count);

// plain fill of a column set with NaN is done by BASIC (TSFX_CONST_NAN)

// twiddle table fill: tw[k] = exp(-2 pi i k / n), k = 0..n/2
cudaError_t launch_fill_twiddle(double2* tw, int n, cudaStream_t st);

}  // namespace tsfx
