// muse_launch.h -- host-side launchers of the templated score kernels.  Each family of instantiations is its own
// translation unit (kernels_*.cu) so that the library builds in parallel; muse_api.cu sees only these entry points.
#pragma once

#include <cuda_runtime.h>

#include <type_traits>

#include "muse_exact.cuh"
#include "muse_screen_big.cuh"
#include "muse_screen_sub.cuh"
#include "muse_screen_multi.cuh"
#include "muse_bounds_tc.cuh"

namespace muse {

// score_exact_kernel<log2m, ., mode> (muse_exact.cuh); log2m = log2(n/2) in 0 .. 13
cudaError_t launch_exact(int mode, int log2m, const ExactParams &p, cudaStream_t st);
cudaError_t launch_exact_batch(int mode, const ExactParams *d_table, int nq, int64_t max_count, cudaStream_t st);
// points per thread of the exact kernel for each FFT size (fixes the twiddle layout of ExactParams::twM)
inline int exact_log2p(int log2m) { return log2m < 4 ? log2m : 4; }

// f(std::integral_constant<int, NZ>()) for nz = NZ in 17 .. 32: the rows of complex slots that hold samples, one
// instantiation of the n <= 2048 kernels per value
template <typename F>
cudaError_t dispatch_nz(int nz, F &&f) {
    switch (nz) {
#define MUSE_NZ_CASE(z) case z: return f(std::integral_constant<int, z>());
        MUSE_NZ_CASE(17) MUSE_NZ_CASE(18) MUSE_NZ_CASE(19) MUSE_NZ_CASE(20) MUSE_NZ_CASE(21) MUSE_NZ_CASE(22)
        MUSE_NZ_CASE(23) MUSE_NZ_CASE(24) MUSE_NZ_CASE(25) MUSE_NZ_CASE(26) MUSE_NZ_CASE(27) MUSE_NZ_CASE(28)
        MUSE_NZ_CASE(29) MUSE_NZ_CASE(30) MUSE_NZ_CASE(31) MUSE_NZ_CASE(32)
#undef MUSE_NZ_CASE
    }
    return cudaErrorInvalidValue;
}

// persistent grid of blocks of `warps` warps: one per SM, fewer when `units` (one per warp) fill fewer
inline int64_t persistent_blocks(int64_t units, int warps, int sm_count) {
    const int64_t blocks = (units + warps - 1) / warps;
    return blocks > sm_count ? sm_count : blocks;
}
template <typename... P, typename... A>
cudaError_t launch_persistent(void (*kern)(P...), int64_t units, int warps, size_t smem, int sm_count, cudaStream_t st, A... args) {
    const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kern<<<(unsigned)persistent_blocks(units, warps, sm_count), warps * 32, smem, st>>>(args...);
    return cudaGetLastError();
}

// fp32 screening + fused second stage: warp kernel (n = 2048)
cudaError_t launch_screen_warp(const ScreenParams &p, int sm_count, cudaStream_t st);
// n = 128 .. 1024: sixteen .. two series per warp (muse_screen_sub.cuh); LOG2T = log2m - 5 = 1 .. 4, one per translation
// unit (kernels_screen_sub<LOG2T>.cu)
template <int LOG2T>
cudaError_t launch_screen_sub(const ScreenParams &p, int sm_count, cudaStream_t st) {
    using C = ScreenSubCfg<LOG2T>;
    return dispatch_nz(C::nz(p.N), [&](auto nz) {
        return launch_persistent(score_screen_sub_kernel<LOG2T, decltype(nz)::value>, (p.count + C::GS - 1) / C::GS, C::warps(p.N), C::smem_bytes(p.N),
                                 sm_count, st, p, (unsigned)C::warp_bytes(p.N), (unsigned)C::row_bytes(p.N));
    });
}
extern template cudaError_t launch_screen_sub<1>(const ScreenParams &, int, cudaStream_t);
extern template cudaError_t launch_screen_sub<2>(const ScreenParams &, int, cudaStream_t);
extern template cudaError_t launch_screen_sub<3>(const ScreenParams &, int, cudaStream_t);
extern template cudaError_t launch_screen_sub<4>(const ScreenParams &, int, cudaStream_t);
// n = 4096 .. 16384 (muse_screen_big.cuh)
cudaError_t launch_screen_big(int log2m, const ScreenParams &p, int sm_count, cudaStream_t st);
// n = 16384: nz = rows of 256 complex slots that hold samples, 17 .. 32, four per translation unit
cudaError_t launch_screen_big13_a(int nz, const ScreenParams &p, int sm_count, cudaStream_t st);
cudaError_t launch_screen_big13_b(int nz, const ScreenParams &p, int sm_count, cudaStream_t st);
cudaError_t launch_screen_big13_c(int nz, const ScreenParams &p, int sm_count, cudaStream_t st);
cudaError_t launch_screen_big13_d(int nz, const ScreenParams &p, int sm_count, cudaStream_t st);

// the second stage for up to RefineMultiCfg::QMAX queries with precomputed bounds (n = 2048)
cudaError_t launch_refine_multi(const ScreenParams &p, const MultiQuery *d_queries, int nq, int sm_count, unsigned *d_next, cudaStream_t st);
// many queries' bounds as one bf16 contraction on the tensor cores (muse_bounds_tc.cuh)
cudaError_t launch_mag_tiles(const ScreenParams &p, unsigned char *a_tiles, float *mid, int sm_count, cudaStream_t st);
cudaError_t launch_weight_tiles(const float4 *const *d_sw, int nq, unsigned char *b_tiles, cudaStream_t st);
cudaError_t launch_bounds_tc(const TcBoundsParams &p, cudaStream_t st);

// rows [first, first + count) of the slab slide forward by k samples in place, the k new samples of row first + i taken from
// d_add[i * k ..]; writes their RowStat and, for odd N, the pad column (kernels_roll.cu)
cudaError_t launch_roll_rows(double *slab, int64_t ld, int N, int64_t first, int64_t count, const double *d_add, int k,
                             RowStat *stat, int sm_count, cudaStream_t st);

// ---- series above n = 16384 (kernels_long.cu): Stockham passes through global memory, two series per transform ----
struct LongParams {
    const double *slab;      // [rows][ld] fp64
    int64_t ld;
    int64_t count;           // series to process
    const int32_t *idx;      // optional gather list
    int N;                   // series length
    int log2n;               // FFT length n = 2^log2n
    int signed_scores;
    const cd *X;             // FFT_n of the reference row / ((N-1) std n), n entries
    const cd *tw;            // exp(-2*pi*i*k/n), n entries
    double *out_score;       // MODE_SCORE: [rows]   MODE_CC: cc[n]
    int32_t *out_lag;
    cd *out_X;               // MODE_REF
    int32_t *out_flag;       // MODE_REF / MODE_CC: 1 when std == 0
    double *stats;           // set by launch_long (inside the work buffer)
};
size_t long_work_bytes(int log2n, long long chunk_pairs);
cudaError_t launch_long_twiddles(cd *tw, int log2n, cudaStream_t st);
cudaError_t launch_long(int mode, LongParams p, void *work, long long chunk_pairs, cudaStream_t st);
// generic xCorr through the same passes: L = nn (a power of two) or a power of two >= 2 nn
size_t long_xcorr_work_bytes(long long L);
cudaError_t launch_long_xcorr(const double *xp, const double *yp, long long nn, long long L, double scale, double *cc, void *work,
                              cudaStream_t st);

}  // namespace muse
