// kernels_screen_big.cu -- instantiations of score_screen_big_kernel (muse_screen_big.cuh), n = 4096 .. 16384.
#include <algorithm>

#include "muse_launch.h"
#include "muse_screen_big.cuh"

namespace muse {

template <int LOG2M, int MINB>
static cudaError_t launch_screen_big_t(const ScreenParams &p, int sm_count, cudaStream_t st) {
    using C = ScreenBigCfg<LOG2M>;
    auto kern = score_screen_big_kernel<LOG2M, MINB, 0>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM);
    if (e != cudaSuccess) return e;
    int per_sm = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, C::T, C::SMEM);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) per_sm = 1;
    // persistent: every block walks a contiguous range of the series
    const int64_t blocks = std::min<int64_t>(p.count, (int64_t)sm_count * per_sm);
    kern<<<(unsigned)blocks, C::T, C::SMEM, st>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_screen_big(int log2m, const ScreenParams &p, int sm_count, cudaStream_t st) {
    switch (log2m) {
        case 13: {      // one instantiation per number of rows that hold samples (kernels_screen_big13_*.cu), MUSE_BIG_MINB13
                        // blocks of 256 threads per SM (2; 3 = an 80-register cap: measured, see DESIGN.md)
            const int nz = (((p.N + 1) >> 1) + ScreenBigCfg<13>::T - 1) / ScreenBigCfg<13>::T;
            if (nz >= 29) return launch_screen_big13_d(nz, p, sm_count, st);
            if (nz >= 25) return launch_screen_big13_c(nz, p, sm_count, st);
            if (nz >= 21) return launch_screen_big13_b(nz, p, sm_count, st);
            return launch_screen_big13_a(nz, p, sm_count, st);
        }
        case 12: return launch_screen_big_t<12, 4>(p, sm_count, st);
        case 11: return launch_screen_big_t<11, 8>(p, sm_count, st);
    }
    return cudaErrorInvalidValue;
}

}  // namespace muse
