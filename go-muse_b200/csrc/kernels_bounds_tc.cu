// kernels_bounds_tc.cu -- instantiations and launchers of muse_bounds_tc.cuh (the multi-query bounds on tcgen05).
#define MUSE_TC_KERNELS
#include "muse_launch.h"

namespace muse {

cudaError_t launch_mag_tiles(const ScreenParams &p, unsigned char *a_tiles, float *mid, int sm_count, cudaStream_t st) {
    using C = ScreenWarpCfg;
    const int warps = C::warps(p.N);
    const size_t wb = C::warp_bytes(p.N);
    return dispatch_nz(C::nz(p.N), [&](auto nz) {
        return launch_persistent(mag_tiles_kernel<decltype(nz)::value>, p.count, warps, (size_t)warps * wb, sm_count, st, p, a_tiles, mid,
                                 (unsigned)wb);
    });
}

cudaError_t launch_weight_tiles(const float4 *const *d_sw, int nq, unsigned char *b_tiles, cudaStream_t st) {
    const int n = TcCfg::TN * (TcCfg::K / 8);
    weight_tiles_kernel<<<(n + 255) / 256, 256, 0, st>>>(d_sw, nq, b_tiles);
    return cudaGetLastError();
}

cudaError_t launch_bounds_tc(const TcBoundsParams &p, cudaStream_t st) {
    cudaError_t e = cudaFuncSetAttribute(bounds_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TcCfg::SMEM);
    if (e != cudaSuccess) return e;
    const int64_t tiles = (p.S + TcCfg::TM - 1) / TcCfg::TM;
    bounds_tc_kernel<<<(unsigned)tiles, TcCfg::THREADS, TcCfg::SMEM, st>>>(p);
    return cudaGetLastError();
}

}  // namespace muse
