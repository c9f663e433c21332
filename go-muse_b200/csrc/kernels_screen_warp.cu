// kernels_screen_warp.cu -- instantiations of score_screen_warp_kernel<NZ> (muse_screen.cuh), n = 2048.
#include "muse_launch.h"

namespace muse {

// one instantiation per number of non-zero rows of 32 complex slots (N = 1026 .. 2048)
cudaError_t launch_screen_warp(const ScreenParams &p, int sm_count, cudaStream_t st) {
    using C = ScreenWarpCfg;
    return dispatch_nz(C::nz(p.N), [&](auto nz) {
        return launch_persistent(score_screen_warp_kernel<decltype(nz)::value>, p.count, C::warps(p.N), C::smem_bytes(p.N), sm_count, st, p,
                                 (unsigned)C::warp_bytes(p.N), (unsigned)C::row_bytes(p.N));
    });
}

}  // namespace muse
