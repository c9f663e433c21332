// kernels_screen_multi.cu -- instantiations of refine_multi_kernel<NZ, LIST> (muse_screen_multi.cuh), n = 2048.
#include "muse_launch.h"

namespace muse {

cudaError_t launch_refine_multi(const ScreenParams &p, const MultiQuery *d_queries, int nq, int sm_count, unsigned *d_next, cudaStream_t st) {
    using C = RefineMultiCfg;
    return dispatch_nz(ScreenWarpCfg::nz(p.N), [&](auto nz) {
        auto kern = p.rows ? refine_multi_kernel<decltype(nz)::value, true> : refine_multi_kernel<decltype(nz)::value, false>;
        const int warps = C::warps(p.N);
        const size_t smem = C::smem_bytes(p.N);
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        const int64_t blocks = persistent_blocks(p.count, warps, sm_count);
        const unsigned first = (unsigned)(blocks * warps);      // the warps' own indices are taken: the counter hands out the rest
        e = cudaMemcpyAsync(d_next, &first, sizeof(first), cudaMemcpyHostToDevice, st);      // pageable source: left the host on return
        if (e != cudaSuccess) return e;
        kern<<<(unsigned)blocks, warps * 32, smem, st>>>(p, d_queries, nq, (unsigned)C::warp_bytes(p.N), d_next);
        return cudaGetLastError();
    });
}

}  // namespace muse
