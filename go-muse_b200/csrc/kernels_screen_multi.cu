// kernels_screen_multi.cu -- instantiations of refine_multi_kernel<NZ> (muse_screen_multi.cuh), n = 2048.
#include "muse_launch.h"

namespace muse {

template <int NZ>
static cudaError_t launch_refine_multi_nz(const ScreenParams &p, const MultiQuery *d_queries, int nq, int sm_count, unsigned *d_next,
                                          cudaStream_t st) {
    using C = RefineMultiCfg;
    auto kern = refine_multi_kernel<NZ>;
    const int warps = C::warps(p.N);
    const size_t smem = C::smem_bytes(p.N);
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int64_t blocks = (p.count + warps - 1) / warps;      // persistent: one block per SM
    if (blocks > sm_count) blocks = sm_count;
    const unsigned first = (unsigned)(blocks * warps);      // the warps' own indices are taken: the counter hands out the rest
    e = cudaMemcpyAsync(d_next, &first, sizeof(first), cudaMemcpyHostToDevice, st);      // pageable source: left the host on return
    if (e != cudaSuccess) return e;
    kern<<<(unsigned)blocks, warps * 32, smem, st>>>(p, d_queries, nq, (unsigned)C::warp_bytes(p.N), d_next);
    return cudaGetLastError();
}

cudaError_t launch_refine_multi(const ScreenParams &p, const MultiQuery *d_queries, int nq, int sm_count, unsigned *d_next, cudaStream_t st) {
    switch (ScreenWarpCfg::nz(p.N)) {
#define MUSE_NZ_CASE(z) case z: return launch_refine_multi_nz<z>(p, d_queries, nq, sm_count, d_next, st);
        MUSE_NZ_CASE(17) MUSE_NZ_CASE(18) MUSE_NZ_CASE(19) MUSE_NZ_CASE(20) MUSE_NZ_CASE(21) MUSE_NZ_CASE(22)
        MUSE_NZ_CASE(23) MUSE_NZ_CASE(24) MUSE_NZ_CASE(25) MUSE_NZ_CASE(26) MUSE_NZ_CASE(27) MUSE_NZ_CASE(28)
        MUSE_NZ_CASE(29) MUSE_NZ_CASE(30) MUSE_NZ_CASE(31) MUSE_NZ_CASE(32)
#undef MUSE_NZ_CASE
    }
    return cudaErrorInvalidValue;
}

}  // namespace muse
