// kernels_remove.cu -- move_rows_kernel: the row moves of muse_group_remove.  Pair i moves local row moves[i].x to local
// row moves[i].y: the whole ld-wide row (for odd N the pad column row[N], the row's mean, goes with it), its RowStat and its
// id in each of the nkeys label columns ([nkeys][cap]).
//
// Every source is at or above the store's new size m and every destination below it, so no element is both read and
// written: the copy can be cut into any pieces.  A row is cut into segments of 32 U 16-byte words (2 KB), one warp per
// segment, consecutive warps on consecutive segments of the same row; rows of any length (up to 2^24 samples) spread over
// as many warps as they have segments.  Rows are 128-byte aligned (ld is a multiple of 16 doubles), so every load and
// store is 16 bytes wide and coalesced.
#include <algorithm>

#include "muse_launch.h"

namespace muse {

static constexpr int MOVE_U = 4;                  // 16-byte words per lane per segment: 2 KB of loads in flight per warp
static constexpr int MOVE_SEG = 32 * MOVE_U;      // 16-byte words per segment
static constexpr int MOVE_THREADS = 256;

__global__ void __launch_bounds__(MOVE_THREADS)
move_rows_kernel(double2 *slab, int64_t ld2, RowStat *stat, int32_t *labels, int nkeys, int64_t cap,
                 const int2 *__restrict__ moves, int64_t count) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarp = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t segs = (ld2 + MOVE_SEG - 1) / MOVE_SEG;
    const int64_t units = count * segs;
    for (int64_t u = warp0; u < units; u += nwarp) {
        const int64_t i = u / segs, s = u - i * segs;
        const int2 mv = moves[i];
        const int64_t off = s * MOVE_SEG, left = ld2 - off;
        const double2 *src = slab + (int64_t)mv.x * ld2 + off;
        double2 *dst = slab + (int64_t)mv.y * ld2 + off;
        double2 v[MOVE_U];
#pragma unroll
        for (int j = 0; j < MOVE_U; j++)
            if (32 * j + lane < left) v[j] = src[32 * j + lane];
#pragma unroll
        for (int j = 0; j < MOVE_U; j++)
            if (32 * j + lane < left) dst[32 * j + lane] = v[j];
        if (s == 0) {      // the row's statistics and label ids: lane 0 the RowStat, lane 1 + k label column k
            for (int t = lane; t <= nkeys; t += 32) {
                if (t == 0) stat[mv.y] = stat[mv.x];
                else labels[(int64_t)(t - 1) * cap + mv.y] = labels[(int64_t)(t - 1) * cap + mv.x];
            }
        }
    }
}

cudaError_t launch_move_rows(double *slab, int64_t ld, RowStat *stat, int32_t *labels, int nkeys, int64_t cap, const int2 *d_moves,
                             int64_t count, int sm_count, cudaStream_t st) {
    if (count <= 0) return cudaSuccess;
    int per_sm = 0;
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, move_rows_kernel, MOVE_THREADS, 0);
    if (e != cudaSuccess) return e;
    const int64_t ld2 = ld / 2;
    const int64_t units = count * ((ld2 + MOVE_SEG - 1) / MOVE_SEG);
    const int64_t warps = MOVE_THREADS / 32;
    const int64_t blocks = std::min<int64_t>((units + warps - 1) / warps, (int64_t)std::max(per_sm, 1) * sm_count);
    move_rows_kernel<<<(unsigned)blocks, MOVE_THREADS, 0, st>>>(reinterpret_cast<double2 *>(slab), ld2, stat, labels, nkeys, cap,
                                                                d_moves, count);
    return cudaGetLastError();
}

}  // namespace muse
