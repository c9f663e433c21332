// kernels_roll.cu -- roll_rows_kernel: every row of a range of the store slides forward by k samples, in place,
//     row <- row[k .. N) ++ add[0 .. k),
// and gets its RowStat (and, for odd N, its pad column) in the same pass.
//
// One warp per row, front to back in chunks of 32 U samples: the warp loads the chunk's sources [c + k, c + k + 32 U)
// (from the row, or from the new samples past N - k) into registers, meets at __syncwarp, then stores [c, c + 32 U).
// The shift is safe in place because of that order: within a chunk every lane's load comes before any lane's store, and
// the loads of a later chunk are at or above c + 32 U + k, past every store made so far.  Cutting a row into segments for
// several warps would break it (segment j + 1 would overwrite samples segment j has not read yet), so rows above
// MUSE_MAX_FUSED_FFT_LEN samples stay one warp per row as well: the roll is a copy, not a performance target at those
// lengths, and one code path keeps the statistics bit-identical to row_stats_kernel's at every length.
// The slab pointer is deliberately not __restrict__: loads and stores of a row alias, and their order is the point.
#include <algorithm>

#include "muse_launch.h"

namespace muse {

static constexpr int ROLL_U = 8;          // samples per lane per chunk: 2 KB of loads in flight per warp
static constexpr int ROLL_THREADS = 256;

__global__ void __launch_bounds__(ROLL_THREADS)
roll_rows_kernel(double *slab, int64_t ld, int N, int64_t first, int64_t count, const double *__restrict__ add, int k,
                 RowStat *__restrict__ stat) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarp = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int keep = N - k;                // samples that stay in the row (moved left by k)
    for (int64_t i = warp0; i < count; i += nwarp) {
        double *row = slab + (first + i) * ld;
        const double *a = add + i * k;
        const double pivot = keep > 0 ? row[k] : a[0];      // the rolled row's first sample, read before any store
        RowSums rs;
        for (int c = 0; c < N; c += 32 * ROLL_U) {
            double v[ROLL_U];
#pragma unroll
            for (int j = 0; j < ROLL_U; j++) {
                const int p = c + 32 * j + lane;
                v[j] = p < keep ? row[p + k] : (p < N ? a[p - keep] : 0.0);
            }
            __syncwarp();
#pragma unroll
            for (int j = 0; j < ROLL_U; j++) {
                const int p = c + 32 * j + lane;
                if (p < N) {
                    row[p] = v[j];
                    rs.add(v[j], pivot);
                }
            }
        }
        const RowStat r = rs.warp_stat(pivot, N);
        if (lane == 0) {
            stat[first + i] = r;
            if (N & 1) row[N] = r.mean;
        }
    }
}

cudaError_t launch_roll_rows(double *slab, int64_t ld, int N, int64_t first, int64_t count, const double *d_add, int k,
                             RowStat *stat, int sm_count, cudaStream_t st) {
    int per_sm = 0;
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, roll_rows_kernel, ROLL_THREADS, 0);
    if (e != cudaSuccess) return e;
    const int64_t warps = ROLL_THREADS / 32;
    const int64_t blocks = std::min<int64_t>((count + warps - 1) / warps, (int64_t)std::max(per_sm, 1) * sm_count);
    roll_rows_kernel<<<(unsigned)blocks, ROLL_THREADS, 0, st>>>(slab, ld, N, first, count, d_add, k, stat);
    return cudaGetLastError();
}

}  // namespace muse
