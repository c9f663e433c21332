// muse_screen_sub.cuh -- the fp32 screening + fused second stage for FFT lengths 128 .. 1024 (series of 65 .. 1024
// samples; go-muse's own benchmark shape is 480 samples, muse_batch_test.go:135-162): the design of
// score_screen_warp_kernel (muse_screen.cuh) with SEVERAL series per warp.
//
// M = n/2 = 32 T complex points per series, T = 2, 4, 8, 16 lanes per series (n = 128, 256, 512, 1024), 32 points per
// lane, so a warp carries GS = 32 / T = 16 .. 2 series side by side.  The transform, the bound and the second stage are
// the blocks of muse_screen.cuh at this T: the n = 2048 kernel's with 32 replaced by T, the mirror exchanges inside each
// T-lane group (shuffles of width T).  The forward exchange goes through the series' own row buffer.
//
// Rows arrive by cp.async.bulk: one mbarrier per warp, GS copies per iteration, re-armed as soon as the rows are in
// registers and the exchange is over (SASS UBLKCP, SYNCS), so a warp's next rows are in flight during its transforms.
//
// The second stage is taken by the WHOLE warp when any of its series needs it (the lanes stay converged: every
// shuffle, lock and barrier below is warp-wide); the groups that did not need it discard the result.  With ~4 % of
// the series needing it on the benchmark's data that is ~15 % of the warp iterations at n = 512.
//
// Same contract as every screening kernel: out_U >= the fp64 score of muse_exact.cuh for every series (or 2.0 =
// undecided), out_L a certain lower bound where the peak is certainly inside the lag window, results of a screened
// run bit-identical to the all-exact run (tests/test_gpu_screen.py).
#pragma once

#include "muse_screen.cuh"

namespace muse {

template <int LOG2T>
struct ScreenSubCfg {
    static_assert(LOG2T >= 1 && LOG2T <= 4, "sub-warp kernel: n = 128 (2 lanes per series), 256 (4), 512 (8) or 1024 (16)");
    static constexpr int LOG2M = LOG2T + 5;
    using G = Geo<LOG2M, 5>;
    static constexpr int T = 1 << LOG2T;
    static constexpr int GS = 32 / T;                 // series per warp
    static constexpr int MAX_WARPS = 12;
    static constexpr int NREF = 2;                    // warp-wide exchange buffers of the second stage, under a lock
    static constexpr size_t SMEM_BUDGET = 227 * 1024;
    static constexpr size_t EX_SERIES = ((size_t)(G::MP + 1) * sizeof(cf) + 127) / 128 * 128;   // one series' padded exchange
    // buffers of a warp's series sit a multiple of 128 bytes plus SKEW apart, which spreads the series over the
    // shared-memory banks: without it the 16 series of a warp at T = 2 (2 lanes x 16 bytes each) hit the same 8 banks on
    // every row read and every exchange.  Measured (kernel, 11.5 GB stores, skew 0 -> 8 T): n = 128 5.17 -> 2.48 ms,
    // n = 256 3.08 -> 2.29 ms, n = 512 2.08 -> 1.92 ms, n = 1024 unchanged
    static constexpr int SKEW = (8 * T) % 128;
    // The cheaper pair bound (muse_screen.cuh) pays where the kernel is bound by instruction issue and costs where it is
    // bound by HBM (it doubles the second stages).  Measured, bin-by-bin sum -> pair bound: n = 128 2.41 -> 2.21 ms,
    // n = 256 2.17 -> 1.97 ms, n = 512 1.84 -> 1.89 ms, n = 1024 1.82 -> 1.84 ms (and n = 2048 2.18 -> 2.11 ms).
    static constexpr bool PAIR_BOUND = LOG2T <= 2;
    static constexpr size_t EX_STRIDE = EX_SERIES + SKEW;
    static constexpr size_t EX_BYTES = (size_t)GS * EX_STRIDE;
    static size_t row_bytes(int N) {
        const size_t r = ((size_t)N * 8 + 127) / 128 * 128;
        return (r > EX_SERIES ? r : EX_SERIES) + SKEW;
    }
    static size_t warp_bytes(int N) { return (size_t)GS * row_bytes(N); }
    static int warps(int N) {
        const size_t w = (SMEM_BUDGET - NREF * EX_BYTES) / warp_bytes(N);
        return (int)(w > MAX_WARPS ? MAX_WARPS : w);
    }
    static size_t smem_bytes(int N) { return (size_t)warps(N) * warp_bytes(N) + NREF * EX_BYTES; }
    static int nz(int N) { return ((N + 1) / 2 + T - 1) / T; }      // rows of T complex slots that hold samples: 17 .. 32
};

#if defined(__CUDACC__)

template <int LOG2T, int NZ>
__global__ void __launch_bounds__(ScreenSubCfg<LOG2T>::MAX_WARPS * 32, 1)
score_screen_sub_kernel(const ScreenParams prm, const unsigned warp_bytes, const unsigned row_bytes) {
    using C = ScreenSubCfg<LOG2T>;
    constexpr int P = 32, T = C::T, GS = C::GS;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ __align__(8) unsigned long long bars[C::MAX_WARPS];
    __shared__ unsigned ex_locks[C::NREF];

    const int w = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int g = lane >> LOG2T;                 // series of the warp's unit this lane works on
    const int t = lane & (T - 1);                // lane within the series
    const int count = (int)prm.count;
    const int units = (count + GS - 1) / GS;     // a unit = GS consecutive series
    const int stride = (int)(gridDim.x * (blockDim.x >> 5));
    const int pos0 = (int)(blockIdx.x * (blockDim.x >> 5)) + w;
    unsigned char *wbuf = smem_raw + (size_t)w * warp_bytes;
    unsigned char *buf = wbuf + (size_t)g * row_bytes;
    const cd *rowc = reinterpret_cast<const cd *>(buf);
    cf *sm = reinterpret_cast<cf *>(buf);        // forward exchange: the series' row buffer itself
    unsigned char *refbase = smem_raw + (size_t)(blockDim.x >> 5) * warp_bytes;
    const int N = prm.N;
    const int Nh = (N + 1) >> 1;
    const unsigned bar = smem_u32(&bars[w]);
    const unsigned bytes = (unsigned)(N + (N & 1)) * 8u;
    const int partner = (T - t) & (T - 1);
    const bool lane0 = (t == 0);
    const bool last_in = t + (NZ - 1) * T < Nh;

    auto issue = [&](int unit) {                 // lane 0 of the warp: the GS rows of a unit (the last unit repeats its last row)
        mbar_expect(bar, bytes * GS);
#pragma unroll
        for (int gg = 0; gg < GS; gg++) {
            int s = unit * GS + gg;
            s = s < count ? s : count - 1;
            if (prm.rows) s = prm.rows[s];
            bulk_copy(smem_u32(wbuf + (size_t)gg * row_bytes), prm.slab + (int64_t)s * prm.ld, bytes, bar);
        }
    };

    if (threadIdx.x < C::NREF) ex_locks[threadIdx.x] = 0u;
    if (lane == 0) {
        mbar_init(bar, 1);
        mbar_init_fence();
        if (pos0 < units) issue(pos0);
    }
    __syncthreads();

    unsigned phase = 0;
    for (int pos = pos0; pos < units; pos += stride, phase ^= 1u) {
        const int sraw = pos * GS + g;
        const bool valid = sraw < count;
        const int spos = valid ? sraw : count - 1;
        const int s = prm.rows ? prm.rows[spos] : spos;      // the series (row of the store) of this work item
        unsigned cut_raw = 0u;
        if (lane == 0) cut_raw = ld_relaxed_u32(prm.cut_bits);
        const RowStat rs = prm.row_stat[s];
        const double mu = rs.mean;
        mbar_wait(bar, phase);

        cf v[P];
        load_centred<NZ, T>(v, rowc, t, mu, last_in);
        __syncwarp();
        const int next = pos + stride;

        // ---- forward FFT_M: pruned radix-32 over stride T, twiddle, exchange, GS radix-T transforms ----
        Dft32Lead<NZ, float>::run(v);
        screen_pass0<T>(v, sm, prm.twp, t);
        __syncwarp();
        if (lane == 0 && next < units) {
            asm volatile("" ::"r"(__float_as_uint(v[P - 1].y)) : "memory");
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            issue(next);
        }
        screen_pass1<T>(v);                             // v[screen_reg<T>(m)] = Z[t + T*m]
        const float acc = screen_bound<T, C::PAIR_BOUND>(v, prm, t, lane0, partner);

        float U = acc * rs.rstd * 1.00001f + MUSE_SCREEN_SLACK;
        if (!(U == U)) U = 2.f;
        float L = -1.f;
        const float cut_now = __uint_as_float(__shfl_sync(0xffffffffu, cut_raw, 0));
        const bool need = U >= cut_now && U < 1.5f;                          // uniform over the T lanes of a series
        if (__any_sync(0xffffffffu, need)) {
            conj_mul_pairs<T>(v, prm.sw, prm.sx, prm.x_mid, t, lane0, partner);
            // ---- inverse FFT_M as swap(FFT(swap(.))) ----
            cf u[P];
#pragma unroll
            for (int j = 0; j < P; j++) u[j] = v[screen_reg<T>(j)];
            Dft<P, float>::run(u);
            {
                const int slot = ex_acquire(ex_locks, lane, w);
                screen_pass0<T>(u, reinterpret_cast<cf *>(refbase + (size_t)slot * C::EX_BYTES + (size_t)g * C::EX_STRIDE), prm.twp, t);
                ex_release(ex_locks, lane, slot);
            }
            screen_pass1<T>(u);         // u[c*T + Perm(jj)] = (cc'[2i+1], cc'[2i]), i = t + c*T + 32*jj
            float m_in, m_out;
            window_maxima<T>(u, t, prm.win_lo, prm.win_len, m_in, m_out);
            if (need) {
                const float rstd = rs.rstd;
                U = refine_decide(U, m_in * rstd, m_out * rstd, L, prm.grouped);
                if (lane0 && valid) atomicAdd(prm.n_refined, 1ull);
            }
            // ---- certain passes at or above the running cut-off: count them, try to raise the cut-off (warp-wide) ----
            const float Lc = (need && valid) ? L : -1.f;
#pragma unroll
            for (int gg = 0; gg < GS; gg++) {
                const float Lg = __shfl_sync(0xffffffffu, Lc, gg * T);
                if (Lg >= prm.thr && Lg >= cut_now) cut_count_and_raise(prm.cut_bits, prm.cut_hist, prm.top_n, Lg, lane);
            }
        }
        if (lane0 && valid) {
            prm.out_U[s] = U;
            if (prm.out_L) prm.out_L[s] = L;
        }
    }
}

#endif  // __CUDACC__

}  // namespace muse
