// muse_screen_multi.cuh -- many reference queries in ONE pass over the slab (SURVEY 8f rank 2 / BASELINE.json configs[4]:
// many references, one store).
//
// go-muse builds one Batch per reference (muse_batch.go:23-52), so Q queries stream the store Q times and transform
// every series Q times.  Nothing about a series' spectrum depends on the reference: the bounds of all queries come from
// one bf16 contraction on the tensor cores (muse_bounds_tc.cuh), and refine_multi_kernel below transforms each row ONCE
// and runs the second stage for every query whose bound needs it.
#pragma once

#include "muse_screen.cuh"

namespace muse {

struct MultiQuery {
    const float4 *sw;     // the query's (w_k, A[k], A[M-k]) table (refine_multi_kernel does not read it)
    const float4 *sx;     // (Xt[k], Xt[M-k]) in fp32, k < M/2
    cf x_mid;             // Xt[M/2]
    float a_mid;          // A[M/2]
    int pad;
    CutState *cut;        // the query's cut-off state
    float *out_U;         // [count] upper bound on the score for this query
};

#if defined(__CUDACC__)

// ---- second stage for up to 256 queries whose bounds were computed elsewhere (muse_bounds_tc.cuh) -------------------
// One pass over the store: a warp loads its row, runs the forward FFT_1024 once, stashes the spectrum in shared memory
// and reads the series' bound against every query of the launch (query q's array out_U[pos], lane l looks after the
// queries l, l + 32, ...).  Every (series, query) pair whose bound reaches that query's RUNNING cut-off takes the second
// stage of muse_screen.cuh (conj(Y) X_q, inverse FFT_1024, maxima inside / outside the lag window), which replaces the
// bound by the tight fp32 one and feeds the query's cut-off histogram.  Afterwards every query is exactly where a
// single-query run is after its screening kernel.  Each warp owns its exchange buffer: with ~10 refinements per series a
// shared, locked buffer would serialise the block.
struct RefineMultiCfg {
    using G = Geo<10, 5>;
#ifndef MUSE_REFINE_WARPS
#define MUSE_REFINE_WARPS 8      // measured (256 queries x 1 M series): 12 warps at 168 registers 112 ms, 10 warps 76 ms, 8 warps at 255 registers 72 ms
#endif
    static constexpr int MAX_WARPS = MUSE_REFINE_WARPS;
    static constexpr int QMAX = 256;            // queries per launch (== TcCfg::TN)
    static constexpr int QI = QMAX / 32;        // bounds per lane
    static constexpr size_t SMEM_BUDGET = 227 * 1024;
    static constexpr size_t STASH_BYTES = (size_t)G::M * sizeof(cf);                                  // 8 KB: the spectrum
    static constexpr size_t EX_BYTES = ScreenWarpCfg::EX_BYTES;                                       // padded FFT exchange buffer
    static size_t warp_bytes(int N) {
        const size_t row = ((size_t)N * 8 + 127) / 128 * 128, own = STASH_BYTES + EX_BYTES;
        return row > own ? row : own;
    }
    // per block: the queries' cut-off words and bound arrays (4 KB), the pass twiddles (31 x 32 cf = 8 KB) and the split
    // twiddles (512 cf = 4 KB) -- every second stage reads both tables, and with ~200 KB of shared memory configured the L1
    // is too small to hold them
    static constexpr size_t TW_BYTES = 31 * 32 * sizeof(cf) + 64, SW_BYTES = (size_t)(G::M / 2) * sizeof(cf);
    static size_t table_bytes() { return (size_t)QMAX * 2 * sizeof(void *) + TW_BYTES + SW_BYTES; }
    static int warps(int N) {
        const size_t w = (SMEM_BUDGET - table_bytes()) / warp_bytes(N);
        return (int)(w > MAX_WARPS ? MAX_WARPS : w);
    }
    static size_t smem_bytes(int N) { return (size_t)warps(N) * warp_bytes(N) + table_bytes(); }
};

template <int NZ>
__global__ void __launch_bounds__(RefineMultiCfg::MAX_WARPS * 32, 1)
refine_multi_kernel(const ScreenParams prm, const MultiQuery *__restrict__ queries, const int nq, const unsigned warp_bytes,
                    unsigned *__restrict__ next_series) {
    using C = RefineMultiCfg;
    constexpr int P = 32, M = C::G::M, QI = C::QI;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ __align__(8) unsigned long long bars[C::MAX_WARPS];

    const int w = threadIdx.x >> 5;
    const int t = threadIdx.x & 31;
    const int nwarps = (int)(blockDim.x >> 5);
    const int count = (int)prm.count;
    // series are handed out by a global counter (the cost of a series varies with the number of its second stages by two
    // orders of magnitude: a fixed assignment left most warps idle behind the unlucky ones); the counter starts at the number
    // of warps of the grid, whose first series is their own index
    const int pos0 = (int)(blockIdx.x * nwarps) + w;
    unsigned char *buf = smem_raw + (size_t)w * warp_bytes;
    const cd *rowc = reinterpret_cast<const cd *>(buf);
    cf *stash = reinterpret_cast<cf *>(buf);                                  // slot j of lane t at [32 j + t]
    cf *ex = reinterpret_cast<cf *>(buf + C::STASH_BYTES);                    // this warp's FFT exchange buffer
    CutState **s_cut = reinterpret_cast<CutState **>(smem_raw + (size_t)nwarps * warp_bytes);      // [QMAX] cut-off states
    float **s_out = reinterpret_cast<float **>(s_cut + C::QMAX);                                   // [QMAX] bound arrays
    cf *s_tw = reinterpret_cast<cf *>(s_out + C::QMAX);                                            // pass twiddles W_1024^(j t)
    cf *s_sw = reinterpret_cast<cf *>(reinterpret_cast<unsigned char *>(s_tw) + C::TW_BYTES);      // split twiddles exp(-2 pi i k / n)
    const int N = prm.N;
    const int Nh = (N + 1) >> 1;      // complex slots holding samples (odd N: the pad column of the last one holds the row's mean, RowStat)
    const unsigned bar = smem_u32(&bars[w]);
    const int partner = (P - t) & (P - 1);
    const bool lane0 = (t == 0);
    const bool last_in = t + (NZ - 1) * 32 < Nh;
    const int nqi = (nq + 31) >> 5;

    if (t == 0) {
        mbar_init(bar, 1);
        mbar_init_fence();
        if (pos0 < count) bulk_load(smem_u32(buf), prm.slab + (int64_t)pos0 * prm.ld, (unsigned)(N + (N & 1)) * 8u, bar);
    }
    for (int q = threadIdx.x; q < C::QMAX; q += blockDim.x) {
        s_cut[q] = q < nq ? queries[q].cut : nullptr;
        s_out[q] = q < nq ? queries[q].out_U : nullptr;
    }
    for (int i = threadIdx.x; i < 31 * 32; i += blockDim.x) s_tw[i] = prm.twp[i];
    for (int i = threadIdx.x; i < M / 2; i += blockDim.x) {
        const float4 s = prm.sw[i];
        s_sw[i] = cf{s.x, s.y};
    }
    __syncthreads();

    unsigned phase = 0;
    int next = 0;
    for (int pos = pos0; pos < count; pos = next, phase ^= 1u) {
        // this series' bounds against all queries and the queries' running cut-offs: in flight under the transform
        float U[QI];
        unsigned cutr[QI];
#pragma unroll
        for (int i = 0; i < QI; i++) {
            U[i] = -1.f;
            cutr[i] = 0x7f800000u;          // +inf: no such query
            if (i < nqi && t + 32 * i < nq) {
                U[i] = s_out[t + 32 * i][pos];
                cutr[i] = ld_relaxed_u32(&s_cut[t + 32 * i]->bits);
            }
        }
        const RowStat rs = prm.row_stat[pos];
        const double mu = rs.mean;
        mbar_wait(bar, phase);

        cf v[P];
        load_centred<NZ, 32>(v, rowc, t, mu, last_in);
        __syncwarp();                       // the row is in registers: its buffer becomes exchange + stash
        if (t == 0) next = (int)atomicAdd(next_series, 1u);
        next = __shfl_sync(0xffffffffu, next, 0);

        Dft32Lead<NZ, float>::run(v);
        screen_pass0<32>(v, ex, s_tw, t);
        screen_pass1<32>(v);                            // v[Perm(j)] = Z[t + 32*j]
#pragma unroll
        for (int j = 0; j < P; j++) stash[32 * j + t] = v[Perm<P>::at(j)];      // every lane reads back only what it wrote

        // which (query group i, lane) pairs take the second stage: one ballot per group, then ONE rolled loop over the
        // pairs -- the second stage is ~45 KB of code, and a copy per group (the loop unrolled) thrashed the instruction
        // cache (measured: 10x slower)
        unsigned todo[QI];
#pragma unroll
        for (int i = 0; i < QI; i++) todo[i] = __ballot_sync(0xffffffffu, U[i] >= __uint_as_float(cutr[i]) && U[i] < 1.5f);
        unsigned changed = 0u;
#pragma unroll 1
        while (true) {
            // next pair: the lowest group with a bit left (warp-uniform select chains: the arrays stay in registers)
            int gi = -1;
            unsigned gm = 0u;
#pragma unroll
            for (int i = QI - 1; i >= 0; i--)
                if (todo[i]) {
                    gi = i;
                    gm = todo[i];
                }
            if (gi < 0) break;
            const int ql = __ffs(gm) - 1;
            float Usel = 0.f;
            unsigned csel = 0u;
#pragma unroll
            for (int i = 0; i < QI; i++) {
                if (i == gi) {
                    todo[i] = gm & (gm - 1);
                    Usel = U[i];
                    csel = cutr[i];
                }
            }
            {
                float Uq = __shfl_sync(0xffffffffu, Usel, ql);
                const float cut_now = __uint_as_float(__shfl_sync(0xffffffffu, csel, ql));
                const MultiQuery mq = queries[32 * gi + ql];
                cf z[P];
#pragma unroll
                for (int j = 0; j < P; j++) z[Perm<P>::at(j)] = stash[32 * j + t];
                conj_mul_pairs<32>(z, s_sw, mq.sx, mq.x_mid, t, lane0, partner);
                cf u[P];
#pragma unroll
                for (int j = 0; j < P; j++) u[j] = z[Perm<P>::at(j)];
                Dft<P, float>::run(u);
                __syncwarp();                           // the previous use of the exchange buffer has been read
                screen_pass0<32>(u, ex, s_tw, t);
                screen_pass1<32>(u);
                float m_in, m_out;
                window_maxima<32>(u, t, prm.win_lo, prm.win_len, m_in, m_out);
                float L = -1.f;
                Uq = refine_decide(Uq, m_in * rs.rstd, m_out * rs.rstd, L, 0);
                if (t == 0) atomicAdd(&mq.cut->refined, 1ull);
                if (L >= prm.thr && L >= cut_now) cut_count_and_raise(&mq.cut->bits, mq.cut->hist, prm.top_n, L, t);
#pragma unroll
                for (int i = 0; i < QI; i++)
                    if (i == gi && t == ql) {
                        U[i] = Uq;
                        changed |= 1u << i;
                    }
            }
        }
#pragma unroll
        for (int i = 0; i < QI; i++)
            if (changed & (1u << i)) s_out[t + 32 * i][pos] = U[i];
        // the stash is no longer needed: hand the buffer to the copy engine for the warp's next row
        __syncwarp();
        if (t == 0 && next < count) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            bulk_load(smem_u32(buf), prm.slab + (int64_t)next * prm.ld, (unsigned)(N + (N & 1)) * 8u, bar);
        }
    }
}

#endif  // __CUDACC__

}  // namespace muse
