// muse_bounds_tc.cuh -- the screening bounds of MANY reference queries as ONE tensor-core contraction
// (BASELINE.json configs[4]: 256 reference queries x 1 M series x 1440 samples).
//
// go-muse builds one Batch per reference (muse_batch.go:23-52) and transforms every series once per query.  The spectral
// bound of muse_screen.cuh,
//     U[s][q] = (1/n) sum_f |Y_s,f| |X_q,f| / std_s * (1 + eps) + slack  >=  score(series s, query q),
// is a product of two NON-NEGATIVE matrices: Mg [S x 1024] (the 512 mirror pairs of magnitudes |2Y_k|, |2Y_(M-k)| of every
// series) times W^T [1024 x Q] (the queries' weights A_q[k] = |X_q,k| / (2n) * (1 or 2)).
// Precision: one bf16 per value (8 mantissa bits, rounded up) makes the bound 1 % looser, and on real data that is fatal:
// the bounds of a third of all series lie within 1 % of a query's top-100 cut-off, so eight times as many pairs took the
// second stage (measured: 33 % instead of 4.4 %).  Every value is therefore split into TWO bf16, x <= hi + lo with hi = x
// truncated and lo = (x - hi) rounded up (16 mantissa bits), and the product is expanded,
//     sum m w  <=  sum m_hi w_hi  +  sum (m_hi w_lo + m_lo w_hi)  +  sum m_lo w_lo,      the last <= 2^-14 of the first,
// three bf16 MMAs per K step into TWO accumulators (the cross terms are 2^-7 of the main term, so their roundings do not
// count; the main accumulator's 1024 non-negative products add at most 1024 * 2^-23 = 1.2e-4 relative when the tensor core
// truncates).  Products of two bf16 are exact in fp32.  The epilogue's factor 1.0003 covers the accumulation, the dropped
// lo x lo term and sqrt.approx.  So:
//   1. mag_tiles_kernel<NZ>   one pass over the store: row (bulk copy) -> forward FFT_1024 -> split -> |2Y| as (hi, lo) bf16
//                             tiles in the layout tcgen05.mma reads (below); bin M/2 (its own mirror) is kept in fp32 per
//                             series and added in the epilogue as a rank-1 term;
//   2. weight_tiles_kernel    the queries' weights as (hi, lo) tiles in the same K order and layout;
//   3. bounds_tc_kernel       per 128 series: D0[128 x 256] += A_hi B_hi^T, D1 += A_hi B_lo^T + A_lo B_hi^T (fp32, all 512
//                             TMEM columns) over 16 K tiles of 64, tcgen05.mma.cta_group::1.kind::f16 issued by one thread,
//                             operands brought in by cp.async.bulk into a 2-stage shared-memory ring of 96 KB stages
//                             (mbarrier full / empty, tcgen05.commit frees a stage), epilogue tcgen05.ld ->
//                             U = (D0 + D1 + mid_s * amid_q) * rstd_s * 1.0003 + slack.
// What the bound gates is only WHICH (series, query) pairs take the fp32 second stage (refine_multi_kernel), so the
// results stay those of the exact fp64 kernel.
//
// Operand layout (UMMA canonical K-major, no swizzle: core matrix = 8 rows x 16 bytes, contiguous): a K tile of 64 bf16
// of R rows (R = 128 series or 256 queries) is [kc = 8][rg = R/8][r8 = 8][8 bf16], i.e. byte offset
//     kc * (R * 16) + (row / 8) * 128 + (row % 8) * 16 + (k % 8) * 2,        kc = (k % 64) / 8,
// so LBO (16-byte K chunk -> next chunk) = R * 16 bytes and SBO (8 rows -> next 8 rows) = 128 bytes, and every tile is one
// contiguous block in global memory: a plain 1-D bulk copy puts it where the tensor core wants it (no tensor map).
// K order: kk = 32 t + 2 j + side for the mirror pair k = t + 32 j (lane t of the transform holds it), side 0 = bin k,
// side 1 = bin M - k; both operands use it, so the contraction does not care.
#pragma once

#include "muse_screen.cuh"

namespace muse {

struct TcCfg {
    static constexpr int K = 1024;            // mirror pairs x 2
    static constexpr int KT = 64;             // bf16 per K tile (8 chunks of 16 bytes)
    static constexpr int NKT = K / KT;        // 16
    static constexpr int TM = 128;            // series per tile (UMMA M)
    static constexpr int TN = 256;            // queries per launch (UMMA N)
    static constexpr int A_PART_BYTES = TM * KT * 2;      // 16 KB: one of (hi, lo)
    static constexpr int B_PART_BYTES = TN * KT * 2;      // 32 KB
    static constexpr int A_TILE_BYTES = 2 * A_PART_BYTES; // hi then lo
    static constexpr int B_TILE_BYTES = 2 * B_PART_BYTES;
    static constexpr int STAGE_BYTES = A_TILE_BYTES + B_TILE_BYTES;      // 96 KB
    static constexpr int STAGES = 2;
    static constexpr int THREADS = 192;       // warp 0: copies, warp 1: MMA + TMEM, warps 2..5: epilogue
    static constexpr size_t SMEM = (size_t)STAGES * STAGE_BYTES + 1024;
    static size_t a_bytes(int64_t S) { return (size_t)((S + TM - 1) / TM) * NKT * A_TILE_BYTES; }
    static constexpr size_t b_bytes() { return (size_t)NKT * B_TILE_BYTES; }
};

struct TcBoundsParams {
    const unsigned char *a_tiles;     // [S/128][16][hi 16 KB, lo 16 KB] bf16 magnitudes (mag_tiles_kernel)
    const unsigned char *b_tiles;     // [16][hi 32 KB, lo 32 KB] bf16 weights of up to 256 queries (weight_tiles_kernel), zero rows beyond nq
    const float *mid;                 // [S] |2Y_(M/2)| of every series
    const float *amid;                // [256] A_q[M/2]
    const RowStat *row_stat;          // [S] (1/std of every series)
    float *const *out_U;              // [nq] per-query bound arrays [S]
    int64_t S;
    int nq;
};

#if defined(__CUDACC__) && defined(MUSE_TC_KERNELS)      // the kernels live in ONE translation unit (kernels_bounds_tc.cu)

// x >= 0 (or NaN / inf) rounded UP to a bf16 bit pattern
__device__ __forceinline__ unsigned bf16_up(float x) { return (__float_as_uint(x) + 0xffffu) >> 16; }
// x >= 0 as two bf16 with hi + lo >= x: hi = x truncated, lo = the (exactly representable) remainder rounded up
__device__ __forceinline__ void bf16_split(float x, unsigned &hi, unsigned &lo) {
    hi = __float_as_uint(x) >> 16;
    lo = bf16_up(x - __uint_as_float(hi << 16));      // inf - inf = NaN: the bound becomes "undecided", as it must
}

// ---- 1. magnitudes of every series in tile layout ----------------------------------------------------------------
// The transform is score_screen_warp_kernel's (one warp per series, row by cp.async.bulk, radix-32 x radix-32 through the
// row buffer); lane t ends with the mirror pairs k = t + 32 j, j < 16.
template <int NZ>
__global__ void __launch_bounds__(ScreenWarpCfg::MAX_WARPS * 32, 1)
mag_tiles_kernel(const ScreenParams prm, unsigned char *__restrict__ a_tiles, float *__restrict__ mid, const unsigned warp_bytes) {
    using C = ScreenWarpCfg;
    constexpr int P = 32;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ __align__(8) unsigned long long bars[C::MAX_WARPS];

    const int w = threadIdx.x >> 5;
    const int t = threadIdx.x & 31;
    const int count = (int)prm.count;
    const int stride = (int)(gridDim.x * (blockDim.x >> 5));
    const int pos0 = (int)(blockIdx.x * (blockDim.x >> 5)) + w;
    unsigned char *buf = smem_raw + (size_t)w * warp_bytes;
    const cd *rowc = reinterpret_cast<const cd *>(buf);
    cf *sm = reinterpret_cast<cf *>(buf);
    const int N = prm.N;
    const int Nh = (N + 1) >> 1;      // complex slots holding samples (odd N: the pad column of the last one holds the row's mean, RowStat)
    const unsigned bar = smem_u32(&bars[w]);
    const int partner = (P - t) & (P - 1);
    const bool lane0 = (t == 0);
    const bool last_in = t + (NZ - 1) * 32 < Nh;

    if (t == 0) {
        mbar_init(bar, 1);
        mbar_init_fence();
        if (pos0 < count) bulk_load(smem_u32(buf), prm.slab + (int64_t)pos0 * prm.ld, (unsigned)(N + (N & 1)) * 8u, bar);
    }
    __syncthreads();

    unsigned phase = 0;
    for (int pos = pos0; pos < count; pos += stride, phase ^= 1u) {
        const double mu = prm.row_stat[pos].mean;
        mbar_wait(bar, phase);
        cf v[P];
        load_centred<NZ, 32>(v, rowc, t, mu, last_in);
        __syncwarp();
        const int next = pos + stride;
        Dft32Lead<NZ, float>::run(v);
        screen_pass0<32>(v, sm, prm.twp, t);
        __syncwarp();
        if (t == 0 && next < count) {       // the exchange is over: the buffer goes back to the copy engine
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            bulk_load(smem_u32(buf), prm.slab + (int64_t)next * prm.ld, (unsigned)(N + (N & 1)) * 8u, bar);
        }
        screen_pass1<32>(v);                            // v[Perm(j)] = Z[t + 32*j]

        unsigned pk[16], pl[16];                        // bf16 (hi | lo) pairs (|2Y_k|, |2Y_(M-k)|), kk = 32 t + 2 j + side
#pragma unroll
        for (int j = 0; j < P / 2; j++) {
            const cf zk = v[Perm<P>::at(j)];
            const cf zm = mirror_of<32>(v, j, lane0, partner);
            const float4 s = prm.sw[t + 32 * j];            // only the split twiddle is used here
            const cf zmc = cconj(zm);
            cf qk, qm;
            split_sq(cadd(zk, zmc), csub(zk, zmc), cf{s.x, s.y}, qk, qm);
            // sqrt.approx is within 2 ulp either way: the epilogue's factor covers it
            unsigned h0, l0, h1, l1;
            bf16_split(sqrt_approx(qk.x + qk.y), h0, l0);
            bf16_split(sqrt_approx(qm.x + qm.y), h1, l1);
            pk[j] = h0 | (h1 << 16);
            pl[j] = l0 | (l1 << 16);
        }
        {
            const int tile = pos >> 7, r = pos & 127;
            unsigned char *dst = a_tiles + ((size_t)tile * TcCfg::NKT + (t >> 1)) * TcCfg::A_TILE_BYTES + (size_t)((t & 1) * 4) * (TcCfg::TM * 16) +
                                 (size_t)(r >> 3) * 128 + (size_t)(r & 7) * 16;
#pragma unroll
            for (int c = 0; c < 4; c++) {
                *reinterpret_cast<uint4 *>(dst + (size_t)c * (TcCfg::TM * 16)) = make_uint4(pk[4 * c], pk[4 * c + 1], pk[4 * c + 2], pk[4 * c + 3]);
                *reinterpret_cast<uint4 *>(dst + TcCfg::A_PART_BYTES + (size_t)c * (TcCfg::TM * 16)) =
                    make_uint4(pl[4 * c], pl[4 * c + 1], pl[4 * c + 2], pl[4 * c + 3]);
            }
        }
        if (lane0) {
            const cf z = v[Perm<P>::at(P / 2)];
            const cf q = pmul(z, z);
            mid[pos] = 2.f * sqrt_approx(q.x + q.y);
        }
    }
}

// ---- 2. the queries' weights in the same K order and tile layout ---------------------------------------------------
// sw[q]: the query's (w_k, A[k], A[M-k]) table, k < 512 (screen_tables_kernel).  One thread per (query row, 16-byte chunk).
__global__ void weight_tiles_kernel(const float4 *const *__restrict__ sw, int nq, unsigned char *__restrict__ b_tiles) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;      // chunk index: [q = 256][chunk = 128]
    if (idx >= TcCfg::TN * (TcCfg::K / 8)) return;
    const int q = idx >> 7, ch = idx & 127;                     // chunk ch holds kk = 8 ch .. 8 ch + 7
    const int t = ch >> 2, c = ch & 3;                          // kk = 32 t + 8 c + e: pairs j = 4 c + e / 2
    unsigned pk[4] = {0u, 0u, 0u, 0u}, pl[4] = {0u, 0u, 0u, 0u};
    if (q < nq) {
        const float4 *tab = sw[q];
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const float4 s = tab[t + 32 * (4 * c + i)];
            unsigned h0, l0, h1, l1;
            bf16_split(s.z, h0, l0);
            bf16_split(s.w, h1, l1);
            pk[i] = h0 | (h1 << 16);
            pl[i] = l0 | (l1 << 16);
        }
    }
    const int ktile = ch >> 3, kc = ch & 7;
    unsigned char *dst = b_tiles + (size_t)ktile * TcCfg::B_TILE_BYTES + (size_t)kc * (TcCfg::TN * 16) + (size_t)(q >> 3) * 128 + (size_t)(q & 7) * 16;
    *reinterpret_cast<uint4 *>(dst) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
    *reinterpret_cast<uint4 *>(dst + TcCfg::B_PART_BYTES) = make_uint4(pl[0], pl[1], pl[2], pl[3]);
}

// ---- 3. the contraction on the tensor cores -------------------------------------------------------------------------
// UMMA shared-memory descriptor, K-major, no swizzle (cute::UMMA::SmemDescriptor: start address, LBO and SBO in units of
// 16 bytes at bits [0,14), [16,30), [32,46); version 1 at [46,48); layout type 0 at [61,64))
__device__ __forceinline__ unsigned long long umma_desc(unsigned smem_addr, unsigned lbo_bytes, unsigned sbo_bytes) {
    return (unsigned long long)((smem_addr >> 4) & 0x3fffu) | ((unsigned long long)((lbo_bytes >> 4) & 0x3fffu) << 16) |
           ((unsigned long long)((sbo_bytes >> 4) & 0x3fffu) << 32) | (1ull << 46);
}
// instruction descriptor of kind::f16 (cute::UMMA::InstrDescriptor): D fp32 (bits [4,6) = 1), A and B bf16 ([7,10) = [10,13) = 1),
// both K-major (bits 15, 16 = 0), N >> 3 at [17,23), M >> 4 at [24,29)
__device__ __forceinline__ constexpr unsigned umma_idesc_bf16(int M, int N) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((unsigned)(N >> 3) << 17) | ((unsigned)(M >> 4) << 24);
}

// 32 consecutive TMEM columns of this thread's lane
__device__ __forceinline__ void tmem_ld32(unsigned taddr, unsigned (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
          "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
          "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}

// D[tmem_d] (+)= A[desc_a] * B[desc_b]^T, one thread on behalf of the block
__device__ __forceinline__ void umma_bf16(unsigned tmem_d, unsigned long long desc_a, unsigned long long desc_b, unsigned idesc, unsigned accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}

__global__ void __launch_bounds__(TcCfg::THREADS, 1)
bounds_tc_kernel(const TcBoundsParams prm) {
    using C = TcCfg;
    extern __shared__ __align__(128) unsigned char smem_raw[];      // aligned to 1024 below
    __shared__ __align__(8) unsigned long long full_bar[C::STAGES], empty_bar[C::STAGES], done_bar;
    __shared__ unsigned tmem_slot;
    __shared__ float s_amid[C::TN];

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tile = blockIdx.x;
    unsigned char *stage0 = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    const unsigned stage_u32 = smem_u32(stage0);

    if (threadIdx.x == 0) {
        for (int i = 0; i < C::STAGES; i++) {
            mbar_init(smem_u32(&full_bar[i]), 1);
            mbar_init(smem_u32(&empty_bar[i]), 1);
        }
        mbar_init(smem_u32(&done_bar), 1);
        mbar_init_fence();
    }
    for (int i = threadIdx.x; i < C::TN; i += blockDim.x) s_amid[i] = i < prm.nq ? prm.amid[i] : 0.f;
    if (warp == 1) {      // all 512 TMEM columns: two 128 x 256 fp32 accumulators
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const unsigned tmem = tmem_slot;

    if (warp == 0) {
        // ===== copies: A tile (this block's 128 series) and B tile (all queries) of every K tile =====
        if (lane == 0) {
            const unsigned char *a_src = prm.a_tiles + (size_t)tile * C::NKT * C::A_TILE_BYTES;
            for (int kt = 0; kt < C::NKT; kt++) {
                const int s = kt % C::STAGES;
                if (kt >= C::STAGES) mbar_wait(smem_u32(&empty_bar[s]), (unsigned)((kt / C::STAGES - 1) & 1));
                const unsigned fb = smem_u32(&full_bar[s]);
                const unsigned dst = stage_u32 + (unsigned)s * C::STAGE_BYTES;
                mbar_expect(fb, (unsigned)C::STAGE_BYTES);
                bulk_copy(dst, a_src + (size_t)kt * C::A_TILE_BYTES, (unsigned)C::A_TILE_BYTES, fb);
                bulk_copy(dst + C::A_TILE_BYTES, prm.b_tiles + (size_t)kt * C::B_TILE_BYTES, (unsigned)C::B_TILE_BYTES, fb);
            }
        }
    } else if (warp == 1) {
        // ===== MMA issue: one thread on behalf of the block =====
        if (lane == 0) {
            constexpr unsigned idesc = umma_idesc_bf16(C::TM, C::TN);
            for (int kt = 0; kt < C::NKT; kt++) {
                const int s = kt % C::STAGES;
                mbar_wait(smem_u32(&full_bar[s]), (unsigned)((kt / C::STAGES) & 1));
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const unsigned a_addr = stage_u32 + (unsigned)s * C::STAGE_BYTES, b_addr = a_addr + C::A_TILE_BYTES;
#pragma unroll
                for (int ks = 0; ks < C::KT / 16; ks++) {      // K = 16 per instruction: two 16-byte chunks
                    const unsigned long long a_hi = umma_desc(a_addr + (unsigned)ks * 2u * (C::TM * 16), C::TM * 16, 128);
                    const unsigned long long a_lo = umma_desc(a_addr + C::A_PART_BYTES + (unsigned)ks * 2u * (C::TM * 16), C::TM * 16, 128);
                    const unsigned long long b_hi = umma_desc(b_addr + (unsigned)ks * 2u * (C::TN * 16), C::TN * 16, 128);
                    const unsigned long long b_lo = umma_desc(b_addr + C::B_PART_BYTES + (unsigned)ks * 2u * (C::TN * 16), C::TN * 16, 128);
                    const unsigned first = (kt | ks) ? 1u : 0u;
                    umma_bf16(tmem, a_hi, b_hi, idesc, first);                // D0 += A_hi B_hi^T
                    umma_bf16(tmem + (unsigned)C::TN, a_hi, b_lo, idesc, first);  // D1 += A_hi B_lo^T
                    umma_bf16(tmem + (unsigned)C::TN, a_lo, b_hi, idesc, 1u);     // D1 += A_lo B_hi^T
                }
                // frees the stage when the MMAs that read it have completed (implies tcgen05.fence::before_thread_sync)
                asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(&empty_bar[s])) : "memory");
            }
            asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(&done_bar)) : "memory");
        }
    } else {
        // ===== epilogue: warp w reads the TMEM lanes of its quarter (w % 4), one series per thread =====
        const int quarter = warp & 3;
        const int64_t srow = (int64_t)tile * C::TM + quarter * 32 + lane;
        const bool live = srow < prm.S;
        float rstd = 0.f, midv = 0.f;
        if (live) {
            rstd = prm.row_stat[srow].rstd;
            midv = prm.mid[srow];
        }
        mbar_wait(smem_u32(&done_bar), 0u);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const unsigned taddr = tmem + ((unsigned)(quarter * 32) << 16);
        for (int c0 = 0; c0 < C::TN; c0 += 32) {
            unsigned r[32], r1[32];
            tmem_ld32(taddr + (unsigned)c0, r);
            tmem_ld32(taddr + (unsigned)(C::TN + c0), r1);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
            for (int i = 0; i < 32; i++) {
                const int q = c0 + i;
                if (q < prm.nq) {      // warp-uniform
                    // D0: 1024 exact non-negative products, accumulated with at most 1.2e-4 lost; D1: the cross terms; 3e-4
                    // covers that, the dropped lo x lo term (< 2^-14) and sqrt.approx (header)
                    const float sum = __uint_as_float(r[i]) + __uint_as_float(r1[i]);
                    float U = fmaf(midv, s_amid[q], sum) * rstd * 1.0003f + MUSE_SCREEN_SLACK;
                    if (!(U == U)) U = 2.f;      // NaN 1/std or NaN samples: the exact kernel decides
                    if (live) prm.out_U[q][srow] = U;      // lanes = consecutive series: 128-byte stores
                }
            }
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    }
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u) : "memory");
    }
}

#endif  // __CUDACC__

}  // namespace muse
