// muse_screen_big.cuh -- the fp32 screening + fused second stage for FFT lengths 4096, 8192 and 16384
// (series of 2050 .. 16384 samples; BASELINE.json configs[3] is 10080 samples = one week at one per minute).
//
// Same mathematics and contract as score_screen_warp_kernel (muse_screen.cuh): a rigorous upper bound
// U = (1/n) sum_f |Y_f||X_f| / std + slack for every series (xcorr.go:160-197 gives max_k |cc[k]| <= U); a series
// whose U reaches the running cut-off goes on to conj(Y)*X, the inverse transform and the maxima of |cc| inside
// and outside the lag window (results.go:46-48), which tighten the bound and feed the cut-off.
//
// Shape: one series = M = n/2 complex points = 32 per thread on T = M/32 threads (one block per series, several
// blocks per SM), Stockham passes through shared memory.  What this file does differently from the first block
// kernel (round 1: 19.6 k warp instructions per series at 43 % issue utilisation):
//   * the LAST forward pass is mirror-paired: a thread transforms butterflies b and 1024 - b, whose outputs
//     k = b + 1024 j and M - k are exactly the mirror pairs of the real split, so the split, the magnitudes and
//     (second stage) conj(Y)*X run in registers -- one shared-memory exchange, two barriers and 64 LDS/STS per
//     thread fewer per series;
//   * the second stage's inverse transform runs the TRANSPOSED pass order (radix R, 32, 32 instead of 32, 32, R)
//     straight from that register layout, so no un-permuting exchange precedes it;
//   * every block walks a CONTIGUOUS range of series (row i+1 is pulled into L2 while row i is transformed), and
//     grouped runs keep a RUNNING lower bound per label group (muse_batch.go:87-89 keeps only a group's best
//     member): a member is refined only while its loose bound still reaches the best lower bound any member of
//     its group has shown so far, instead of every member of every group;
//   * row loads go out 16 x 16 bytes per thread at a time.
// All per-thread phases are __host__ __device__: tests/cpp/emulate_big.cpp runs them thread by thread on the CPU
// against a direct O(n^2) correlation before any GPU time is spent.
#pragma once

#include "muse_screen.cuh"

namespace muse {

template <int LOG2M>
struct ScreenBigCfg {
    static_assert(LOG2M >= 11 && LOG2M <= 13, "big kernel: n = 4096, 8192, 16384");
    static constexpr int M = 1 << LOG2M;
    static constexpr int P = 32;
    static constexpr int T = M / P;                   // threads per series == block size (64, 128, 256)
    static constexpr int NWARP = T / 32;
    static constexpr int LR = LOG2M - 10;             // last forward pass / first inverse pass radix R = M / 1024
    static constexpr int R = 1 << LR;                 // 2, 4, 8
    static constexpr int NB = P / R;                  // butterflies of radix R per thread (16, 8, 4)
    static constexpr int NPAIR = NB / 2;              // mirror pairs of butterflies per thread
    static constexpr int TP = T + (T >> 5);           // pad5(t + T*x) = pad5(t) + TP*x
    static constexpr int JP = 1024 + 32;              // pad5(b + 1024*j) = pad5(b) + JP*j
    static constexpr int TR = T + (T >> LR);          // padR(t + T*x) = padR(t) + TR*x
    // exchange buffer: forward and inverse pass 1' -> 2' use pad5 (one spare element per 32), inverse pass 0' -> 1'
    // uses padR (one spare element per R)
    static constexpr int SM_ELEMS = M + (M >> LR) + 2;
    static constexpr size_t EX_BYTES = ((size_t)SM_ELEMS * 8 + 127) / 128 * 128;
    // Table loads were the kernel's long-scoreboard stalls: two blocks' exchange buffers leave 64 KB of L1, and only 35 % of
    // the table sectors hit it.  Measured per 1.25 M x 10080 (ungrouped / grouped), tables in shared memory: none 39.9 / 42.9 ms,
    // forward twiddles 38.8 / 41.3 ms (the default), + sb 40.4 / 43.2 ms, + inverse twiddles 41.0 / 43.5 ms (what is left of L1
    // is then too small for the rest).
#ifndef MUSE_BIG_SMEM_TW
#define MUSE_BIG_SMEM_TW 1
#endif
#if MUSE_BIG_SMEM_TW
    // the forward passes' twiddles (TWF0, TWF1: 22.5 KB at n = 16384) ride in shared memory behind the exchange buffer;
    // MUSE_BIG_SMEM_TW = 2: the pair-bound weights sb too (16 KB); 3: the inverse passes' twiddles instead (16 KB)
    static constexpr int TW_SMEM = MUSE_BIG_SMEM_TW == 3 ? (10 * T + 31 * (T / 32) + 1024 + 31 * 32) : (10 * T + 31 * (T / 32));
    static constexpr size_t SB_SMEM = MUSE_BIG_SMEM_TW == 2 ? (size_t)(M / 2) * 4 : 0;
    static constexpr size_t SMEM = EX_BYTES + (size_t)TW_SMEM * 8 + SB_SMEM;
#else
    static constexpr size_t SMEM = (size_t)SM_ELEMS * 8;
#endif
    // fp32 twiddle tables of this kernel, ONE array (fill_big_twiddles), sized to stay L1-resident next to two blocks'
    // exchange buffers (a full W_M^(j t) table is 64 KB at n = 16384 and every load of it went to L2):
    //   forward pass 0: W_M^(j t) = W_M^(8 a t) * W_M^(b t), j = 8 a + b:   A [3 x T] (a = 1..3), B [7 x T] (b = 1..7)
    //   forward pass 1: W_T^(j p) [31 x T/32]
    //   inverse pass 0': W_M^b [1024], the higher powers W_M^(j b), j < R, by multiplication
    //   inverse pass 1': W_1024^(j p) [31 x 32]
    static constexpr int TWF0_OFF = 0;
    static constexpr int TWF1_OFF = 10 * T;
    static constexpr int TWI0_OFF = TWF1_OFF + 31 * (T / 32);
    static constexpr int TWI1_OFF = TWI0_OFF + 1024;
    static constexpr int TW_TOTAL = TWI1_OFF + 31 * 32;
};

template <typename TW, typename FN>
inline void fill_big_twiddles(int log2m, TW *out, FN unit_root /* (num, den) -> TW */) {
    const int M = 1 << log2m, T = M / 32;
    for (int a = 1; a < 4; a++)
        for (int t = 0; t < T; t++) out[(a - 1) * T + t] = unit_root((long long)8 * a * t, (long long)M);
    for (int b = 1; b < 8; b++)
        for (int t = 0; t < T; t++) out[(3 + b - 1) * T + t] = unit_root((long long)b * t, (long long)M);
    TW *p1 = out + 10 * T;
    for (int j = 1; j < 32; j++)
        for (int p = 0; p < T / 32; p++) p1[(j - 1) * (T / 32) + p] = unit_root((long long)j * p, (long long)T);
    TW *i0 = p1 + 31 * (T / 32);
    for (int b = 0; b < 1024; b++) i0[b] = unit_root((long long)b, (long long)M);
    TW *i1 = i0 + 1024;
    for (int j = 1; j < 32; j++)
        for (int p = 0; p < 32; p++) i1[(j - 1) * 32 + p] = unit_root((long long)j * p, 1024LL);
}

MUSE_HD float big_sqrt(float x) {
#if defined(__CUDA_ARCH__)
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
#else
    return sqrtf(x);
#endif
}

MUSE_HD float4 big_load_f4(const float4 *p) {
#if defined(__CUDA_ARCH__)
    // 16-byte table entry that must not displace the per-pass twiddles from L1
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
    return r;
#else
    return *p;
#endif
}

// ---- forward passes (Stockham, radix 32, 32, R) ------------------------------------------------------------
// pass 0: inputs v[j] = z[t + T*j]; writes y[32 t + j] * W_M^(j t) (pad5)
// NZ: rows (register slots) of the zero-padded input that hold samples; the first radix-4 stage is pruned for the rest
template <int LOG2M, int NZ = 32>
MUSE_HD void big_fwd_pass0(cf *v, cf *sm, int t, const cf *tw) {
    using C = ScreenBigCfg<LOG2M>;
    Dft32Lead<NZ, float>::run(v);
    cf *dst = sm + 33 * t;
    const cf *twt = tw + C::TWF0_OFF + t;
    cf wb[8];
#pragma unroll
    for (int b = 1; b < 8; b++) wb[b] = twt[(3 + b - 1) * C::T];
    dst[0] = v[Perm<32>::at(0)];
#pragma unroll
    for (int b = 1; b < 8; b++) dst[b] = cmul(v[Perm<32>::at(b)], wb[b]);
#pragma unroll
    for (int a = 1; a < 4; a++) {
        const cf wa = twt[(a - 1) * C::T];
        dst[8 * a] = cmul(v[Perm<32>::at(8 * a)], wa);
#pragma unroll
        for (int b = 1; b < 8; b++) dst[8 * a + b] = cmul(v[Perm<32>::at(8 * a + b)], cmul(wa, wb[b]));
    }
}
// loads of passes whose butterfly is the thread itself: inputs t + T*j under pad5
template <int LOG2M>
MUSE_HD void big_load_stride_t(cf *v, const cf *sm, int t) {
    using C = ScreenBigCfg<LOG2M>;
    const int pt = t + (t >> 5);
#pragma unroll
    for (int j = 0; j < 32; j++) v[j] = sm[pt + C::TP * j];
}
// pass 1: butterfly t: p = t / 32, q = t % 32; writes y[q + 1024 p + 32 j] * W_T^(j p) (pad5)
template <int LOG2M>
MUSE_HD void big_fwd_pass1(cf *v, cf *sm, int t, const cf *twb) {
    using C = ScreenBigCfg<LOG2M>;
    Dft<32, float>::run(v);
    const int p = t >> 5, q = t & 31;
    cf *dst = sm + q + 1056 * p;
    const cf *tw = twb + C::TWF1_OFF + p;
    dst[0] = v[Perm<32>::at(0)];
#pragma unroll
    for (int j = 1; j < 32; j++) dst[33 * j] = cmul(v[Perm<32>::at(j)], tw[(j - 1) * (C::T / 32)]);
}
// Butterflies of the last pass that thread t owns: pair slot c2 holds b_lo = u and b_hi = 1024 - u, u = t + T*c2
// (u == 0: b_lo = 0 and b_hi = 512, the two butterflies that are their own mirrors).
MUSE_HD int big_b_hi(int u) { return u == 0 ? 512 : 1024 - u; }
// last pass: radix R over inputs b + 1024 j; on return v[(2 c2 + h) R + Perm<R>(j)] = Z[b + 1024 j]
template <int LOG2M>
MUSE_HD void big_fwd_last(cf *v, const cf *sm, int t) {
    using C = ScreenBigCfg<LOG2M>;
#pragma unroll
    for (int c2 = 0; c2 < C::NPAIR; c2++) {
        const int u = t + C::T * c2;
        const int bh = big_b_hi(u);
        const int plo = u + (u >> 5), phi = bh + (bh >> 5);
#pragma unroll
        for (int j = 0; j < C::R; j++) {
            v[(2 * c2) * C::R + j] = sm[plo + C::JP * j];
            v[(2 * c2 + 1) * C::R + j] = sm[phi + C::JP * j];
        }
    }
#pragma unroll
    for (int i = 0; i < C::NB; i++) Dft<C::R, float>::run(v + i * C::R);
}

// One mirror pair of the real split: 2 Y_k = e + w o, 2 conj(Y_(M-k)) = e - w o (muse_fft.cuh); adds
// |2Y_k| A[k] + |2Y_(M-k)| A[M-k] to acc2.  s = (w_k, A[k], A[M-k]).
MUSE_HD void big_split_acc(cf zk, cf zm, float4 s, cf &acc2) {
    const cf zmc = cconj(zm);
    const cf e = cadd(zk, zmc);
    const cf o = cmul_negi(csub(zk, zmc));
    const cf wo = cmul(o, cf{s.x, s.y});
    const cf y1 = cadd(e, wo);
    const cf y2 = csub(e, wo);
    const cf q1 = pmul(y1, y1), q2 = pmul(y2, y2);
    const cf mag{big_sqrt(q1.x + q1.y), big_sqrt(q2.x + q2.y)};
    acc2 = pfma(mag, cf{s.z, s.w}, acc2);
}

// The pair bound of muse_screen.cuh on the same pair: |2Y_k| A[k] + |2Y_(M-k)| A[M-k] <= sqrt(|e|^2 + |d|^2) B[k'].
MUSE_HD void big_pair_acc(cf zk, cf zm, float b, cf &acc2) {
    const cf zmc = cconj(zm);
    const cf e = cadd(zk, zmc);
    const cf d = csub(zk, zmc);
    const cf q = pfma(d, d, pmul(e, e));
    acc2.x = fmaf(big_sqrt(q.x + q.y), b, acc2.x);
}
// PAIR: the cheaper, looser pair bound (what the kernel uses: 45.8 -> 43.0 ms per 1.25 M x 10080 ungrouped, 48.0 -> 46.4 ms
// grouped, with 27 % more second stages); !PAIR: the bin-by-bin sum (MUSE_BIG_BINS builds, and the CPU emulation's reference)
#define MUSE_BIG_ACC(zk, zm, idx)                                        \
    do {                                                                 \
        if constexpr (PAIR) big_pair_acc(zk, zm, sb[idx], acc2);         \
        else big_split_acc(zk, zm, big_load_f4(sw + (idx)), acc2);       \
    } while (0)

// The thread's share of sum_k |2Y_k| A_k, from the registers big_fwd_last left.  Pair slot c2, index j:
// k = u + 1024 j sits in lo[Perm(j)], its mirror M - k = (1024 - u) + 1024 (R-1-j) in hi[Perm(R-1-j)]; the table
// entry is that of k' = min(k, M - k).  u == 0 (thread 0, slot 0): butterfly 0 pairs j with R - j (j = 0: DC and
// Nyquist; j = R/2: bin M/2, its own mirror, |2Y| = 2|Z|), butterfly 512 pairs j with R-1-j.
template <int LOG2M, bool PAIR = false>
MUSE_HD float big_split_bound(const cf *v, int t, const float4 *sw, float a_mid, const float *sb = nullptr) {
    (void)sb;
    using C = ScreenBigCfg<LOG2M>;
    constexpr int R = C::R, M = C::M;
    cf acc2{0.f, 0.f};
    float extra = 0.f;
#pragma unroll
    for (int c2 = 0; c2 < C::NPAIR; c2++) {
        const int u = t + C::T * c2;
        const cf *lo = v + (2 * c2) * R, *hi = v + (2 * c2 + 1) * R;
        if (c2 == 0 && u == 0) {
            MUSE_BIG_ACC(lo[Perm<R>::at(0)], lo[Perm<R>::at(0)], 0);
#pragma unroll
            for (int j = 1; j < R / 2; j++) MUSE_BIG_ACC(lo[Perm<R>::at(j)], lo[Perm<R>::at(R - j)], 1024 * j);
            {
                const cf z = lo[Perm<R>::at(R / 2)];
                const cf q = pmul(z, z);
                extra = big_sqrt(q.x + q.y) * (2.f * a_mid);
            }
#pragma unroll
            for (int j = 0; j < R / 2; j++) MUSE_BIG_ACC(hi[Perm<R>::at(j)], hi[Perm<R>::at(R - 1 - j)], 512 + 1024 * j);
        } else {
#pragma unroll
            for (int j = 0; j < R; j++) {
                const cf a = lo[Perm<R>::at(j)], b = hi[Perm<R>::at(R - 1 - j)];
                if (j < R / 2) MUSE_BIG_ACC(a, b, u + 1024 * j);
                else MUSE_BIG_ACC(b, a, M - u - 1024 * j);
            }
        }
    }
    return acc2.x + acc2.y + extra;
}

// Second stage, in place in the same registers: conj(Y)*X on every mirror pair (pointwise_pair stores the swapped
// values the inverse-as-forward transform wants).
template <int LOG2M>
MUSE_HD void big_pointwise(cf *v, int t, const float4 *sw, const float4 *sx, cf x_mid) {
    using C = ScreenBigCfg<LOG2M>;
    constexpr int R = C::R, M = C::M;
#pragma unroll
    for (int c2 = 0; c2 < C::NPAIR; c2++) {
        const int u = t + C::T * c2;
        cf *lo = v + (2 * c2) * R, *hi = v + (2 * c2 + 1) * R;
        if (c2 == 0 && u == 0) {
            cf ok, om;
            {
                const float4 s = big_load_f4(sw), x = big_load_f4(sx);
                pointwise_pair(lo[Perm<R>::at(0)], lo[Perm<R>::at(0)], cf{s.x, s.y}, cf{x.x, x.y}, cf{x.z, x.w}, ok, om);
                lo[Perm<R>::at(0)] = ok;
            }
#pragma unroll
            for (int j = 1; j < R / 2; j++) {
                const float4 s = big_load_f4(sw + 1024 * j), x = big_load_f4(sx + 1024 * j);
                pointwise_pair(lo[Perm<R>::at(j)], lo[Perm<R>::at(R - j)], cf{s.x, s.y}, cf{x.x, x.y}, cf{x.z, x.w}, ok, om);
                lo[Perm<R>::at(j)] = ok;
                lo[Perm<R>::at(R - j)] = om;
            }
            {
                cf &mid = lo[Perm<R>::at(R / 2)];      // bin M/2: w = exp(-i pi/2) = -i
                pointwise_pair(mid, mid, cf{0.f, -1.f}, x_mid, x_mid, ok, om);
                mid = ok;
            }
#pragma unroll
            for (int j = 0; j < R / 2; j++) {
                const float4 s = big_load_f4(sw + 512 + 1024 * j), x = big_load_f4(sx + 512 + 1024 * j);
                pointwise_pair(hi[Perm<R>::at(j)], hi[Perm<R>::at(R - 1 - j)], cf{s.x, s.y}, cf{x.x, x.y}, cf{x.z, x.w}, ok, om);
                hi[Perm<R>::at(j)] = ok;
                hi[Perm<R>::at(R - 1 - j)] = om;
            }
        } else {
#pragma unroll
            for (int j = 0; j < R; j++) {
                cf &a = lo[Perm<R>::at(j)], &b = hi[Perm<R>::at(R - 1 - j)];
                cf ok, om;
                if (j < R / 2) {
                    const float4 s = big_load_f4(sw + u + 1024 * j), x = big_load_f4(sx + u + 1024 * j);
                    pointwise_pair(a, b, cf{s.x, s.y}, cf{x.x, x.y}, cf{x.z, x.w}, ok, om);
                    a = ok;
                    b = om;
                } else {
                    const int kk = M - u - 1024 * j;
                    const float4 s = big_load_f4(sw + kk), x = big_load_f4(sx + kk);
                    pointwise_pair(b, a, cf{s.x, s.y}, cf{x.x, x.y}, cf{x.z, x.w}, ok, om);
                    b = ok;
                    a = om;
                }
            }
        }
    }
}

// ---- inverse as a forward transform of the swapped values, pass order R, 32, 32 ------------------------------
// pass 0': butterfly b has its inputs x[b + 1024 j] in registers (big_fwd_last's layout, slot Perm<R>(j));
// writes y[R b + j] * W_M^(j b) under padR: (R + 1) b + j
template <int LOG2M>
MUSE_HD void big_inv_pass0(cf *v, cf *sm, int t, const cf *twi) {
    using C = ScreenBigCfg<LOG2M>;
    constexpr int R = C::R;
#pragma unroll
    for (int c2 = 0; c2 < C::NPAIR; c2++) {
        const int u = t + C::T * c2;
#pragma unroll
        for (int h = 0; h < 2; h++) {
            const int b = h == 0 ? u : big_b_hi(u);
            cf *x = v + (2 * c2 + h) * R;
            cf w[R];
#pragma unroll
            for (int j = 0; j < R; j++) w[j] = x[Perm<R>::at(j)];
            Dft<R, float>::run(w);
            cf *dst = sm + (R + 1) * b;
            dst[0] = w[Perm<R>::at(0)];
            cf pw[R];                          // W_M^(j b): j = 1 from the table, the rest by products of depth <= 3
            pw[1] = twi[C::TWI0_OFF + b];
#pragma unroll
            for (int j = 2; j < R; j++) pw[j] = cmul(pw[j / 2], pw[j - j / 2]);
#pragma unroll
            for (int j = 1; j < R; j++) dst[j] = cmul(w[Perm<R>::at(j)], pw[j]);
        }
    }
}
// pass 1': butterfly t: p = t / R, q = t % R; inputs t + T j under padR; writes y[q + 32 R p + R j] * W_1024^(j p) (pad5)
template <int LOG2M>
MUSE_HD void big_inv_pass1_load(cf *v, const cf *sm, int t) {
    using C = ScreenBigCfg<LOG2M>;
    const int ptr = t + (t >> C::LR);
#pragma unroll
    for (int j = 0; j < 32; j++) v[j] = sm[ptr + C::TR * j];
}
template <int LOG2M>
MUSE_HD void big_inv_pass1(cf *v, cf *sm, int t, const cf *twi) {
    using C = ScreenBigCfg<LOG2M>;
    constexpr int R = C::R;
    Dft<32, float>::run(v);
    const int p = t >> C::LR, q = t & (R - 1);
    cf *dst = sm + q + 33 * R * p;
    const cf *tw = twi + C::TWI1_OFF + p;
    dst[0] = v[Perm<32>::at(0)];
#pragma unroll
    for (int j = 1; j < 32; j++) dst[R * j + ((R * j) >> 5)] = cmul(v[Perm<32>::at(j)], tw[(j - 1) * 32]);
}
// pass 2': inputs t + T j (pad5, big_load_stride_t), radix 32, no twiddles: v[Perm<32>(j)] = (cc'[2i+1], cc'[2i]),
// i = t + T j, cc' = std * cc rotated by pad (zeros trail here, lead in xcorr.go:176-181).
// Maxima of |cc'| inside / outside the lag window (rotated index: (idx - win_lo) mod n <= win_len).
template <int LOG2M>
MUSE_HD void big_window_max(const cf *v, int t, int win_lo, int win_len, float &m_in, float &m_out) {
    using C = ScreenBigCfg<LOG2M>;
    m_in = 0.f;
    m_out = 0.f;
    const int base = 2 * t - win_lo;
#pragma unroll
    for (int j = 0; j < 32; j++) {
        const int off = 2 * C::T * j;
        window_pair(v[Perm<32>::at(j)], base + off, win_len, 2 * C::M - 1, window_row_hit(off, 2 * C::T, win_lo, win_len, 2 * C::M), m_in,
                    m_out);
    }
}

#if defined(__CUDACC__)

__device__ __forceinline__ void big_l2_prefetch(const void *p, unsigned bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}

#ifndef MUSE_BIG_LOAD_BATCH
#define MUSE_BIG_LOAD_BATCH 16
#endif

// NZ = ceil(Nh / T) in 17 .. 32 as a template parameter (the n = 16384 launcher instantiates all sixteen, as the warp
// kernel does): rows below NZ - 1 load without a predicate, row NZ - 1 with one, the rows above are zeros that are neither
// loaded nor converted, and the first radix-4 stage of pass 0 skips them.  NZ = 0: decided at run time (n = 4096, 8192).
template <int LOG2M, int MINB, int NZ = 0>
__global__ void __launch_bounds__(ScreenBigCfg<LOG2M>::T, MINB)
score_screen_big_kernel(const ScreenParams prm) {
    using C = ScreenBigCfg<LOG2M>;
    constexpr int P = 32, T = C::T, NW = C::NWARP, LB = MUSE_BIG_LOAD_BATCH;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ float2 red_f[2][NW];                  // block reductions, double-buffered by use
    __shared__ unsigned bc_word[2];                  // running cut-off and the group's running lower bound, from thread 0
    cf *sm = reinterpret_cast<cf *>(smem_raw);
#if MUSE_BIG_SMEM_TW
    cf *s_tw = reinterpret_cast<cf *>(smem_raw + C::EX_BYTES);
    for (int i = threadIdx.x; i < C::TW_SMEM; i += C::T) s_tw[i] = prm.twi[i];
    float *s_sb = reinterpret_cast<float *>(s_tw + C::TW_SMEM);
    if (C::SB_SMEM)
        for (int i = threadIdx.x; i < C::M / 2; i += C::T) s_sb[i] = prm.sb[i];
    __syncthreads();
    const cf *twf = s_tw;
    const cf *twinv = MUSE_BIG_SMEM_TW == 3 ? s_tw : prm.twi;
    const float *sbp = C::SB_SMEM ? s_sb : prm.sb;
#else
    const cf *twf = prm.twi;
    const cf *twinv = prm.twi;
    const float *sbp = prm.sb;
#endif

    const int t = threadIdx.x;
    const int N = prm.N;
    const int Nh = (N + 1) >> 1;      // complex slots holding samples (odd N: the pad column of the last one holds the row's mean, RowStat)
    const int count = (int)prm.count;
    const unsigned row_bytes = (unsigned)(N + (N & 1)) * 8u;
    // contiguous range of series per block
    const int chunk = (count + (int)gridDim.x - 1) / (int)gridDim.x;
    const int pos_lo = (int)blockIdx.x * chunk;
    const int pos_hi = min(pos_lo + chunk, count);
    // the series of work item pos (filtered runs: the listed rows, so the prefetch fetches listed rows, not a range)
    auto row_of = [&](int pos) { return prm.rows ? prm.rows[pos] : pos; };
    if (t == 0 && pos_lo < pos_hi) big_l2_prefetch(prm.slab + (int64_t)row_of(pos_lo) * prm.ld, row_bytes);

    for (int pos = pos_lo; pos < pos_hi; pos++) {
        const int row = row_of(pos);
        const double *rowp = prm.slab + (int64_t)row * prm.ld;
        unsigned cut_raw = 0u, lg_raw = 0u;
        unsigned long long *gslot = nullptr;
        if (t == 0) {
            if (pos + 1 < pos_hi) big_l2_prefetch(prm.slab + (int64_t)row_of(pos + 1) * prm.ld, row_bytes);
            cut_raw = ld_relaxed_u32(prm.cut_bits);
            if (prm.group_L) {
                gslot = prm.group_L + prm.slot_of[row];
                lg_raw = ld_relaxed_u32(reinterpret_cast<const unsigned *>(gslot));      // low word: float bits of the best lower bound so far
            }
        }
        const RowStat rs = prm.row_stat[row];
        const double mu = rs.mean;

        // ---- centred samples -> fp32 registers, LB x 16 bytes in flight per thread ----
        cf v[P];
#pragma unroll
        for (int b0 = 0; b0 < P; b0 += LB) {
            cd x[LB];
#pragma unroll
            for (int q = 0; q < LB; q++) {
                const int j = t + (b0 + q) * T;
if constexpr (NZ > 0) {
                    if (b0 + q < NZ - 1) x[q] = load_pair_stream(rowp + 2 * j);
                    else if (b0 + q == NZ - 1) x[q] = j < Nh ? load_pair_stream(rowp + 2 * j) : cd{mu, mu};
                    else x[q] = cd{mu, mu};
                } else {
                    // rows below 16 always hold samples (N > n/2): no predicate, no (mu, mu) preset (C4: 42.1 -> 41.2 ms)
                    x[q] = (b0 + q < P / 2 || j < Nh) ? load_pair_stream(rowp + 2 * j) : cd{mu, mu};
                }
            }
#pragma unroll
            for (int q = 0; q < LB; q++) {
                if (NZ > 0 && b0 + q >= NZ) v[b0 + q] = cf{0.f, 0.f};
                else v[b0 + q] = cf{(float)(x[q].x - mu), (float)(x[q].y - mu)};      // exactly 0 in the padding
            }
        }

        // ---- forward FFT_M; ends with Z in registers in mirror-paired order ----
        big_fwd_pass0<LOG2M, NZ == 0 ? 32 : NZ>(v, sm, t, twf);
        __syncthreads();
        big_load_stride_t<LOG2M>(v, sm, t);
        __syncthreads();
        big_fwd_pass1<LOG2M>(v, sm, t, twf);
        __syncthreads();
        big_fwd_last<LOG2M>(v, sm, t);

        // ---- bound ----
#if defined(MUSE_BIG_BINS)
        float acc = big_split_bound<LOG2M, false>(v, t, prm.sw, prm.a_mid, sbp);
#else
        float acc = big_split_bound<LOG2M, true>(v, t, prm.sw, prm.a_mid, sbp);
#endif
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
        if ((t & 31) == 0) red_f[0][t >> 5].x = acc;
        if (t == 0) {
            bc_word[0] = cut_raw;
            bc_word[1] = lg_raw;
        }
        __syncthreads();                                             // also: every last-pass load of the exchange buffer is done
        acc = red_f[0][0].x;
#pragma unroll
        for (int w = 1; w < NW; w++) acc += red_f[0][w].x;
        const float cut_now = __uint_as_float(bc_word[0]);
        const float lg_now = __uint_as_float(bc_word[1]);
        // rstd is NaN for a row no fp32 statement may be made about (RowStat); NaN/Inf samples make acc NaN:
        // either way the bound is NaN and the exact kernel decides
        float U = acc * rs.rstd * 1.00001f + MUSE_SCREEN_SLACK;
        if (!(U == U)) U = 2.f;
        float L = -1.f;
        signed char W = 0;
        if (U >= cut_now && U >= lg_now && U < 1.5f) {               // block-uniform
            big_pointwise<LOG2M>(v, t, prm.sw, prm.sx, prm.x_mid);
            big_inv_pass0<LOG2M>(v, sm, t, twinv);
            __syncthreads();
            big_inv_pass1_load<LOG2M>(v, sm, t);
            __syncthreads();
            big_inv_pass1<LOG2M>(v, sm, t, twinv);
            __syncthreads();
            big_load_stride_t<LOG2M>(v, sm, t);
            Dft<32, float>::run(v);
            float m_in, m_out;
            big_window_max<LOG2M>(v, t, prm.win_lo, prm.win_len, m_in, m_out);
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                m_in = fmaxf(m_in, __shfl_xor_sync(0xffffffffu, m_in, off));
                m_out = fmaxf(m_out, __shfl_xor_sync(0xffffffffu, m_out, off));
            }
            if ((t & 31) == 0) red_f[1][t >> 5] = make_float2(m_in, m_out);
            __syncthreads();
            float2 mx = red_f[1][0];
#pragma unroll
            for (int w = 1; w < NW; w++) {
                mx.x = fmaxf(mx.x, red_f[1][w].x);
                mx.y = fmaxf(mx.y, red_f[1][w].y);
            }
            const float rstd = rs.rstd;
            const float s_in = mx.x * rstd, s_out = mx.y * rstd;
            U = refine_decide(U, s_in, s_out, L, prm.grouped);
            if (prm.grouped) {
                // the window is the business of the group's representative only (results.go:46-48 after muse_batch.go:87-89)
                float Lw = -1.f;
                const float uw = refine_decide(2.f, s_in, s_out, Lw, 0);
                W = uw < 0.f ? -1 : (Lw >= 0.f ? 1 : 0);
            }
            if (t == 0) {
                atomicAdd(prm.n_refined, 1ull);
                if (gslot && L > lg_now) atomicMax(gslot, (unsigned long long)__float_as_uint(L));
            }
            if (!prm.grouped && t < 32 && L >= prm.thr && L >= cut_now) cut_count_and_raise(prm.cut_bits, prm.cut_hist, prm.top_n, L, t);
        }
        if (t == 0) {
            prm.out_U[row] = U;
            if (prm.out_L) prm.out_L[row] = L;
            if (prm.out_W) prm.out_W[row] = W;
        }
        // no barrier here: the exchange buffer was last read before the reduction barrier of whichever path ran, and
        // red_f / bc_word are next written three barriers into the next iteration
    }
}

#endif  // __CUDACC__

}  // namespace muse
