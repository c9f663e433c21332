// muse_screen.cuh -- fp32 screening pass: a rigorous UPPER BOUND on every series' score.
//
// For the score of xcorr.go:160-197 / muse_batch.go:74-77,
//     score = min(1, max_k |cc[k]|),   cc[k] = (1/n) * sum_f C_f * exp(+2*pi*i*f*k/n),
//     C_f = conj(Y_f) * X_f,
// the triangle inequality gives  max_k |cc[k]| <= (1/n) * sum_f |Y_f| * |X_f|  =: U.
// The warp and sub-warp kernels (n <= 2048) bound U itself once more, by Cauchy-Schwarz on each mirror pair (f, n/2 - f)
// of the half-length transform: |2Y_k| A[k] + |2Y_(M-k)| A[M-k] <= sqrt(|2Y_k|^2 + |2Y_(M-k)|^2) sqrt(A[k]^2 + A[M-k]^2), and
// the first factor is sqrt(2 (|e|^2 + |d|^2)) straight from e = Z_k + conj(Z_(M-k)), d = Z_k - conj(Z_(M-k)) -- no split
// twiddle, one square root per pair.  Still an upper bound on the score, a little looser (it passes 5.5 % of the
// benchmark's series to the second stage instead of 3.6 %), a third cheaper in the loop every series runs.
// U needs only the FORWARD transform of the series, no inverse, no arg-max.  The kernel
// computes U in fp32 (forward FFT_M of the half-length packing, split, |Y_f|, dot with the
// precomputed |X_f| weights) and adds a slack that covers every fp32 rounding in the
// chain, so that U >= exact fp64 score holds for every series.  Batch.Run then sends only
// series whose U can still reach the top-N cut-off through the exact fp64 kernel
// (muse_exact.cuh); its results are therefore identical to scoring everything exactly.
//
// Error budget (all in units of the normalised score, |cc| <= 1):
//   * input: y - pivot is formed in fp64, then rounded to fp32: |err| <= 2^-24 * 2*max|y-mean|
//     per sample, and max|y-mean| <= sqrt(N-1)*std, so the induced cc error is
//     <= ||x'||_2 * sqrt(N) * 2^-23 * sqrt(N-1) * ... <= 2^-23 * sqrt(N) ~ 4.5e-6 at N = 1440;
//   * fp32 FFT (radix-32 x radix-32): relative l2 error of the spectrum <~ 10 * 2^-24 ~ 6e-7,
//     which moves U by at most ||X||_2*||dY||_2/n <= 6e-7;
//   * mean, std, magnitude and accumulation roundings: each <= ~1e-6 relative.
// The sum stays below 2e-5 for N <= 16384; SCREEN_SLACK = 1e-4 leaves a 5x margin over that budget and 450x over the
// worst error observed on the adversarial generator at every FFT length (2.2e-7, profiles/screen_error_survey.json).
// The slack is what sends series to the exact kernel: every series whose score lies within 2 slacks of the top-N cut-off
// is re-scored in fp64 (at 2e-4, rounds 1 and 2a: 4.0 k of 1 M series at C3, 777 k of 256 M pairs = 11.7 of 62 ms at C5).
// tests/test_gpu_screen.py checks U >= exact on adversarial inputs (offsets of 1e9, spikes,
// 1e-12 and 1e+12 amplitudes, trends) and records the smallest observed margin.
#pragma once

#include <vector_functions.h>   // float4 / make_float4 (host builds of the emulators too)
#include <vector_types.h>

#include "muse_score.cuh"

namespace muse {

typedef cx<float> cf;

#ifndef MUSE_SCREEN_SLACK
#define MUSE_SCREEN_SLACK 1e-4f
#endif
// warp kernel: sample variance window.  std >= 1e-10: a flushed magnitude (< 1.1e-19) is below
// 1.1e-9 in units of the score per bin; std <= 1e14: |2Y_k|^2 <= (4*N*std)^2 * N < 3e38.
#define MUSE_SCREEN_VAR_MIN 1e-20f
#define MUSE_SCREEN_VAR_MAX 1e28f
// |mean| <= 1e8 * std: the fp64 sum of N values of size |mean| is uncertain by at most
// N * 2^-53 * N * |mean| (sequential worst case), i.e. the mean by 1.6e-13 * |mean| at N = 1440; a
// shift of the mean by d moves a score by at most d / std, so the limit keeps the disagreement
// between this kernel's mean and the exact kernel's (summed in another order) below 2e-5, a tenth of
// the slack.  Rows beyond it are flagged once per store by row_offset_flags_kernel (a register for
// the mean across the FFT costs this kernel 5 %) and always go to the exact kernel.
#define MUSE_SCREEN_OFFSET_MAX 1e8
// running cut-off: lower bounds are counted in MUSE_CUT_BINS = 64^3 bins of [0, 1] (3.8e-6 wide, far below the
// slack), with 64^2 and 64 group counters above them (MUSE_CUT_WORDS counters in all)
#define MUSE_CUT_BINS 262144
#define MUSE_CUT_WORDS (64 + 64 * 64 + MUSE_CUT_BINS)

// The running cut-off of a run (of one query of a multi-query run), armed by init_cut_kernel / init_cut_batch_kernel.
struct CutState {
    unsigned bits;                    // running lower bound on the final top-N cut-off (float bits, only ever raised)
    unsigned claims;                  // warp kernel: claims of series handed out so far
    unsigned long long refined;       // series that took the fused second stage
    unsigned hist[MUSE_CUT_WORDS];    // 64 coarse, 64*64 middle, 64^3 fine counts of lower bounds
};

// Per-row statistics of the store, computed once per appended row (the batched mean/std kernel of the
// z-normalisation, xcorr.go:84-95): the fp64 mean, and 1/std in fp32 -- or NaN when no fp32 statement may be
// made about the row (constant row, variance outside [MUSE_SCREEN_VAR_MIN, MUSE_SCREEN_VAR_MAX], non-finite
// samples, |mean| > MUSE_SCREEN_OFFSET_MAX * std): the NaN propagates into the bound and sends the series to
// the exact kernel.
struct alignas(16) RowStat {
    double mean;
    float rstd;
    unsigned pad;
};

struct ScreenParams {
    const double *slab;
    int64_t ld;
    int64_t count;
    int N;
    const cf *twp;        // per-pass twiddles (fill_pass_twiddles), fp32
    const float4 *sw;     // (w_k.x, w_k.y, A[k], A[M-k]) for k < M/2: split twiddle exp(-2*pi*i*k/n), weights |X|/(2n)*(1|2) rounded up
    const float *sb;      // warp and sub-warp kernels: B[k] = sqrt(2 (A[k]^2 + A[M-k]^2)) rounded up, k < M/2 (the pair bound below)
    float a_mid;          // A[M/2]
    // ---- fused second stage ----
    const float4 *sx;     // (Xt[k].x, Xt[k].y, Xt[M-k].x, Xt[M-k].y) in fp32, k < M/2 (Xt = X/(2n))
    cf x_mid;             // Xt[M/2]
    float *out_L;         // [count] certain lower bound on a score that certainly passes the lag filter, else -1
    const RowStat *row_stat;          // [count] fp64 mean and fp32 1/std of each row (row_stats_kernel, once per appended row)
    unsigned *cut_bits;   // running lower bound on the final top-N cut-off (float bits, only ever raised)
    unsigned *cut_hist;   // [MUSE_CUT_WORDS] 64 coarse, 64*64 middle, 64^3 fine counts of lower bounds
    unsigned long long *n_refined;
    unsigned *next_claim; // warp kernel: counter of the claims of series handed out so far (cleared with the cut-off state)
    int top_n;            // series needed above the cut before it may rise
    int win_lo, win_len;  // lag window in the kernel's rotated cc index: (idx - win_lo) mod n <= win_len
    float thr;            // threshold rounded up to fp32 (a lower bound must reach it to count)
    int grouped;          // grouped run: every series is refined, bounds ignore the window, no cut-off
    float *out_U;         // [count] upper bound on the score (already clamped to <= 1 + slack)
    // ---- muse_screen_big.cuh ----
    const cf *twi;        // fp32 twiddles of the transposed inverse (fill_big_inverse_twiddles)
    const int64_t *slot_of;           // grouped runs: group-table slot of every series
    unsigned long long *group_L;      // grouped runs: [slots] running best lower bound of each group (float bits, low word)
    signed char *out_W;   // grouped runs: [count] 1 = peak certainly inside the lag window, -1 = certainly outside, 0 = undecided
};

// ---- maxima of |cc'| inside / outside the lag window (rotated index: (idx - win_lo) mod n <= win_len) ----
// A register pair r holds (cc'[idx + 1], cc'[idx]).  The pairs of one ROW of the transform's output (one register slot
// over the threads of a series) cover row_len consecutive lags starting at `off`; whether any of them can be inside
// the window depends on the row alone, i.e. on kernel parameters: the test runs on the uniform datapath and all but the
// two or three rows the window touches take one 3-input max per pair instead of two compares, two masks and four
// selects.  Used by the block kernel of muse_screen_big.cuh (C4: 43.0 -> 42.1 ms ungrouped, 46.1 -> 45.0 ms grouped); in the
// warp kernels the 32 uniform branches cost more than they save (C3 2.10 -> 2.17 ms, C5's second stages 39.3 -> 42.3 ms).
MUSE_HD bool window_row_hit(int off, int row_len, int win_lo, int win_len, int n) {
    const int d = (off - win_lo) & (n - 1);
    return d <= win_len || d > n - row_len;
}
MUSE_HD void window_pair(cx<float> r, int idx, int win_len, int nmask, bool hit, float &m_in, float &m_out) {
    const float a0 = fabsf(r.y), a1 = fabsf(r.x);
    if (hit) {
        const bool in0 = (idx & nmask) <= win_len;
        const bool in1 = ((idx + 1) & nmask) <= win_len;
        m_in = fmaxf(m_in, fmaxf(in0 ? a0 : 0.f, in1 ? a1 : 0.f));
        m_out = fmaxf(m_out, fmaxf(in0 ? 0.f : a0, in1 ? 0.f : a1));
    } else {
        m_out = fmaxf(m_out, fmaxf(a0, a1));
    }
}

#if defined(__CUDACC__)

template <int T>
__device__ __forceinline__ float group_sum_f(float x) {
#pragma unroll
    for (int off = T / 2; off > 0; off >>= 1) x += __shfl_xor_sync(0xffffffffu, x, off);
    return x;
}

// ---- cp.async.bulk / mbarrier plumbing of the screening kernels and the tensor-core bounds (SASS UBLKCP, SYNCS) ----
__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }

// a block's barriers are initialised, then published by one mbar_init_fence before the first copy or wait
__device__ __forceinline__ void mbar_init(unsigned bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect(unsigned bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_copy(unsigned dst, const void *src, unsigned bytes, unsigned bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
                 "r"(bytes), "r"(bar)
                 : "memory");
}
// one copy that completes the barrier's current phase
__device__ __forceinline__ void bulk_load(unsigned dst, const void *src, unsigned bytes, unsigned bar) {
    mbar_expect(bar, bytes);
    bulk_copy(dst, src, bytes, bar);
}
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity) {
    unsigned done;
    do {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
    } while (!done);
}

// sqrt.approx.ftz.f32 (one MUFU): 2 ulp, covered by the 1e-5 relative slack of the bound.  A
// subnormal |2Y_k|^2 is flushed to 0; the variance window MUSE_SCREEN_VAR_MIN/MAX keeps every
// bin that matters at the 1e-9 level far away from both ends of the fp32 range.
__device__ __forceinline__ float sqrt_approx(float x) {
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

__device__ __forceinline__ unsigned ld_relaxed_u32(const unsigned *p) {
    unsigned r;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(r) : "l"(p) : "memory");
    return r;
}

__device__ __forceinline__ void mbar_test(unsigned bar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "}\n" ::"r"(bar),
        "r"(parity)
        : "memory");
}

// Warp-collective: count the certain lower bound L of a series that certainly passes the filter and
// try to raise the running cut-off to the top_n-th largest lower bound counted so far.  All counts
// only grow, so every value read is a lower bound on the true count and any cut-off derived from
// them stays valid; lanes walk the counters from the top down, three levels of 64.
// One level of the walk: lanes read the 64 counters of a group from the top down (two per lane), find the
// counter in which the running count reaches `need`, and return its index within the group (-1: the
// group does not hold enough); `need` is reduced by what lies above that counter.
__device__ __forceinline__ int cut_level(const unsigned *cnt, int t, unsigned &need) {
    const unsigned h = ld_relaxed_u32(&cnt[63 - 2 * t]), l = ld_relaxed_u32(&cnt[62 - 2 * t]);
    unsigned incl = h + l;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const unsigned o = __shfl_up_sync(0xffffffffu, incl, off);
        if (t >= off) incl += o;
    }
    const unsigned excl = incl - (h + l);
    const unsigned hit = __ballot_sync(0xffffffffu, incl >= need);
    if (!hit) return -1;
    const int leader = __ffs(hit) - 1;
    const bool upper = excl + h >= need;
    const int idx = upper ? 63 - 2 * t : 62 - 2 * t;
    const unsigned above = upper ? excl : excl + h;
    need -= __shfl_sync(0xffffffffu, above, leader);
    return __shfl_sync(0xffffffffu, idx, leader);
}

// cut_bits / cut_hist / top_n: the cut-off state of ScreenParams, or of one query of a multi-query run.  Arguments that
// are kernel parameters are taken by reference here and in the blocks below, so that they are read where they are used.
// Counts the lower bound L in the three levels of the histogram.
__device__ __forceinline__ void cut_hist_add(unsigned *const &cut_hist, float L) {
    int bin = (int)(L * (float)MUSE_CUT_BINS);
    bin = bin < 0 ? 0 : (bin >= MUSE_CUT_BINS ? MUSE_CUT_BINS - 1 : bin);
    unsigned *coarse = cut_hist, *mid = coarse + 64, *fine = mid + 64 * 64;
    atomicAdd(&fine[bin], 1u);
    atomicAdd(&mid[bin >> 6], 1u);
    atomicAdd(&coarse[bin >> 12], 1u);
}

// Warp-collective: raises the cut-off to the lower edge of the bin that holds the top_n-th largest count (nothing when
// fewer were counted).
__device__ __forceinline__ void cut_walk(unsigned *const &cut_bits, const unsigned *const &cut_hist, const int &top_n, int t) {
    const unsigned *coarse = cut_hist, *mid = coarse + 64, *fine = mid + 64 * 64;
    unsigned need = (unsigned)top_n;
    const int c = cut_level(coarse, t, need);
    if (c < 0) return;
    const int m = cut_level(mid + c * 64, t, need);
    if (m < 0) return;                  // the three levels are incremented separately: a reader may see them out of step
    const int f = cut_level(fine + (c * 64 + m) * 64, t, need);
    if (f < 0) return;
    if (t == 0) atomicMax(cut_bits, __float_as_uint((float)((c * 64 + m) * 64 + f) / (float)MUSE_CUT_BINS));
}

__device__ __forceinline__ void cut_count_and_raise(unsigned *const &cut_bits, unsigned *const &cut_hist, const int &top_n, float L, int t) {
    if (t == 0) cut_hist_add(cut_hist, L);
    __syncwarp();
    cut_walk(cut_bits, cut_hist, top_n, t);
}

// Refined decision for one series from the fp32 maxima of |cc| inside / outside the lag window
// (both already divided by std): returns the new upper bound (-1: certainly outside the window,
// results.go:46-48 drops the series) and sets L when the peak is certainly inside.
// |fp32 cc - exact cc| <= MUSE_SCREEN_SLACK / 2 in score units (error budget above, with the inverse
// transform doubling the FFT term); every decision leaves a full slack.
// grouped != 0: the window is not this series' business (its group's representative is decided by
// the scores alone, muse_batch.go:87-89): upper and lower bound on the score itself.
__device__ __forceinline__ float refine_decide(float U, float s_in, float s_out, float &L, int grouped) {
    if (!(s_in == s_in) || !(s_out == s_out)) return U;
    const float u32 = fminf(fmaxf(s_in, s_out) * 1.00001f, 1.f) + MUSE_SCREEN_SLACK;
    if (grouped) {
        L = fmaxf(fminf(fmaxf(s_in, s_out) * 0.99999f, 1.f) - MUSE_SCREEN_SLACK, 0.f);
        return fminf(U, u32);
    }
    if (s_out * 0.99999f - MUSE_SCREEN_SLACK > s_in * 1.00001f + MUSE_SCREEN_SLACK) return -1.f;
    if (s_in * 0.99999f - MUSE_SCREEN_SLACK > s_out * 1.00001f + MUSE_SCREEN_SLACK)
        L = fminf(s_in * 0.99999f, 1.f) - MUSE_SCREEN_SLACK;      // certainly inside
    return fminf(U, u32);
}

// ---- the register-resident half-length transform of the n <= 2048 kernels, T = 2 .. 32 lanes per series ----
// M = 32 T complex points, 32 per lane.  Pass 0 is one radix-32 DFT per lane over the inputs z[t + T r]; pass 1 is
// GS = 32 / T radix-T DFTs per lane.  Output k = t + T m (m = slot) then sits in register screen_reg<T>(m), and its
// mirror M - k in lane (T - t) % T, slot 31 - m (lane 0: its own slot (32 - m) % 32; k = 0 pairs with itself and yields
// the DC and Nyquist terms, k = M/2 is lane 0's slot 16).  Every shuffle below has width T.  At T = 32 this is the
// n = 2048 layout: GS = 1 and screen_reg<32>(m) = Perm<32>::at(m).

// register of slot m after the last pass: butterfly m % GS, its output m / GS
template <int T>
MUSE_HD constexpr int screen_reg(int m) {
    return (m % (32 / T)) * T + Perm<T>::at(m / (32 / T));
}

// Centred samples in fp32 straight from the row buffer: v[r] = row[t + T r] - mean for the NZ rows of T complex slots that
// hold samples, 0 beyond.  last_in: this lane's slot of the last row holds samples (odd N: the slot past them holds the
// row's mean, RowStat; it and the slots beyond the row are read as mu, i.e. as 0).
template <int NZ, int T>
__device__ __forceinline__ void load_centred(cf (&v)[32], const cd *rowc, int t, double mu, bool last_in) {
#pragma unroll
    for (int r = 0; r < 32; r++) {
        if (r < NZ) {
            const cd x = (r == NZ - 1 && !last_in) ? cd{mu, mu} : rowc[t + r * T];
            v[r] = cf{(float)(x.x - mu), (float)(x.y - mu)};
        } else {
            v[r] = cf{0.f, 0.f};
        }
    }
}

// Pass 0 after its radix-32 DFT, which the caller runs (Dft32Lead<NZ> on the zero-padded forward input, Dft<32> on the
// inverse's, ahead of taking a locked exchange buffer): twiddle W_M^(j t) from tw (the pass twiddles), scatter into the
// exchange buffer ex, gather the inputs of pass 1.
template <int T>
__device__ __forceinline__ void screen_pass0(cf (&v)[32], cf *ex, const cf *const &tw, int t) {
    constexpr int LOG2M = 5 + (T >= 2) + (T >= 4) + (T >= 8) + (T >= 16) + (T >= 32);
    using G = Geo<LOG2M, 5>;
#pragma unroll
    for (int j = 0; j < 32; j++) {
        cf val = v[Perm<32>::at(j)];
        if (j > 0) val = cmul(val, tw[(j - 1) * T + t]);
        ex[G::pad(32 * t + j)] = val;
    }
    __syncwarp();
    fft_pass_load<LOG2M, 5, 1, float>(v, ex, t);
}

// pass 1: v[screen_reg<T>(m)] = Z[t + T m]
template <int T>
__device__ __forceinline__ void screen_pass1(cf *v) {
#pragma unroll
    for (int c = 0; c < 32 / T; c++) Dft<T, float>::run(v + c * T);
}

// Z[M - k] for k = t + T m, m < 16 (the layout above)
template <int T>
__device__ __forceinline__ cf mirror_of(const cf (&v)[32], int m, bool lane0, int partner) {
    const cf zp = v[screen_reg<T>(31 - m)];
    const cf zs = v[screen_reg<T>((32 - m) & 31)];
    cf src, zm;
    src.x = lane0 ? zs.x : zp.x;
    src.y = lane0 ? zs.y : zp.y;
    zm.x = __shfl_sync(0xffffffffu, src.x, partner, T);
    zm.y = __shfl_sync(0xffffffffu, src.y, partner, T);
    return zm;
}

// The real split of a mirror pair from e = Z_k + conj(Z_(M-k)), d = Z_k - conj(Z_(M-k)) and the split twiddle
// w = exp(-2 pi i k / n): the squared parts of 2Y_k (qk) and 2conj(Y_(M-k)) (qm), |2Y_k|^2 = qk.x + qk.y.  The caller
// adds them where it takes the square root: that keeps its order of the additions and square roots.
__device__ __forceinline__ void split_sq(cf e, cf d, cf w, cf &qk, cf &qm) {
    const cf wo = cmul(cmul_negi(d), w);
    const cf y1 = cadd(e, wo);                      // 2*Y_k
    const cf y2 = csub(e, wo);                      // 2*conj(Y_(M-k))
    qk = pmul(y1, y1);
    qm = pmul(y2, y2);
}

// This lane's series' sum_k |2Y_k| A[k] (the bound U before 1/std and the slack), summed over its T lanes.  PAIR: the
// pair bound: 2Y_k = e + w o and 2conj(Y_(M-k)) = e - w o with |w| = 1 give |2Y_k|^2 + |2Y_(M-k)|^2 = 2 (|e|^2 + |d|^2),
// d = Z_k - conj(Z_(M-k)) (|d| = |o|), so by Cauchy-Schwarz
//   |2Y_k| A[k] + |2Y_(M-k)| A[M-k] <= sqrt(|e|^2 + |d|^2) * B[k]:
// no twiddle, one square root per pair.  It passes 5.5 % of the benchmark's series on to the second stage where the
// bin-by-bin sum (!PAIR) passed 3.6 %, for a third fewer instructions in this loop on every series.
template <int T, bool PAIR>
__device__ __forceinline__ float screen_bound(const cf (&v)[32], const ScreenParams &prm, int t, bool lane0, int partner) {
    float acc = 0.f;
#pragma unroll
    for (int m = 0; m < 16; m++) {
        const cf zk = v[screen_reg<T>(m)];
        const cf zm = mirror_of<T>(v, m, lane0, partner);
        const cf zmc = cconj(zm);
        const cf e = cadd(zk, zmc);
        if constexpr (PAIR) {
            const cf d = csub(zk, zmc);
            const cf q = pfma(d, d, pmul(e, e));
            acc = fmaf(sqrt_approx(q.x + q.y), prm.sb[t + T * m], acc);
        } else {
            const float4 sv = prm.sw[t + T * m];            // (w_k.x, w_k.y, A[k], A[M-k])
            cf qk, qm;
            split_sq(e, csub(zk, zmc), cf{sv.x, sv.y}, qk, qm);
            acc = fmaf(sqrt_approx(qk.x + qk.y), sv.z, fmaf(sqrt_approx(qm.x + qm.y), sv.w, acc));
        }
    }
    {   // k = M/2: lane 0, slot 16 (weight 0 on the other lanes)
        const cf z = v[screen_reg<T>(16)];
        const cf q = pmul(z, z);
        acc = fmaf(sqrt_approx(q.x + q.y), lane0 ? 2.f * prm.a_mid : 0.f, acc);
    }
    return group_sum_f<T>(acc);
}

__device__ __forceinline__ cf split_twiddle(float4 s) { return cf{s.x, s.y}; }      // (w_k, A[k], A[M-k]) of ScreenParams::sw
__device__ __forceinline__ cf split_twiddle(cf s) { return s; }

// conj(Y)*X on the mirror pairs of the split (pointwise_pair), in place: Z'[k] -> own slot m; Z'[M-k] -> the partner's
// slot 31 - m (lane 0: its own slot 32 - m); k = M/2 pairs with itself (w = -i).  sw: split twiddles, k < M/2 (float4 or
// cf); sx, x_mid: the reference's Xt.  Leaves the swapped values the inverse, swap(FFT(swap(.))), starts from.
template <int T, typename SW>
__device__ __forceinline__ void conj_mul_pairs(cf (&v)[32], const SW *const &sw, const float4 *const &sx, const cf &x_mid, int t, bool lane0,
                                               int partner) {
#pragma unroll
    for (int m = 0; m < 16; m++) {
        const cf zk = v[screen_reg<T>(m)];
        const cf zm = mirror_of<T>(v, m, lane0, partner);
        const cf w = split_twiddle(sw[t + T * m]);
        const float4 x = sx[t + T * m];
        cf ok, om;
        pointwise_pair(zk, zm, w, cf{x.x, x.y}, cf{x.z, x.w}, ok, om);
        cf rcv;
        rcv.x = __shfl_sync(0xffffffffu, om.x, partner, T);
        rcv.y = __shfl_sync(0xffffffffu, om.y, partner, T);
        v[screen_reg<T>(m)] = ok;
        cf &hi = v[screen_reg<T>(31 - m)];
        hi.x = lane0 ? hi.x : rcv.x;
        hi.y = lane0 ? hi.y : rcv.y;
        if (m > 0) {
            cf &own = v[screen_reg<T>(32 - m)];
            own.x = lane0 ? om.x : own.x;
            own.y = lane0 ? om.y : own.y;
        }
    }
    cf &mid = v[screen_reg<T>(16)];
    cf ok, om;
    pointwise_pair(mid, mid, cf{0.f, -1.f}, x_mid, x_mid, ok, om);
    mid.x = lane0 ? ok.x : mid.x;
    mid.y = lane0 ? ok.y : mid.y;
}

// Maxima of |cc'| inside and outside the lag window over the series' T lanes, from the inverse's output in u
// (u[c T + Perm<T>(jj)] = (cc'[2i+1], cc'[2i]), i = t + c T + 32 jj; cc' = std * cc rotated by pad).
template <int T>
__device__ __forceinline__ void window_maxima(const cf (&u)[32], int t, const int &win_lo, const int &win_len, float &m_in, float &m_out) {
    m_in = 0.f;
    m_out = 0.f;
    const int base = 2 * t - win_lo;
#pragma unroll
    for (int c = 0; c < 32 / T; c++) {
#pragma unroll
        for (int jj = 0; jj < T; jj++) {
            const cf r = u[c * T + Perm<T>::at(jj)];
            const int i2 = base + 2 * (c * T + 32 * jj);
            const bool in0 = (i2 & (64 * T - 1)) <= win_len;      // n = 2 M = 64 T
            const bool in1 = ((i2 + 1) & (64 * T - 1)) <= win_len;
            const float a0 = fabsf(r.y), a1 = fabsf(r.x);
            m_in = fmaxf(m_in, in0 ? a0 : 0.f);
            m_out = fmaxf(m_out, in0 ? 0.f : a0);
            m_in = fmaxf(m_in, in1 ? a1 : 0.f);
            m_out = fmaxf(m_out, in1 ? 0.f : a1);
        }
    }
#pragma unroll
    for (int off = T / 2; off > 0; off >>= 1) {
        m_in = fmaxf(m_in, __shfl_xor_sync(0xffffffffu, m_in, off));
        m_out = fmaxf(m_out, __shfl_xor_sync(0xffffffffu, m_out, off));
    }
}

#if defined(__CUDACC__)
// RowStat from the sums s1 = sum (y - pivot), s2 = sum (y - pivot)^2 of a row of N samples.
__device__ __forceinline__ RowStat make_row_stat(double pivot, double s1, double s2, int N) {
    const double mean = pivot + s1 / N;
    const double var = (s2 - s1 * s1 / N) / (N - 1);
    const bool ok = var >= (double)MUSE_SCREEN_VAR_MIN && var <= (double)MUSE_SCREEN_VAR_MAX &&
                    mean * mean <= MUSE_SCREEN_OFFSET_MAX * MUSE_SCREEN_OFFSET_MAX * var;      // false for NaN / Inf
    RowStat r;
    r.mean = mean;
    r.rstd = ok ? (float)(1.0 / sqrt(var)) : __int_as_float(0x7fc00000);
    r.pad = 0u;
    return r;
}

// The sums of one row for its RowStat, taken by one warp: about the row's first sample (the pivot), lane l adding samples
// l, l + 32, l + 64, ... in that order, then reduced with xor shuffles.  row_stats_kernel and roll_rows_kernel
// (kernels_roll.cu) both go through this, so a rolled row's RowStat is bit-identical to the one the same row gets at ingest.
struct RowSums {
    double s1 = 0.0, s2 = 0.0;
    __device__ __forceinline__ void add(double v, double pivot) {
        const double x = v - pivot;
        s1 += x;
        s2 = fma(x, x, s2);
    }
    // every lane of the warp calls this; every lane gets the row's RowStat
    __device__ __forceinline__ RowStat warp_stat(double pivot, int N) {
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            s1 += __shfl_xor_sync(0xffffffffu, s1, off);
            s2 += __shfl_xor_sync(0xffffffffu, s2, off);
        }
        return make_row_stat(pivot, s1, s2, N);
    }
};
#endif

// RowStat of rows first .. first+count-1; for an odd series length the row's mean is also written into the first pad
// column of the row (ld >= N + 1 then), so that the screening kernels, which read rows as pairs of samples, see a
// centred value of exactly 0 there whatever the ingest left in it.  One warp per row; sums are taken about the row's first sample so
// that the one-pass variance does not cancel (|row[0] - mean| <= sqrt(N-1) * std, so the cancellation costs at
// most a factor N of the 1e-16).
static __global__ void row_stats_kernel(double *__restrict__ slab, int64_t ld, int N, int64_t first, int64_t count,
                                 RowStat *__restrict__ stat) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarp = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t i = warp0; i < count; i += nwarp) {
        const double *row = slab + (first + i) * ld;
        const double pivot = row[0];
        RowSums rs;
        for (int k = lane; k < N; k += 32) rs.add(row[k], pivot);
        const RowStat r = rs.warp_stat(pivot, N);
        if (lane == 0) {
            stat[first + i] = r;
            if (N & 1) slab[(first + i) * ld + N] = r.mean;
        }
    }
}

struct ScreenWarpCfg {
    using G = Geo<10, 5>;                       // M = 1024 = 32 x 32: one warp per series
    static constexpr int MAX_WARPS = 12;        // 3 warps per scheduler at up to 168 registers per thread (16 at 128 measured equal)
    static constexpr int NREF = 2;              // exchange buffers for the (rare) second stage, shared under a lock
    static constexpr int CLAIM = 2;             // consecutive series per claim from the hand-out counter (a power of two)
    static constexpr size_t SMEM_BUDGET = 227 * 1024;
    static constexpr size_t EX_BYTES = ((size_t)(G::MP + 1) * sizeof(cf) + 127) / 128 * 128;   // padded FFT exchange buffer
    static size_t row_bytes(int N) { const size_t r = ((size_t)N * 8 + 127) / 128 * 128; return r > EX_BYTES ? r : EX_BYTES; }
    static size_t warp_bytes(int N) { return row_bytes(N); }
    static int warps(int N) {
        const size_t w = (SMEM_BUDGET - NREF * EX_BYTES) / warp_bytes(N);
        return (int)(w > MAX_WARPS ? MAX_WARPS : w);
    }
    static size_t smem_bytes(int N) { return (size_t)warps(N) * warp_bytes(N) + NREF * EX_BYTES; }
    static int nz(int N) { return ((N + 1) / 2 + 31) / 32; }
};

__device__ __forceinline__ int ex_acquire(unsigned *locks, int t, int hint) {
    int slot = hint & (ScreenWarpCfg::NREF - 1);
    while (true) {
        unsigned old = 1u;
        if (t == 0) old = atomicCAS(&locks[slot], 0u, 1u);
        if (__shfl_sync(0xffffffffu, old, 0) == 0u) break;
        slot = (slot + 1) & (ScreenWarpCfg::NREF - 1);
    }
    return slot;
}
__device__ __forceinline__ void ex_release(unsigned *locks, int t, int slot) {
    __syncwarp();
    if (t == 0) {
        __threadfence_block();
        atomicExch(&locks[slot], 0u);
    }
}

// Persistent kernel, one block per SM, every warp an independent pipeline over its own series:
// its row buffer is refilled by the next cp.async.bulk as soon as the 23 x 16 bytes per lane
// are in registers, so the DRAM latency of row i+1 hides behind the FFT of row i and ~10 rows
// per SM are in flight at any time.  The FFT exchange goes through a separate per-warp buffer.
//
// Work hand-out: a warp takes CLAIM consecutive series at a time.  Claim r < W (the warps of the
// grid) is warp r's own; later claims come from a device counter (prm.next_claim, cleared with the
// cut-off state), claim W + c to the warp whose increment of it returned c.  A fixed stride of W series
// aliases with any store whose rows repeat with a period dividing W (W = 1776 on 148 SMs; the
// benchmark's rows repeat rect, line, noise, and only rect rows take the second stage): some warps
// got every expensive row and the rest of the SM idled behind them.  The claim is issued at the
// top of the last iteration of a claim and consumed at the re-arm, behind the first FFT pass, so
// its L2 round trip stays off the critical path; the index then waits in shared memory (next_of),
// not in a register across the rest of the FFT.
//
// NZ = ceil(N/64) (17..32 for n = 2048) is a template parameter so that the loads, the
// conversions and the first radix-4 stage of the zero rows disappear at compile time.  The
// |Y_f| bound is invariant under rotation of the padded series, so the zeros trail.
//
// Split: lane t holds Z[t + 32j] in slot j (the transform's layout at T = 32).  Bins k and M-k share
// e = Z[k] + conj(Z[M-k]) and w*o, 2Y[k] = e + w*o, 2conj(Y[M-k]) = e - w*o, so each lane walks only
// j < 16 (k < 512) and gets both magnitudes from one mirror exchange.  Only k = 512 (lane 0, slot 16,
// its own mirror) is left over: |2Y[512]| = 2|Z[512]|.
//
// Fused second stage: U is loose (it ignores every phase), and on the benchmark's data
// a few percent of the series have U above the top-N cut-off.  A warp whose U reaches the
// RUNNING cut-off therefore goes on, with the spectrum still in registers: conj(Y)*X in fp32,
// inverse FFT, max |cc| inside and outside the lag window.  That replaces U by the much
// tighter u32 = |cc|_max/std + slack (or by -1 when the peak is certainly outside the window:
// the series fails results.go:46-48), and yields a certain LOWER bound for series that certainly
// pass the filter.  Lower bounds are counted in a global histogram; the top_n-th largest so far
// is a valid lower bound on the final cut-off and becomes the new running cut-off (it only ever
// rises, so a stale read is merely less sharp).  Afterwards only series with out_U >= final cut
// -- a few hundred -- need the exact fp64 kernel.  The cc index is rotated by pad = n - N against
// xcorr.go's (zeros trail here, lead there): true index = (idx - pad) mod n.
template <int NZ>
__global__ void __launch_bounds__(ScreenWarpCfg::MAX_WARPS * 32, 1)
score_screen_warp_kernel(const ScreenParams prm, const unsigned warp_bytes, const unsigned row_bytes) {
    using C = ScreenWarpCfg;
    constexpr int P = 32;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ __align__(8) unsigned long long bars[C::MAX_WARPS];
    __shared__ unsigned ex_locks[C::NREF];
    __shared__ int next_of[C::MAX_WARPS];      // the warp's next series: written at the re-arm, read at the end of the iteration

    const int w = threadIdx.x >> 5;
    const int t = threadIdx.x & 31;
    // 32-bit series indices (a store holds < 2^31 series): the kernel sits on a register cliff at 168
    const int count = (int)prm.count;
    const int grid_warps = (int)(gridDim.x * (blockDim.x >> 5));
    const int pos0 = ((int)(blockIdx.x * (blockDim.x >> 5)) + w) * C::CLAIM;
    unsigned char *buf = smem_raw + (size_t)w * warp_bytes;
    const cd *rowc = reinterpret_cast<const cd *>(buf);
    cf *sm = reinterpret_cast<cf *>(buf);                       // forward exchange: the row buffer itself
    unsigned char *refbase = smem_raw + (size_t)(blockDim.x >> 5) * warp_bytes;
    const int N = prm.N;
    const int Nh = (N + 1) >> 1;      // complex slots holding samples (odd N: the pad column of the last one holds the row's mean, RowStat)
    const unsigned bar = smem_u32(&bars[w]);
    const int partner = (P - t) & (P - 1);
    const bool lane0 = (t == 0);
    const bool last_in = t + (NZ - 1) * 32 < Nh;      // is this lane's slot of the last row a sample?

    if (threadIdx.x < C::NREF) ex_locks[threadIdx.x] = 0u;
    if (t == 0) {
        mbar_init(bar, 1);
        mbar_init_fence();
        if (pos0 < count) bulk_load(smem_u32(buf), prm.slab + (int64_t)pos0 * prm.ld, (unsigned)(N + (N & 1)) * 8u, bar);
    }
    __syncthreads();

    // mbarrier phase parity = iteration parity; it rides in bit 31 of the loop counter (count < 2^31):
    // a separate loop-carried register is one too many for the allocator at 168 and gets spilled
    unsigned pp = (unsigned)pos0;
    while ((int)(pp & 0x7fffffffu) < count) {
        const int pos = (int)(pp & 0x7fffffffu);
        const unsigned phase = pp >> 31;
        const bool claim_ends = (pos & (C::CLAIM - 1)) == C::CLAIM - 1;
        // running cut-off: one lane reads it (so that the whole warp takes the same branch below) at
        // the top of the iteration; the value is consumed only after U is known, a thousand
        // instructions later, so the L2 round trip stays off the critical path.  +inf = no refinement
        unsigned cut_raw = 0u, claim = 0u;
        if (t == 0) {
            cut_raw = ld_relaxed_u32(prm.cut_bits);
            // consumed at the re-arm.  An increment, not atomicAdd(.., 1): ptxas turns that (and atomicInc with a constant
            // limit) into a warp-aggregated atomic whose shuffle of the result waits for the L2 round trip right here.  The
            // limit never wraps the counter: a claim is made only after a series < count that ends a claim, at most
            // count / CLAIM times.
            if (claim_ends) claim = atomicInc(prm.next_claim, (unsigned)count);
        }
        const RowStat rs = prm.row_stat[pos];   // fp64 mean and 1/std from the ingest pass (xcorr.go:84-95); in flight with the row
        const double mu = rs.mean;
        mbar_wait(bar, phase);      // every lane waits itself (one polling lane + __syncwarp measured 3x slower)

        cf v[P];
        load_centred<NZ, 32>(v, rowc, t, mu, last_in);
        __syncwarp();                       // the row is consumed: the buffer becomes the exchange buffer

        // ---- forward FFT_1024: pruned radix-32, twiddle, exchange through smem, radix-32 ----
        Dft32Lead<NZ, float>::run(v);
        screen_pass0<32>(v, sm, prm.twp, t);
        __syncwarp();
        if (t == 0) {                       // the exchange is over: hand the buffer to the copy engine for the next row
            // next < grid_warps * CLAIM + count < 2^31: the counter stays below count / CLAIM
            const int next = claim_ends ? (grid_warps + (int)claim) * C::CLAIM : pos + 1;
            next_of[w] = next;
            if (next < count) {
                asm volatile("" ::"r"(__float_as_uint(v[P - 1].y)) : "memory");
                // the generic-proxy reads and writes of the exchange are ordered before the async-proxy write of the copy
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                bulk_load(smem_u32(buf), prm.slab + (int64_t)next * prm.ld, (unsigned)(N + (N & 1)) * 8u, bar);
            }
        }
        screen_pass1<32>(v);                            // v[Perm(j)] = Z[t + 32*j]
        const float acc = screen_bound<32, true>(v, prm, t, lane0, partner);

        // rstd is NaN for a row no fp32 statement may be made about (RowStat); NaN/Inf samples make acc NaN:
        // either way the bound is NaN and the exact kernel decides
        float U = acc * rs.rstd * 1.00001f + MUSE_SCREEN_SLACK;
        if (!(U == U)) U = 2.f;
        float L = -1.f;
        // The broadcast must not be scheduled before this point: it would wait for the load
        // issued at the top of the iteration (measured: +8 % kernel time).  Its source lane
        // therefore depends on acc, which exists only now; it is 0 unless acc has one particular
        // NaN pattern, and then lane 1's zeros merely send the series through the refinement.
        const int bsrc = (__float_as_uint(acc) == 0x7fc12345u) ? 1 : 0;
        const float cut_now = __uint_as_float(__shfl_sync(0xffffffffu, cut_raw, bsrc));
        if (U >= cut_now && U < 1.5f) {      // warp-uniform: U comes out of a butterfly reduction
            // ---- conj(Y)*X: conj_mul_pairs<32>, written out because with it ptxas swaps the registers of the last row's
            //      two copies of mu at NZ = 24, 28 and 32 ----
#pragma unroll
            for (int j = 0; j < P / 2; j++) {
                const cf zk = v[Perm<P>::at(j)];
                const cf zm = mirror_of<32>(v, j, lane0, partner);
                const float4 s = prm.sw[t + 32 * j];
                const float4 x = prm.sx[t + 32 * j];
                cf ok, om;
                pointwise_pair(zk, zm, cf{s.x, s.y}, cf{x.x, x.y}, cf{x.z, x.w}, ok, om);
                cf rcv;
                rcv.x = __shfl_sync(0xffffffffu, om.x, partner);
                rcv.y = __shfl_sync(0xffffffffu, om.y, partner);
                v[Perm<P>::at(j)] = ok;
                cf &hi = v[Perm<P>::at(P - 1 - j)];
                hi.x = lane0 ? hi.x : rcv.x;
                hi.y = lane0 ? hi.y : rcv.y;
                if (j > 0) {
                    cf &own = v[Perm<P>::at(P - j)];
                    own.x = lane0 ? om.x : own.x;
                    own.y = lane0 ? om.y : own.y;
                }
            }
            {   // k = 512 pairs with itself (lane 0, slot 16); w_512 = -i
                cf &mid = v[Perm<P>::at(P / 2)];
                cf ok, om;
                pointwise_pair(mid, mid, cf{0.f, -1.f}, prm.x_mid, prm.x_mid, ok, om);
                mid.x = lane0 ? ok.x : mid.x;
                mid.y = lane0 ? ok.y : mid.y;
            }
            // ---- inverse FFT_1024 as swap(FFT(swap(.))) (pointwise_pair stores the swapped values) ----
            cf u[P];
#pragma unroll
            for (int j = 0; j < P; j++) u[j] = v[Perm<P>::at(j)];
            Dft<P, float>::run(u);
            {
                const int slot = ex_acquire(ex_locks, t, w);
                screen_pass0<32>(u, reinterpret_cast<cf *>(refbase + (size_t)slot * C::EX_BYTES), prm.twp, t);
                ex_release(ex_locks, t, slot);
            }
            screen_pass1<32>(u);        // u[Perm(j)] = (cc'[2i+1], cc'[2i]), i = t + 32*j; cc' = std * cc rotated by pad
            float m_in, m_out;
            window_maxima<32>(u, t, prm.win_lo, prm.win_len, m_in, m_out);
            const float rstd = rs.rstd;
            const float s_in = m_in * rstd, s_out = m_out * rstd;
            U = refine_decide(U, s_in, s_out, L, prm.grouped);
            if (t == 0) atomicAdd(prm.n_refined, 1ull);
            // ---- a certain pass at or above the running cut-off: count it and try to raise the cut-off ----
            if (L >= prm.thr && L >= cut_now) cut_count_and_raise(prm.cut_bits, prm.cut_hist, prm.top_n, L, t);
        }
        if (t == 0) {
            prm.out_U[pos] = U;
            if (prm.out_L) prm.out_L[pos] = L;
        }
        __syncwarp();                       // next_of[w] of lane 0's re-arm
        pp = (unsigned)next_of[w] | (~pp & 0x80000000u);
    }
}

#endif  // __CUDACC__

}  // namespace muse
