// muse_select.cuh -- everything downstream of the per-series scores: group keys,
// group max BEFORE the filter (muse_batch.go:87-89), the Results filter
// (results.go:46-52) and the top-N selection (results.go:55-87), on the device.
//
// Ordering rules (the reference is nondeterministic on ties because Go map iteration
// is random, SURVEY F4; we fix one admissible order):
//   group representative: highest |score|, ties -> lowest series index
//   top-N:                highest |score|, ties -> lowest series index
// NaN scores never pass results.go:46-52 and are left out of the group max.
#pragma once

#include <stdint.h>
#include <string.h>

#include <type_traits>

#if defined(__CUDACC__)
#include <cuda_runtime.h>
#include "muse_screen.cuh"

namespace muse {

__device__ __forceinline__ unsigned long long score_bits(double s) {
    // |s| as ordered bits: non-negative doubles order like their uint64 patterns
    return (unsigned long long)__double_as_longlong(fabs(s));
}

// Canonical group key of series i from its label ids: (id+1) packed in 64/ncols bits per
// column (id < 0 -> 0: "label absent", all such series share a group as labels.go:61-65
// skips absent keys).  Rank independent, so shards can be merged on it.
#define MUSE_MAX_KEY_COLS 16
struct KeyCols {
    const int32_t *col[MUSE_MAX_KEY_COLS];
    int ncols;
    int bits[MUSE_MAX_KEY_COLS];   // key bits of each column: 64 / ncols each when every cardinality fits (rank independent),
                                   // else ceil(log2(cardinality)) per column of THIS store (sum <= 64)
};

__device__ __forceinline__ unsigned long long canonical_key(const KeyCols &kc, int64_t i) {
    unsigned long long key = 0;
    for (int c = 0; c < kc.ncols; c++) {
        const unsigned long long v = (unsigned long long)(kc.col[c][i] + 1);
        key = (kc.bits[c] >= 64) ? v : ((key << kc.bits[c]) | v);
    }
    return key;
}

// slot of a key in the group table: dense (mixed radix over the per-column cardinalities)
// or an open-addressing hash table keyed by the canonical key.
struct GroupTable {
    unsigned long long *gmax;   // [slots] best |score| bits
    int32_t *gidx;              // [slots] representative (local series index)
    unsigned long long *hkeys;  // [slots] hash mode: canonical key + 1 (0 = empty)
    int64_t slots;              // power of two in hash mode
    int dense;                  // 1: dense index
    int64_t radix[MUSE_MAX_KEY_COLS];   // dense: cardinality (max id + 2) per column
};

// slot of `key` (!= 0) in an open-addressing table of `slots` (a power of two) keys, 0 = empty: the slot that holds it,
// or the empty slot it claims
__device__ __forceinline__ long long hash_slot(unsigned long long *hkeys, long long slots, unsigned long long key) {
    unsigned long long h = key * 0x9E3779B97F4A7C15ull;
    h ^= h >> 32;
    long long s = (long long)(h & (unsigned long long)(slots - 1));
    for (;;) {
        const unsigned long long cur = hkeys[s];
        if (cur == key) return s;
        if (cur == 0ull) {
            const unsigned long long old = atomicCAS(&hkeys[s], 0ull, key);
            if (old == 0ull || old == key) return s;
        }
        s = (s + 1) & (slots - 1);
    }
}

__device__ __forceinline__ int64_t table_slot(const GroupTable &gt, const KeyCols &kc, int64_t i) {
    if (gt.dense) {
        int64_t s = 0;
        for (int c = 0; c < kc.ncols; c++) s = s * gt.radix[c] + (int64_t)(kc.col[c][i] + 1);
        return s;
    }
    return hash_slot(gt.hkeys, gt.slots, canonical_key(kc, i) + 1ull);
}

// Warp-aggregated append: every lane whose `take` is set gets its own position in a list whose length is *n, with one
// atomic per warp, and calls store(position).  All 32 lanes of the warp call it.
template <typename Store>
__device__ __forceinline__ void warp_append(unsigned long long *n, bool take, Store store) {
    const unsigned mask = __ballot_sync(0xffffffffu, take);
    if (mask == 0u) return;
    const int lane = threadIdx.x & 31, leader = __ffs(mask) - 1;
    unsigned long long base = 0;
    if (lane == leader) base = atomicAdd(n, (unsigned long long)__popc(mask));
    base = __shfl_sync(0xffffffffu, base, leader);
    if (take) store(base + (unsigned long long)__popc(mask & ((1u << lane) - 1u)));
}

// pass 1: slot per series + atomicMax of |score| bits
__global__ void group_max_kernel(GroupTable gt, KeyCols kc, const double *__restrict__ score, int64_t S,
                                 int64_t *__restrict__ slot_of) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= S) return;
    const int64_t s = table_slot(gt, kc, i);
    slot_of[i] = s;
    const double sc = score[i];
    if (sc == sc) atomicMax(&gt.gmax[s], score_bits(sc));
}

// slot of every series in the group table (hash mode: inserts the key)
__global__ void group_slots_kernel(GroupTable gt, KeyCols kc, int64_t S, int64_t *__restrict__ slot_of) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < S) slot_of[i] = table_slot(gt, kc, i);
}

// Grouped screening: slot per series + atomicMax of the fp32 LOWER bounds of the members' scores
// (float bits in the low word of gmax; non-negative floats order like their bit patterns).
__global__ void group_lower_bound_kernel(GroupTable gt, KeyCols kc, const float *__restrict__ lower, int64_t S,
                                         int64_t *__restrict__ slot_of) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= S) return;
    const int64_t s = table_slot(gt, kc, i);
    slot_of[i] = s;
    const float lo = lower[i];
    if (lo >= 0.f) atomicMax(&gt.gmax[s], (unsigned long long)__float_as_uint(lo));
}

// ... and the members that can still be their group's representative: upper bound >= the group's
// best lower bound (the true representative always qualifies, and so does every member that ties it)
// A member whose upper bound is below thr_lo (<= the threshold) cannot be the representative of a group that passes
// results.go:46-52 -- if it were, the whole group would fail -- so it is left out as well.
// cut_bits (may be NULL): float bits of a lower bound on the top_n-th best group that certainly passes the filter
// (group_cut_find_kernel): a member below it cannot be the representative of a group of the top-N.
__global__ void group_contenders_kernel(GroupTable gt, const float *__restrict__ upper, int64_t S,
                                        const int64_t *__restrict__ slot_of, float thr_lo, int32_t *__restrict__ out,
                                        unsigned long long *n, const unsigned *__restrict__ cut_bits) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (cut_bits) thr_lo = fmaxf(thr_lo, __uint_as_float(*cut_bits));
    bool take = false;
    if (i < S) {
        const unsigned long long g = gt.gmax[slot_of[i]];
        take = upper[i] >= thr_lo && upper[i] >= __uint_as_float((unsigned)g);
        // every possible representative of the group has its peak certainly outside the lag window: the group fails
        // results.go:46-48 whatever the exact scores are (flags of group_uncertain_kernel; only set in that mode)
        if (cut_bits && !((g >> 33) & 1ull)) take = false;
    }
    warp_append(n, take, [&](unsigned long long pos) { out[pos] = (int32_t)i; });
}

// ---- a cut-off for grouped single-GPU runs -----------------------------------------------------------------------
// After the screening pass a group's running lower bound L_g (low word of gmax) bounds its score from below (muse_batch.go:87-89:
// the group's score is its best member's).  The group certainly PASSES results.go:46-52 when L_g reaches the threshold and
// every member that can still be its representative (upper bound >= L_g) has its peak certainly inside the lag window
// (out_W == 1).  The top_n-th largest L_g among those groups is a lower bound on the score of the last group Results will
// keep, so members below it need no exact score: a group whose true best member lies below it is ranked behind top_n
// groups that are scored exactly, whatever score its other members give it.  (Not for shard partials: a group's
// representative may sit in another shard.)
// 1. flag the groups with a possible representative that is not certainly inside the window (bit 32 of gmax) / not certainly
//    outside it (bit 33: a group without it certainly fails the filter and needs no exact score either)
__global__ void group_uncertain_kernel(GroupTable gt, const float *__restrict__ upper, const signed char *__restrict__ W, int64_t S,
                                       const int64_t *__restrict__ slot_of) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= S) return;
    const int64_t s = slot_of[i];
    const float Lg = __uint_as_float((unsigned)gt.gmax[s]);
    if (!(upper[i] < Lg)) {                                  // NaN / undecided bounds count as possible
        const unsigned long long f = (W[i] != 1 ? 1ull << 32 : 0ull) | (W[i] != -1 ? 1ull << 33 : 0ull);
        atomicOr(&gt.gmax[s], f);
    }
}
// 2. count the certain groups' lower bounds in the three-level histogram of the running cut-off (muse_screen.cuh)
__global__ void group_cut_count_kernel(GroupTable gt, double threshold, unsigned *hist) {
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= gt.slots) return;
    const unsigned long long g = gt.gmax[s];
    if ((g >> 32) & 1ull) return;
    const float L = __uint_as_float((unsigned)g);
    if (!(L > 0.f) || (double)L < threshold) return;
    cut_hist_add(hist, L);
}
// 3. one warp: the lower edge of the bin that holds the top_n-th largest counted bound (nothing when fewer were counted)
__global__ void group_cut_find_kernel(const unsigned *hist, int top_n, unsigned *cut_bits) {
    cut_walk(cut_bits, hist, top_n, threadIdx.x);
}

// pass 2: lowest series index among the members that hold the group max
__global__ void group_rep_kernel(GroupTable gt, const double *__restrict__ score, int64_t S,
                                 const int64_t *__restrict__ slot_of) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= S) return;
    const double sc = score[i];
    if (sc != sc) return;
    const int64_t s = slot_of[i];
    if (score_bits(sc) == gt.gmax[s]) atomicMin(&gt.gidx[s], (int32_t)i);
}

struct FilterArgs {
    int64_t max_lag;
    double threshold;
    int sign_filter;
    int apply;   // 0: emit every representative unfiltered (multi-GPU grouped partials)
};

MUSE_HD bool passed(const FilterArgs &f, double sc, int lag) {
    // results.go:46-52
    const int64_t al = lag < 0 ? -(int64_t)lag : (int64_t)lag;
    return al <= f.max_lag && fabs(sc) >= f.threshold &&
           (f.sign_filter == 0 || (sc > 0.0 && f.sign_filter == 1) || (sc < 0.0 && f.sign_filter == -1));
}

// The counters of a run (d_counters, and one set per query of a multi-query launch).
struct RunCounters {
    unsigned long long cand;       // candidates (Cand::n)
    unsigned long long selected;   // candidates the radix select gathered
    unsigned long long listed;     // length of the exact list (fused runs) / series re-scored in the pilot round
    unsigned long long refined;    // series that took the fused second stage / re-scored in the second round
};

// Candidate = a group representative that passed the filter.
struct Cand {
    unsigned long long *key;   // |score| bits
    int32_t *idx;              // local series index
    int32_t *lagsgn;           // 2*lag + (score < 0)
    unsigned long long *n;     // counter
};

// score and lag of a candidate from its |score| bits and 2*lag + (score < 0)
MUSE_HD double cand_score(unsigned long long key, int lagsgn) {
    double a;
    memcpy(&a, &key, sizeof(a));
    return (lagsgn & 1) ? -a : a;
}
MUSE_HD int cand_lag(int lagsgn) { return (lagsgn - (lagsgn & 1)) / 2; }

// candidate a precedes candidate b in (|score| desc, index asc) -- on |score| bits, which order like the non-negative scores
template <typename Idx>
MUSE_HD bool key_precedes(unsigned long long ka, Idx ia, unsigned long long kb, Idx ib) {
    return ka > kb || (ka == kb && ia < ib);
}

__device__ __forceinline__ void emit_candidate(const Cand &out, bool emit, double sc, int32_t idx, const int32_t *__restrict__ lag) {
    warp_append(out.n, emit, [&](unsigned long long pos) {
        out.key[pos] = score_bits(sc);
        out.idx[pos] = idx;
        out.lagsgn[pos] = 2 * lag[idx] + (sc < 0.0 ? 1 : 0);
    });
}

// Emit candidates.  slot_of == NULL: ungrouped (every series is its own representative).
__global__ void emit_candidates_kernel(GroupTable gt, const int64_t *__restrict__ slot_of,
                                       const double *__restrict__ score, const int32_t *__restrict__ lag,
                                       int64_t S, FilterArgs f, Cand out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool emit = false;
    double sc = 0.0;
    if (i < S) {
        sc = score[i];
        emit = (sc == sc);
        if (emit && slot_of) emit = (gt.gidx[slot_of[i]] == (int32_t)i);
        if (emit && f.apply) emit = passed(f, sc, lag[i]);
    }
    emit_candidate(out, emit, sc, (int32_t)i, lag);
}

// Emit candidates from a LIST of series (the fused path's exact list): entry i < min(*n_list, limit) is a
// series with an exact score; the ones that pass results.go:46-52 are appended like emit_candidates_kernel does.
__device__ __forceinline__ void emit_listed_body(const int32_t *__restrict__ list, const unsigned long long *__restrict__ n_list,
                                                 long long limit, const double *__restrict__ score, const int32_t *__restrict__ lag,
                                                 const FilterArgs &f, const Cand &out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned long long n = *n_list;
    bool emit = false;
    double sc = 0.0;
    int32_t idx = 0;
    if (i < limit && (unsigned long long)i < n) {
        idx = list[i];
        sc = score[idx];
        emit = (sc == sc) && (!f.apply || passed(f, sc, lag[idx]));
    }
    emit_candidate(out, emit, sc, idx, lag);
}

__global__ void emit_listed_kernel(const int32_t *__restrict__ list, const unsigned long long *__restrict__ n_list,
                                   long long limit, const double *__restrict__ score, const int32_t *__restrict__ lag,
                                   FilterArgs f, Cand out) {
    emit_listed_body(list, n_list, limit, score, lag, f, out);
}

// Per-query pointers of the batched tails of muse_multi_run (one launch per stage, blockIdx.y = query).
struct MultiTail {
    const float *U;                 // [S] the query's bounds after the second stages
    const CutState *cut;            // the query's cut-off state
    int32_t *list;                  // series whose bound reaches the cut-off
    RunCounters *counters;
    double *score;                  // [S] exact scores of the listed series
    int32_t *lag;
    unsigned long long *ckey;       // candidates
    int32_t *cidx, *clag;
    void *out;                      // PartialRec[top_n]: the query's result records
};

__global__ void emit_listed_batch_kernel(const MultiTail *__restrict__ tails, long long limit, FilterArgs f) {
    const MultiTail t = tails[blockIdx.y];
    emit_listed_body(t.list, &t.counters->listed, limit, t.score, t.lag, f, Cand{t.ckey, t.cidx, t.clag, &t.counters->cand});
}

// ---- device-side top-N of a short candidate list, written as muse_partial records ------
// Rank by counting: candidate i's position in the (|score| desc, index asc) order is the number of
// candidates that come before it; those with a position < top_n write their own muse_partial
// record to that slot.  n^2 comparisons spread over the whole GPU (n ~ 4.5 k at C3: ~10 us; a
// one-block bitonic sort of the same list took 180 us).  Slots min(n, top_n) .. capacity-1 are
// padded with flags = 1 (ignored by the merge).  A multi-GPU step can then all-gather the records
// straight from device memory: no host round trip between the scores and the collective.
// flags = 2 in record 0 tells the caller that the list was too long for this kernel (or that the
// fused path's exact launch did not cover its list): it then takes the host path.
#define MUSE_PARTIAL_RANK_CAP 32768
struct PartialRec {           // == muse_partial (include/muse_b200.h)
    unsigned long long group_key;
    double score;
    long long series_idx;
    int lag;
    int flags;
};

// Position of candidate (k, ix) in the (|score| desc, index asc) order: the number of the n candidates that come before it,
// counted by the calling warp.  Its lanes stride over the list, four independent loads in flight per lane (the list is 48 KB
// at C3: L1/L2 resident, but one dependent load per step made this kernel 31 us).
template <typename Idx>
__device__ __forceinline__ unsigned rank_of(const unsigned long long *__restrict__ ckey, const Idx *__restrict__ cidx, unsigned long long n,
                                            unsigned long long k, typename std::make_unsigned<Idx>::type ix, int lane) {
    using U = decltype(ix);      // indices compare unsigned: they are >= 0
    unsigned before = 0;
    unsigned long long j = lane;
    for (; j + 96 < n; j += 128) {
        const unsigned long long k0 = ckey[j], k1 = ckey[j + 32], k2 = ckey[j + 64], k3 = ckey[j + 96];
        const U i0 = (U)cidx[j], i1 = (U)cidx[j + 32], i2 = (U)cidx[j + 64], i3 = (U)cidx[j + 96];
        before += key_precedes(k0, i0, k, ix) ? 1u : 0u;
        before += key_precedes(k1, i1, k, ix) ? 1u : 0u;
        before += key_precedes(k2, i2, k, ix) ? 1u : 0u;
        before += key_precedes(k3, i3, k, ix) ? 1u : 0u;
    }
    for (; j < n; j += 32) {
        const unsigned long long kj = ckey[j];
        before += (kj > k || (kj == k && (U)cidx[j] < ix)) ? 1u : 0u;      // the index is loaded only on a tie
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) before += __shfl_xor_sync(0xffffffffu, before, off);
    return before;
}

// The top_n of the n candidates (ckey, cidx, clag) by rank, as records in slots 0 .. top_n - 1 and padding up to `capacity`
// (record 0 flagged 2 instead when `overflow`).  Candidate indices are global_offset + cidx; the series index is the
// group key of an ungrouped run.  store(d, slot, rec) writes a record to destination d < ndest: the padding by every
// thread to all destinations, a ranked record by the lanes of its warp, one destination each.
template <typename Idx, typename Store>
__device__ __forceinline__ void rank_topn(const unsigned long long *__restrict__ ckey, const Idx *__restrict__ cidx,
                                          const int32_t *__restrict__ clag, unsigned long long n, bool overflow, long long top_n,
                                          long long global_offset, long long capacity, int ndest, Store store) {
    const long long gtid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long take = overflow ? 0 : ((long long)n < top_n ? (long long)n : top_n);
    for (long long r = take + gtid; r < capacity; r += (long long)gridDim.x * blockDim.x) {
        const PartialRec pad{0ull, 0.0, 0ll, 0, (overflow && r == 0) ? 2 : 1};
        for (int d = 0; d < ndest; d++) store(d, r, pad);
    }
    if (overflow) return;
    // one warp per candidate
    const int lane = threadIdx.x & 31;
    const unsigned long long nwarps = ((unsigned long long)gridDim.x * blockDim.x) >> 5;
    for (unsigned long long i = (unsigned long long)gtid >> 5; i < n; i += nwarps) {
        const unsigned long long k = ckey[i];
        const Idx ix = cidx[i];
        const unsigned before = rank_of(ckey, cidx, n, k, ix, lane);
        if ((long long)before < top_n) {
            const int ls = clag[i];
            const long long gi = global_offset + (long long)ix;
            const PartialRec rec{(unsigned long long)gi, cand_score(k, ls), gi, cand_lag(ls), 0};
            for (int d = lane; d < ndest; d += 32) store(d, (long long)before, rec);
        }
    }
}

// the list is too long for rank_topn, or (exact_list_bound >= 0) the fused path's exact launch did not cover its list
__device__ __forceinline__ bool topn_overflow(const RunCounters &c, long long exact_list_bound) {
    return c.cand > MUSE_PARTIAL_RANK_CAP || (exact_list_bound >= 0 && c.listed > (unsigned long long)exact_list_bound);
}

__device__ __forceinline__ void partial_topn_body(const unsigned long long *__restrict__ ckey, const int32_t *__restrict__ cidx,
                                                  const int32_t *__restrict__ clag, const RunCounters *__restrict__ counters, long long top_n,
                                                  long long global_offset, long long exact_list_bound, PartialRec *__restrict__ out, long long capacity) {
    rank_topn(ckey, cidx, clag, counters->cand, topn_overflow(*counters, exact_list_bound), top_n, global_offset, capacity, 1,
              [&](int, long long r, const PartialRec &rec) { out[r] = rec; });
}

__global__ void __launch_bounds__(256)
partial_topn_kernel(const unsigned long long *__restrict__ ckey, const int32_t *__restrict__ cidx,
                    const int32_t *__restrict__ clag, const RunCounters *__restrict__ counters, long long top_n,
                    long long global_offset, long long exact_list_bound, PartialRec *__restrict__ out, long long capacity) {
    partial_topn_body(ckey, cidx, clag, counters, top_n, global_offset, exact_list_bound, out, capacity);
}
__global__ void __launch_bounds__(256)
partial_topn_batch_kernel(const MultiTail *__restrict__ tails, long long top_n, long long global_offset, long long exact_list_bound) {
    const MultiTail t = tails[blockIdx.y];
    partial_topn_body(t.ckey, t.cidx, t.clag, t.counters, top_n, global_offset, exact_list_bound, static_cast<PartialRec *>(t.out), top_n);
}

// ---- the same top-N, pushed straight into every GPU's receive buffer over NVLink peer memory ------
// Multi-GPU exchange fused into the selection: instead of leaving the shard's records in local memory
// for a collective, every record is stored to slot [rank] of the receive buffer of EVERY rank (peer
// pointers from cudaIpcOpenMemHandle; 32-byte stores over NVLink / NVSwitch), the last block of the grid
// fences (system scope) and releases flag[rank] = epoch on every peer.  exchange_wait_kernel then
// acquires all the flags of the local buffer: when it returns, the records of all shards are local.
#define MUSE_EXCHANGE_MAX_RANKS 16
struct ExchangePeers {
    PartialRec *recs[MUSE_EXCHANGE_MAX_RANKS];            // base of rank r's receive records for this parity: [world][capacity]
    unsigned long long *flags[MUSE_EXCHANGE_MAX_RANKS];   // rank r's flags for this parity: [world]
    int world, rank;
    unsigned long long epoch;
    unsigned *done_blocks;                                // local: blocks of this launch that have finished
};

__device__ __forceinline__ void st_release_sys_u64(unsigned long long *p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys_u64(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

// true in the last block of the grid to finish, once everything this GPU stored is ordered (system scope) before the flags
// that block releases
__device__ __forceinline__ bool last_block_fenced(unsigned *done_blocks) {
    __shared__ bool last;
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) last = (atomicAdd(done_blocks, 1u) == gridDim.x - 1);
    __syncthreads();
    if (!last) return false;
    __threadfence_system();
    return true;
}
// by the last block: flag [rank] of every rank = word, and the block counter ready for the next launch
__device__ __forceinline__ void release_flags(const ExchangePeers &ex, unsigned long long word) {
    if (threadIdx.x < ex.world) st_release_sys_u64(&ex.flags[threadIdx.x][ex.rank], word);
    if (threadIdx.x == 0) *ex.done_blocks = 0u;
}

__global__ void __launch_bounds__(256)
partial_topn_push_kernel(const unsigned long long *__restrict__ ckey, const int32_t *__restrict__ cidx,
                         const int32_t *__restrict__ clag, const RunCounters *__restrict__ counters, long long top_n,
                         long long global_offset, long long exact_list_bound, long long capacity, ExchangePeers ex) {
    const bool overflow = topn_overflow(*counters, exact_list_bound);
    const long long slot0 = (long long)ex.rank * capacity;
    rank_topn(ckey, cidx, clag, counters->cand, overflow, top_n, global_offset, capacity, ex.world,
              [&](int d, long long r, const PartialRec &rec) { ex.recs[d][slot0 + r] = rec; });
    if (!last_block_fenced(ex.done_blocks)) return;
    // flag word: (epoch << 32) | records in the slot (the whole slot: it is padded), 0xffffffff = take the host path
    release_flags(ex, (ex.epoch << 32) | (overflow ? 0xffffffffull : (unsigned long long)capacity));
}

// Lane r waits until rank r's flag in the LOCAL buffer has reached `epoch` (bounded spin); status != 0: timed out.
__global__ void exchange_wait_kernel(const unsigned long long *flags, int world, unsigned long long epoch,
                                     long long timeout_cycles, int *status) {
    const int r = threadIdx.x;
    bool ok = true;
    if (r < world) {
        const long long t0 = clock64();
        while ((ld_acquire_sys_u64(&flags[r]) >> 32) < epoch) {
            if (clock64() - t0 > timeout_cycles) {
                ok = false;
                break;
            }
            __nanosleep(200);
        }
    }
    if (!ok) *status = 1;
}

// ---- many references against a sharded store: every shard's per-query top-N lists in ONE exchange step -----------------
// The send table holds q_step lists of top_n records (what muse_multi_run returns for the step's queries on this shard,
// sorted by (|score| desc, global index asc)) followed by the q_step record counts.  Record j of query q goes to
// [q * top_n + j] of slot [rank] of every rank's receive buffer; j >= count[q] is padding (flags = 1).  failed != 0: this
// rank's local run failed after the step began -- it stores no records and releases the failure marker instead, so that its
// peers return in the same step rather than wait for records that never come.
// Low 32 bits of a flag word that mark a failed sender (0xffffffff already means "take the host path").
#define MUSE_EXCHANGE_RANK_FAILED 0xfffffffeull
__global__ void __launch_bounds__(256)
multi_records_push_kernel(const PartialRec *__restrict__ table, const long long *__restrict__ counts, int q_step, long long top_n,
                          long long capacity, int failed, ExchangePeers ex) {
    const long long total = (long long)q_step * top_n;
    const long long slot0 = (long long)ex.rank * capacity;
    if (!failed) {
        for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += (long long)gridDim.x * blockDim.x) {
            const long long q = g / top_n, j = g - q * top_n;
            const PartialRec rec = j < counts[q] ? table[g] : PartialRec{0ull, 0.0, 0ll, 0, 1};
            for (int d = 0; d < ex.world; d++) ex.recs[d][slot0 + g] = rec;
        }
    }
    if (!last_block_fenced(ex.done_blocks)) return;
    release_flags(ex, (ex.epoch << 32) | (failed ? MUSE_EXCHANGE_RANK_FAILED : (unsigned long long)total));
}

// a precedes b in (|score| desc, global series index asc), the order of results.go:81-85 with ties by index
MUSE_HD bool rec_precedes(const PartialRec &a, const PartialRec &b) {
    const double sa = fabs(a.score), sb = fabs(b.score);
    return sa > sb || (sa == sb && a.series_idx < b.series_idx);
}

// Per-query merge of `world` sorted lists into the global top_n: one CTA per query (blockIdx.x).  List r of query q starts at
// recs[r * rank_stride + q * top_n] -- the exchange's receive buffer ([world][capacity]) and a gathered array
// ([world][n_refs][top_n]) have that same layout.  Each list is valid records in order, then padding (flags != 0), so a
// record's place in the merged order is its own index plus, in every other list, the number of records before it: one
// binary search per list, O(world * top_n * log top_n) per query and no shared-memory bound on top_n.  Equal keys in two
// lists (not produced by disjoint shards) go to the lower rank first, so positions stay distinct.  The lists were filtered on
// their shards: no filter here.  out[q * top_n ..] gets the merged list padded with flags = 1; n_out[q] (may be NULL) its length.
__device__ __forceinline__ long long list_count_before(const PartialRec *__restrict__ list, long long top_n, const PartialRec &x,
                                                       bool or_equal) {
    long long lo = 0, hi = top_n;      // first k whose record does not come before x (padding never does)
    while (lo < hi) {
        const long long mid = (lo + hi) >> 1;
        const PartialRec y = list[mid];
        const bool before = y.flags == 0 && (rec_precedes(y, x) || (or_equal && !rec_precedes(x, y)));
        if (before) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

__global__ void __launch_bounds__(256)
multi_merge_kernel(const PartialRec *__restrict__ recs, int world, long long rank_stride, long long top_n,
                   PartialRec *__restrict__ out, long long *__restrict__ n_out) {
    const long long q = blockIdx.x;
    const PartialRec *base = recs + q * top_n;
    PartialRec *o = out + q * top_n;
    __shared__ unsigned long long total;
    if (threadIdx.x == 0) total = 0ull;
    __syncthreads();
    for (int r = threadIdx.x; r < world; r += blockDim.x) {     // valid records of list r: the first padding record
        const PartialRec *list = base + (long long)r * rank_stride;
        long long lo = 0, hi = top_n;
        while (lo < hi) {
            const long long mid = (lo + hi) >> 1;
            if (list[mid].flags == 0) lo = mid + 1;
            else hi = mid;
        }
        atomicAdd(&total, (unsigned long long)lo);
    }
    for (long long g = threadIdx.x; g < (long long)world * top_n; g += blockDim.x) {
        const int r = (int)(g / top_n);
        const long long j = g - (long long)r * top_n;
        const PartialRec x = base[(long long)r * rank_stride + j];
        if (x.flags != 0) continue;
        long long pos = j;
        for (int s = 0; s < world && pos < top_n; s++)
            if (s != r) pos += list_count_before(base + (long long)s * rank_stride, top_n, x, s < r);
        if (pos < top_n) o[pos] = x;
    }
    __syncthreads();
    const long long n = (long long)total < top_n ? (long long)total : top_n;
    for (long long k = n + threadIdx.x; k < top_n; k += blockDim.x) o[k] = PartialRec{0ull, 0.0, 0ll, 0, 1};
    if (threadIdx.x == 0 && n_out) n_out[q] = n;
}

// ---- grouped shards: every group representative (unfiltered, SURVEY F2) pushed to every GPU ------------------------
// Flags carry (epoch << 32) | record count of the sender (0xffffffff: more representatives than the buffer holds).
// One thread per series: the representative of its group (lowest index among the members holding the group max,
// muse_batch.go:87-89) builds its muse_partial record -- the rank-independent group key included -- and stores it into
// slot [rank] of every rank's receive buffer.
__global__ void __launch_bounds__(256)
group_records_push_kernel(GroupTable gt, KeyCols kc, const int64_t *__restrict__ slot_of, const double *__restrict__ score,
                          const int32_t *__restrict__ lag, long long S, long long global_offset, long long capacity,
                          unsigned long long *__restrict__ n_local, ExchangePeers ex) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < S) {
        const double sc = score[i];
        if (sc == sc && gt.gidx[slot_of[i]] == (int32_t)i) {
            const unsigned long long pos = atomicAdd(n_local, 1ull);
            if ((long long)pos < capacity) {
                const long long gi = global_offset + i;
                const PartialRec rec{canonical_key(kc, i), sc, gi, lag[i], 0};
                for (int d = 0; d < ex.world; d++) ex.recs[d][(long long)ex.rank * capacity + (long long)pos] = rec;
            }
        }
    }
    if (!last_block_fenced(ex.done_blocks)) return;
    const unsigned long long n = *n_local;
    release_flags(ex, (ex.epoch << 32) | (n > (unsigned long long)capacity ? 0xffffffffull : n));
    if (threadIdx.x == 0) *n_local = 0ull;
}

// ---- merge of all shards' records on the device: group max across shards BEFORE the filter (muse_batch.go:87-89, ties ->
// lowest global series index), filter (results.go:46-52), top-N (results.go:55-87); only top_n records go to the host ------
struct MergeState {
    unsigned long long *hkeys;     // [slots] group key + 1 (0 = empty)
    unsigned long long *gmax;      // [slots] best |score| bits of the group
    unsigned long long *gidx;      // [slots] lowest global series index among the records holding it
    long long slots;               // power of two
    unsigned long long *ckey;      // candidates: |score| bits
    long long *cidx;               //             global series index
    int32_t *clag;                 //             2 * lag + (score < 0)
    unsigned long long *counters;  // [0] candidates, [1] status (1: some shard overflowed), [2] records seen
};

__device__ __forceinline__ long long merge_slot(const MergeState &m, unsigned long long group_key) {
    return hash_slot(m.hkeys, m.slots, group_key + 1ull);
}

// record j of shard r is live when j < the count its flag word carries
__device__ __forceinline__ bool merge_record(const PartialRec *recs, const unsigned long long *flags, int world, long long capacity,
                                             long long g, PartialRec &out) {
    const long long r = g / capacity, j = g - r * capacity;
    if (r >= world) return false;
    const unsigned long long n = flags[r] & 0xffffffffull;
    if (n == 0xffffffffull || (unsigned long long)j >= n) return false;
    out = recs[g];
    return !(out.flags & 1) && out.score == out.score;
}

__global__ void merge_max_kernel(MergeState m, const PartialRec *__restrict__ recs, const unsigned long long *__restrict__ flags, int world,
                                 long long capacity) {
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g < world && (flags[g] & 0xffffffffull) == 0xffffffffull) m.counters[1] = 1ull;      // a shard had more records than its slot holds
    PartialRec p;
    if (!merge_record(recs, flags, world, capacity, g, p)) return;
    atomicMax(&m.gmax[merge_slot(m, p.group_key)], score_bits(p.score));
}
__global__ void merge_rep_kernel(MergeState m, const PartialRec *__restrict__ recs, const unsigned long long *__restrict__ flags, int world,
                                 long long capacity) {
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    PartialRec p;
    if (!merge_record(recs, flags, world, capacity, g, p)) return;
    const long long s = merge_slot(m, p.group_key);
    if (score_bits(p.score) == m.gmax[s]) atomicMin(&m.gidx[s], (unsigned long long)p.series_idx);
}
__global__ void merge_emit_kernel(MergeState m, const PartialRec *__restrict__ recs, const unsigned long long *__restrict__ flags, int world,
                                  long long capacity, FilterArgs f) {
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    PartialRec p;
    bool emit = merge_record(recs, flags, world, capacity, g, p);
    if (emit) {
        const long long s = merge_slot(m, p.group_key);
        emit = score_bits(p.score) == m.gmax[s] && (unsigned long long)p.series_idx == m.gidx[s] && passed(f, p.score, p.lag);
    }
    warp_append(&m.counters[0], emit, [&](unsigned long long pos) {
        m.ckey[pos] = score_bits(p.score);
        m.cidx[pos] = p.series_idx;
        m.clag[pos] = 2 * p.lag + (p.score < 0.0 ? 1 : 0);
    });
}
// rank by counting, as partial_topn_kernel, on (|score| desc, GLOBAL series index asc); out[0 .. top_n) padded with flags = 1,
// out[0].flags = 2 when the list is too long for this kernel or a shard overflowed (the caller takes the host path)
__global__ void __launch_bounds__(256)
merged_topn_kernel(MergeState m, long long top_n, PartialRec *__restrict__ out) {
    const unsigned long long n = m.counters[0];
    rank_topn(m.ckey, m.cidx, m.clag, n, n > MUSE_PARTIAL_RANK_CAP || m.counters[1] != 0ull, top_n, 0ll, top_n, 1,
              [&](int, long long r, const PartialRec &rec) { out[r] = rec; });
}

// ---- radix select of the top_n candidates by (key desc, idx asc) ---------------------
// 96-bit composite (key, ~idx) examined 16 bits at a time, most significant first.
// State lives on the device; round r narrows [prefix] and the remaining rank.
struct SelectState {
    unsigned long long prefix_key;   // decided high bits of key
    unsigned int prefix_idx;         // decided high bits of ~idx
    unsigned long long want;         // how many still to take inside the current bucket
    unsigned int hist[65536];
    unsigned int done_blocks;
};

__device__ __forceinline__ unsigned digit_of(unsigned long long key, unsigned nidx, int r) {
    return r < 4 ? (unsigned)((key >> (48 - 16 * r)) & 0xffffull) : (unsigned)((nidx >> (16 * (5 - r))) & 0xffffu);
}
__device__ __forceinline__ bool prefix_match(const SelectState *st, unsigned long long key, unsigned nidx, int r) {
    if (r == 0) return true;
    if (r <= 4) {
        const int sh = 64 - 16 * r;
        return sh >= 64 ? true : ((key >> sh) == (st->prefix_key >> sh));
    }
    if (key != st->prefix_key) return false;
    const int sh = 32 - 16 * (r - 4);
    return (nidx >> sh) == (st->prefix_idx >> sh);
}

__global__ void select_round_kernel(SelectState *st, const unsigned long long *__restrict__ key,
                                    const int32_t *__restrict__ idx, unsigned long long ncand, int r) {
    const unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    bool in = false;
    unsigned d = 0;
    if (i < ncand) {
        const unsigned long long k = key[i];
        const unsigned ni = ~(unsigned)idx[i];
        in = prefix_match(st, k, ni, r);
        d = digit_of(k, ni, r);
    }
    // scores cluster in a few digits: one atomic per distinct digit per warp, not per lane
    const unsigned active = __ballot_sync(0xffffffffu, in);
    if (in) {
        const unsigned peers = __match_any_sync(active, d);
        if ((threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&st->hist[d], (unsigned)__popc(peers));
    }
    __shared__ bool last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) last = (atomicAdd(&st->done_blocks, 1u) == gridDim.x - 1);
    __syncthreads();
    if (!last) return;
    __threadfence();
    // the last block scans the histogram from the top digit down (single thread per 64 bins
    // then a serial pass over 1024 partials is plenty for a 64K table)
    __shared__ unsigned long long part[1024];
    unsigned long long s = 0;
    for (int b = 0; b < 64; b++) s += st->hist[threadIdx.x * 64 + b];
    part[threadIdx.x] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long want = st->want, acc = 0;
        int g = 1023;
        for (; g > 0; g--) {
            if (acc + part[g] >= want) break;
            acc += part[g];
        }
        int d = g * 64 + 63;
        for (; d > g * 64; d--) {
            if (acc + st->hist[d] >= want) break;
            acc += st->hist[d];
        }
        // digit d holds the boundary; everything above it is taken outright
        st->want = want - acc;
        if (r < 4) st->prefix_key |= ((unsigned long long)d) << (48 - 16 * r);
        else st->prefix_idx |= ((unsigned)d) << (16 * (5 - r));
        st->done_blocks = 0;
    }
    __syncthreads();
    for (int b = 0; b < 64; b++) st->hist[threadIdx.x * 64 + b] = 0;
}

// Gather every candidate whose composite is >= the selected boundary.
__global__ void select_gather_kernel(const SelectState *st, const unsigned long long *__restrict__ key,
                                     const int32_t *__restrict__ idx, unsigned long long ncand,
                                     const int32_t *__restrict__ lagsgn,
                                     unsigned long long *__restrict__ out_key, int32_t *__restrict__ out_idx,
                                     int32_t *__restrict__ out_lagsgn, unsigned long long *out_n) {
    const unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ncand) return;
    const unsigned long long k = key[i];
    const unsigned ni = ~(unsigned)idx[i];
    const bool take = k > st->prefix_key || (k == st->prefix_key && ni >= st->prefix_idx);
    if (take) {
        const unsigned long long pos = atomicAdd(out_n, 1ull);
        out_key[pos] = k;
        out_idx[pos] = idx[i];
        out_lagsgn[pos] = lagsgn[i];
    }
}

}  // namespace muse
#endif
