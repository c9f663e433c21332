// muse_api.cu -- the C ABI of include/muse_b200.h: handles, device memory, launches.
//
// Host code here only moves bytes, sizes launches and finishes the <= top_n sized tail
// (sorting the selected records); all arithmetic on series data happens in the kernels.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <deque>
#include <memory>
#include <mutex>
#include <thread>
#include <unordered_map>
#include <utility>
#include <vector>

#include "../../include/muse_b200.h"
#include "muse_launch.h"
#include "muse_select.cuh"
#include "muse_synth.cuh"
#include "muse_xcorr.cuh"

using namespace muse;

// ------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

static int fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

// A failed runtime call: its error is reported here, so it must not resurface in a later cudaGetLastError() check.
static int cuda_fail(cudaError_t e, const char *call, const char *file, int line) {
    (void)cudaGetLastError();
    return fail(e == cudaErrorMemoryAllocation ? MUSE_ERR_OUT_OF_MEMORY : MUSE_ERR_CUDA, "%s failed: %s (%s:%d)", call,
                cudaGetErrorString(e), file, line);
}

#define CU(call)                                                                 \
    do {                                                                         \
        cudaError_t e_ = (call);                                                 \
        if (e_ != cudaSuccess) return cuda_fail(e_, #call, __FILE__, __LINE__); \
    } while (0)

extern "C" const char *muse_last_error(void) { return g_err; }
extern "C" const char *muse_version(void) { return "muse_b200 0.1 (sm_100a)"; }

// ------------------------------------------------------------------------------------
// owners of device and page-locked memory and of events
// ------------------------------------------------------------------------------------
// Every device and page-locked allocation of the library is one of these (muse_host_alloc hands its memory to the caller),
// so whoever holds the owner frees it, on every path.  g_held counts the bytes they hold: [0] device, [1] page-locked.
static std::atomic<int64_t> g_held[2];

template <typename T, bool Pinned>
class Buf {
  public:
    Buf() = default;
    Buf(Buf &&o) noexcept { swap(o); }
    Buf &operator=(Buf &&o) noexcept {      // the old contents go to `o`, which frees them
        swap(o);
        return *this;
    }
    ~Buf() { release(); }
    T *get() const { return p_; }
    operator T *() const { return p_; }
    T *operator->() const { return p_; }
    int64_t cap() const { return cap_; }
    // Room for n elements: when n exceeds the capacity, the buffer is freed and reallocated; the contents are not kept.
    cudaError_t grow(int64_t n) {
        if (n <= cap_) return cudaSuccess;
        release();
        const size_t bytes = sizeof(T) * (size_t)n;
        cudaError_t e = Pinned ? cudaHostAlloc((void **)&p_, bytes, cudaHostAllocDefault) : cudaMalloc((void **)&p_, bytes);
        if (e != cudaSuccess) {
            p_ = nullptr;
            return e;
        }
        cap_ = n;
        g_held[Pinned] += (int64_t)bytes;
        return cudaSuccess;
    }

  private:
    void swap(Buf &o) {
        std::swap(p_, o.p_);
        std::swap(cap_, o.cap_);
    }
    void release() {      // cudaFree waits for the device, so work still queued on the buffer is done first
        if (!p_) return;
        if (Pinned) cudaFreeHost(p_);
        else cudaFree(p_);
        g_held[Pinned] -= (int64_t)(sizeof(T) * (size_t)cap_);
        p_ = nullptr;
        cap_ = 0;
    }
    T *p_ = nullptr;
    int64_t cap_ = 0;
};
template <typename T>
using DevBuf = Buf<T, false>;
using PinnedBuf = Buf<unsigned char, true>;

// K events, created together on first use
template <int K>
class Events {
  public:
    Events() = default;
    Events(Events &&o) noexcept { std::swap(e_, o.e_); }
    Events &operator=(Events &&o) noexcept {
        std::swap(e_, o.e_);
        return *this;
    }
    ~Events() {
        for (cudaEvent_t e : e_)
            if (e) cudaEventDestroy(e);
    }
    cudaEvent_t operator[](int i) const { return e_[i]; }
    cudaError_t create(unsigned flags = cudaEventDefault) {
        for (cudaEvent_t &e : e_) {
            const cudaError_t r = e ? cudaSuccess : cudaEventCreateWithFlags(&e, flags);
            if (r != cudaSuccess) return r;
        }
        return cudaSuccess;
    }

  private:
    cudaEvent_t e_[K] = {};
};

extern "C" int muse_held_bytes(int64_t *device_bytes, int64_t *pinned_bytes) {
    if (!device_bytes || !pinned_bytes) return fail(MUSE_ERR_INVALID_ARG, "muse_held_bytes: NULL argument");
    *device_bytes = g_held[0].load();
    *pinned_bytes = g_held[1].load();
    return MUSE_OK;
}

// ------------------------------------------------------------------------------------
// handles
// ------------------------------------------------------------------------------------
// Everything a batch needs per run whose size follows the store (not the reference): kept in a small
// per-context pool across muse_batch_create / muse_batch_destroy, because cudaMalloc / cudaFree /
// cudaHostAlloc of these cost milliseconds to seconds (measured: a NewBatch + Run + destroy cycle per
// request spent 3 s in cudaFree/cudaFreeHost once in four) while the run itself takes 2.7 ms.
#define MUSE_MAX_LABEL_KEYS 64   // label-key columns of a store (the facade adds one all-absent column)
#define MUSE_SCRATCH_POOL 272   // scratch sets kept per context (MUSE_MULTI_GROUP + MUSE_MULTI_SEPARATE): room for the batches
                                // of a tensor-core launch group and of a group of separate batches in muse_multi_run
#define MUSE_MULTI_GROUP 256    // queries of one launch of the tensor-core multi-query path (== TcCfg::TN == RefineMultiCfg::QMAX)
#define MUSE_MULTI_SEPARATE 16  // queries of one group of separate batches in muse_multi_run (one upload, one round trip)
#define MUSE_DEVICE_TOPN_MAX 65536   // top_n of a device-side top-N: its records come back through the mailbox
#define MUSE_SELECT_CHUNK 32768      // candidates that come back with their count (run_select)
// The pinned mailbox of a batch for the small device->host results (one copy per round trip).
struct Mailbox {
    int32_t flag;          // the reference's std-zero flag (no screening tables)
    float mid[4];          // screening tables: [0] the std-zero flag (as float bits), [1] A[M/2], [2..3] Xt[M/2]
    RunCounters counters;
    union {
        struct {           // run_select: the first candidates
            unsigned long long key[MUSE_SELECT_CHUNK];
            int32_t idx[MUSE_SELECT_CHUNK], lagsgn[MUSE_SELECT_CHUNK];
        } cand;
        muse_partial recs[MUSE_DEVICE_TOPN_MAX];   // the device-side top-N
    };
};
static_assert(sizeof(Mailbox::cand) <= sizeof(Mailbox::recs) && sizeof(Mailbox::recs) == sizeof(muse_partial) * MUSE_DEVICE_TOPN_MAX,
              "the device-side top-N records size the mailbox");

// The device-side top-N of top_n records applies when the mailbox holds them and the sort scratch d_skey, 8 bytes per entry
// of `capacity` entries, holds them as records.
static bool device_topn_fits(int64_t top_n, int64_t capacity) {
    return top_n > 0 && top_n <= MUSE_DEVICE_TOPN_MAX && top_n * (int64_t)(sizeof(muse_partial) / 8) <= capacity;
}

struct RunScratch {
    int64_t scratch_cap = 0;                  // entries of the twelve arrays below (ensure_scratch)
    DevBuf<double> d_score;
    DevBuf<int32_t> d_lag;
    DevBuf<int64_t> d_slot;
    DevBuf<unsigned long long> d_ckey, d_skey;
    DevBuf<int32_t> d_cidx, d_sidx;
    DevBuf<int32_t> d_clag, d_slag;           // 2*lag + sign of the candidates (muse_select.cuh Cand)
    DevBuf<float> d_U;
    DevBuf<int32_t> d_list;
    DevBuf<float> d_L;                        // lower bounds (grouped screened runs, diagnostic entry point)
    DevBuf<signed char> d_W;                  // grouped screened runs: lag-window verdict of every refined series (ScreenParams::out_W)
    DevBuf<int32_t> d_rows;                   // filtered runs: the selected local rows in ascending order (muse_batch_run_where)
    DevBuf<int32_t> d_where_off;              // filtered runs: per-block offsets of the selection, then its length
    Buf<Mailbox, true> h_pin;
    DevBuf<RunCounters> d_counters;
    DevBuf<SelectState> d_sel;
    DevBuf<int32_t> d_flag;
    DevBuf<CutState> d_cut;                   // fused refinement state
    // group table
    DevBuf<unsigned long long> d_gmax, d_hkeys;
    DevBuf<int32_t> d_gidx;
    // tables of the reference side.  tab_n: the FFT length the twiddle tables (twM, twn, twp_f, swtw) were filled
    // for -- a set that comes back from the pool with the same n keeps them, only the per-reference ones
    // (d_ref, Xt, sw_f, sx_f, d_mid) are rewritten by muse_batch_create
    int64_t tab_n = 0;
    int tab_screen = 0;                       // twp_f / swtw / sw_f / sx_f exist for tab_n
    DevBuf<double> d_ref;                     // padded copy of the reference row
    DevBuf<cd> Xt, twM, twn;
    DevBuf<cf> twp_f;                         // fp32 screening pass: per-pass twiddles
    DevBuf<cf> twi_f;                         // n = 4096 .. 16384: twiddle tables of muse_screen_big.cuh
    DevBuf<float2> swtw;                      // split twiddles exp(-2*pi*i*k/n), k < M/2, fp32
    DevBuf<float4> sw_f;                      // fused kernels: (twn, A[k], A[M-k]) per k < M/2
    DevBuf<float4> sx_f;                      // fused refinement: (Xt[k], Xt[M-k]) in fp32 per k < M/2
    DevBuf<float> sb_f;                       // warp / sub-warp kernels: sqrt(2 (A[k]^2 + A[M-k]^2)) rounded up per k < M/2
    DevBuf<float> d_mid;                      // [0] std-zero flag of the reference (as float bits), [1] A[M/2], [2..3] Xt[M/2] in fp32
    Events<4> ev;
};

struct muse_ctx {
    int device = 0;
    int sm_count = 0;
    cudaStream_t stream = nullptr;       // the stream in use
    cudaStream_t own_stream = nullptr;   // created with the context
    std::mutex mu;
    std::deque<RunScratch> pool;    // scratch sets of destroyed batches, reused by the next muse_batch_create (a deque: taking
                                    // the front set moves no other set)
    PinnedBuf h_stage[3];           // pinned staging ring for rows that arrive in pageable host memory (muse_group_append, muse_group_roll)
    Events<3> stage_ev;
    DevBuf<double> d_roll;          // device buffer of the new samples of muse_group_roll: at most MUSE_STAGE_BYTES
    DevBuf<int2> d_moves;           // (from, to) row pairs of muse_group_remove: MUSE_MOVE_CHUNK entries once the first row moves
    // multi-query bounds on the tensor cores (muse_bounds_tc.cuh): magnitudes of the store and weights of a launch's queries
    DevBuf<unsigned char> tc_a, tc_b;     // bf16 tiles: [S/128][16][16 KB] and [16][32 KB]
    DevBuf<float> tc_mid, tc_amid;        // [S] |2Y_(M/2)| per series, [256] A_q[M/2] per query
    DevBuf<void *> tc_ptrs;               // device: [256] sw tables, [256] bound arrays
    DevBuf<unsigned> d_multi_next;        // work counter of refine_multi_kernel
    DevBuf<unsigned char> d_mt;           // parameter tables and results of a multi-query launch (MultiTables), device and pinned host
    PinnedBuf h_mt;
    Events<5> mt_ev;                // stage boundaries of the last multi-query launch group: start, magnitudes, bounds, second stages, end
    int64_t multi_refined = 0, multi_rescored = 0;      // totals of the last muse_multi_run (second stages, fp64 re-scorings)
    DevBuf<MultiQuery> d_multi_q;   // query table of refine_multi_kernel (MUSE_MULTI_GROUP entries)
    DevBuf<double> d_multi_refs;    // [MUSE_MULTI_GROUP][d_multi_ld] reference rows of a muse_multi_run group, pad columns kept zero
    int64_t d_multi_ld = 0, d_multi_n = 0;
    DevBuf<int32_t> d_where_rows;   // muse_multi_run_where: the selection shared by every reference of the call (ascending local rows)
    DevBuf<int32_t> d_where_off;    // its per-tile offsets, then its length
};

struct muse_group {
    muse_ctx *ctx = nullptr;
    int64_t N = 0;          // series length
    int64_t ld = 0;         // row stride in doubles (multiple of 16 -> 128-byte rows)
    int64_t cap = 0, size = 0;
    DevBuf<double> slab;    // [cap][ld]
    int nkeys = 0;
    DevBuf<int32_t> labels; // [nkeys][cap]
    int32_t max_id[MUSE_MAX_LABEL_KEYS] = {};
    int64_t global_offset = 0;
    DevBuf<RowStat> row_stat;   // [cap] screening: fp64 mean and fp32 1/std of each row (filled lazily up to stats_upto)
    int64_t stats_upto = 0;
};

struct muse_batch : RunScratch {
    muse_ctx *ctx = nullptr;
    muse_group *g = nullptr;
    int64_t N = 0, n = 0;
    int log2m = 0;
    // fp32 screening pass (n = 128 .. 16384): the tables live in RunScratch
    int screen_ok = 0;
    float a_mid = 0.f;
    cf x_mid = {};
    muse_timing timing = {};
    // the last run's state that muse_batch_last_timing reads after the call has returned (finish_pending_timing, settle_counters)
    int timing_pending = 0;    // the last run was queued without a final synchronisation (muse_batch_run_partial_device)
    int fused_run = 0;         // 1: score_fused, 2: score_fused_grouped (d_counters: listed = exact list length)
    // n > MUSE_MAX_FUSED_FFT_LEN: Stockham passes through global memory (kernels_long.cu); Xt holds n entries, twM the n twiddles
    int is_long = 0;
    DevBuf<unsigned char> d_long;   // work buffer of launch_long
    long long long_pairs = 0;       // pairs of series per chunk d_long was sized for
};

extern "C" void muse_batch_destroy(muse_batch *b);
struct BatchDestroy {
    void operator()(muse_batch *b) const { muse_batch_destroy(b); }
};
using BatchPtr = std::unique_ptr<muse_batch, BatchDestroy>;   // a batch that goes back through muse_batch_destroy

static inline cudaStream_t bstream(const muse_batch *b) { return b->ctx->stream; }

// ------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------
extern "C" int muse_ctx_create(int device, muse_ctx **out) {
    if (!out) return fail(MUSE_ERR_INVALID_ARG, "muse_ctx_create: out is NULL");
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(MUSE_ERR_NO_DEVICE, "no CUDA device (%s); muse_b200 has no CPU fallback",
                    e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    if (device < 0 || device >= count) return fail(MUSE_ERR_INVALID_ARG, "device %d out of range [0,%d)", device, count);
    CU(cudaSetDevice(device));
    std::unique_ptr<muse_ctx> c(new muse_ctx());
    c->device = device;
    CU(cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, device));
    CU(cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking));
    c->stream = c->own_stream;
    *out = c.release();
    return MUSE_OK;
}

extern "C" void muse_ctx_destroy(muse_ctx *c) {
    if (!c) return;
    cudaSetDevice(c->device);
    const cudaStream_t own = c->own_stream;
    delete c;      // the pool and every buffer of the context
    cudaStreamDestroy(own);
}

extern "C" int muse_ctx_synchronize(muse_ctx *c) {
    if (!c) return fail(MUSE_ERR_INVALID_ARG, "ctx is NULL");
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    return MUSE_OK;
}

extern "C" int muse_ctx_set_stream(muse_ctx *c, void *cuda_stream) {
    if (!c) return fail(MUSE_ERR_INVALID_ARG, "ctx is NULL");
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    c->stream = cuda_stream ? (cudaStream_t)cuda_stream : c->own_stream;
    return MUSE_OK;
}

extern "C" int muse_host_alloc(void **out, int64_t bytes) {
    if (!out || bytes < 0) return fail(MUSE_ERR_INVALID_ARG, "muse_host_alloc: bad argument");
    CU(cudaHostAlloc(out, (size_t)bytes, cudaHostAllocDefault));
    return MUSE_OK;
}

extern "C" void muse_host_free(void *p) {
    if (p) cudaFreeHost(p);
}

// ------------------------------------------------------------------------------------
// series store
// ------------------------------------------------------------------------------------
static int group_reserve(muse_group *g, int64_t want) {
    if (want <= g->cap) return MUSE_OK;
    int64_t ncap = std::max<int64_t>(want, g->cap + g->cap / 2);
    ncap = std::max<int64_t>(ncap, 16);
    DevBuf<double> nslab;
    DevBuf<int32_t> nlab;
    DevBuf<RowStat> nstat;
    cudaError_t e = nslab.grow(ncap * g->ld);
    if (e == cudaSuccess && g->nkeys > 0) e = nlab.grow(ncap * g->nkeys);
    if (e == cudaSuccess) e = nstat.grow(ncap);
    if (e == cudaSuccess && g->size > 0) {
        e = cudaMemcpyAsync(nslab, g->slab, sizeof(double) * (size_t)g->size * (size_t)g->ld, cudaMemcpyDeviceToDevice, g->ctx->stream);
        for (int k = 0; k < g->nkeys && e == cudaSuccess; k++)
            e = cudaMemcpyAsync(nlab + (size_t)k * ncap, g->labels + (size_t)k * g->cap, sizeof(int32_t) * (size_t)g->size,
                                cudaMemcpyDeviceToDevice, g->ctx->stream);
        if (e == cudaSuccess && g->stats_upto > 0)
            e = cudaMemcpyAsync(nstat, g->row_stat, sizeof(RowStat) * (size_t)g->stats_upto, cudaMemcpyDeviceToDevice, g->ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(g->ctx->stream);
    }
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        return fail(e == cudaErrorMemoryAllocation ? MUSE_ERR_OUT_OF_MEMORY : MUSE_ERR_CUDA, "growing the store to %lld series: %s",
                    (long long)ncap, cudaGetErrorString(e));
    }
    std::swap(g->slab, nslab);      // the old arrays are freed on the way out
    std::swap(g->labels, nlab);
    std::swap(g->row_stat, nstat);
    g->cap = ncap;
    return MUSE_OK;
}

// RowStat of rows [first, first + count): the batched mean / sample-std kernel of the z-normalisation (xcorr.go:84-95),
// queued right behind the copy that brought the rows in, so that no Run ever pays a separate pass over the slab.
static int queue_row_stats(muse_group *g, int64_t first, int64_t count) {
    if (count <= 0) return MUSE_OK;
    const unsigned grid = (unsigned)std::min<int64_t>((count + 7) / 8, (int64_t)g->ctx->sm_count * 16);
    row_stats_kernel<<<grid, 256, 0, g->ctx->stream>>>(g->slab, g->ld, (int)g->N, first, count, g->row_stat);
    CU(cudaGetLastError());
    return MUSE_OK;
}

extern "C" int muse_group_create(muse_ctx *ctx, int64_t series_len, int32_t n_label_keys, int64_t capacity_hint,
                                 muse_group **out) {
    if (!ctx || !out) return fail(MUSE_ERR_INVALID_ARG, "muse_group_create: NULL argument");
    if (series_len < 2)
        return fail(MUSE_ERR_INVALID_ARG, "series length %lld: the sample std needs at least 2 samples (xcorr.go:88)",
                    (long long)series_len);
    if (n_label_keys < 0 || n_label_keys > MUSE_MAX_LABEL_KEYS)
        return fail(MUSE_ERR_INVALID_ARG, "n_label_keys %d not in [0,%d]", n_label_keys, MUSE_MAX_LABEL_KEYS);
    CU(cudaSetDevice(ctx->device));
    std::unique_ptr<muse_group> g(new muse_group());
    g->ctx = ctx;
    g->N = series_len;
    g->ld = (series_len + 15) / 16 * 16;
    g->nkeys = n_label_keys;
    for (int k = 0; k < MUSE_MAX_LABEL_KEYS; k++) g->max_id[k] = -1;
    int rc = group_reserve(g.get(), std::max<int64_t>(capacity_hint, 16));
    if (rc != MUSE_OK) return rc;
    *out = g.release();
    return MUSE_OK;
}

extern "C" void muse_group_destroy(muse_group *g) {
    if (!g) return;
    cudaSetDevice(g->ctx->device);
    delete g;
}

// Pageable host rows of `width` doubles -> the device through a ring of three pinned buffers: MUSE_STAGE_THREADS host threads
// copy chunk c into buffer c % 3 while chunk c - 1 is on the wire (at most two DMA copies outstanding, so a buffer is free
// again when its turn comes).  A chunk is a whole number of rows, at most MUSE_STAGE_BYTES; queue(r0, nr, pinned) enqueues on
// the context's stream the copy (and whatever follows it) that takes rows [r0, r0 + nr) out of the pinned buffer.
#define MUSE_STAGE_BYTES ((size_t)64 << 20)
static int64_t stage_rows_per_chunk(int64_t width) { return (int64_t)(MUSE_STAGE_BYTES / (sizeof(double) * (size_t)width)); }

template <typename Queue>
static int stage_rows(muse_ctx *c, const double *rows, int64_t n_rows, int64_t width, Queue &&queue) {
    for (PinnedBuf &h : c->h_stage) CU(h.grow(MUSE_STAGE_BYTES));
    CU(c->stage_ev.create(cudaEventDisableTiming));
    cudaStream_t st = c->stream;
    const size_t row_bytes = sizeof(double) * (size_t)width;
    if (row_bytes > MUSE_STAGE_BYTES) return fail(MUSE_ERR_UNSUPPORTED, "a row of %zu bytes exceeds the staging buffer", row_bytes);
    const int64_t rows_per_chunk = stage_rows_per_chunk(width);
    const int64_t n_chunks = (n_rows + rows_per_chunk - 1) / rows_per_chunk;
    unsigned hw = std::thread::hardware_concurrency();
    const char *env = getenv("MUSE_STAGE_THREADS");
    int n_threads = env ? atoi(env) : (int)std::min<unsigned>(hw ? hw : 4u, 12u);
    if (n_threads < 1) n_threads = 1;
    if ((size_t)n_rows * row_bytes < ((size_t)8 << 20)) n_threads = 1;      // small copies: not worth the threads
    std::vector<std::atomic<int>> done((size_t)n_chunks);
    for (auto &d : done) d.store(0, std::memory_order_relaxed);
    std::atomic<int64_t> writable(std::min<int64_t>(n_chunks, 2));      // chunks whose buffer may be filled
    std::atomic<bool> abort_flag(false);
    auto worker = [&](int w) {
        for (int64_t ch = 0; ch < n_chunks; ch++) {
            if (abort_flag.load(std::memory_order_relaxed)) return;
            while (writable.load(std::memory_order_acquire) <= ch) {
                if (abort_flag.load(std::memory_order_relaxed)) return;
                std::this_thread::yield();
            }
            const int64_t r0 = ch * rows_per_chunk, nr = std::min<int64_t>(rows_per_chunk, n_rows - r0);
            const size_t bytes = (size_t)nr * row_bytes;
            const size_t lo = bytes * (size_t)w / (size_t)n_threads / 64 * 64, hi = (w + 1 == n_threads) ? bytes : bytes * (size_t)(w + 1) / (size_t)n_threads / 64 * 64;
            if (hi > lo) memcpy(c->h_stage[ch % 3] + lo, reinterpret_cast<const unsigned char *>(rows) + (size_t)r0 * row_bytes + lo, hi - lo);
            done[(size_t)ch].fetch_add(1, std::memory_order_release);
        }
    };
    std::vector<std::thread> pool;
    for (int w = 1; w < n_threads; w++) pool.emplace_back(worker, w);
    cudaError_t e = cudaSuccess;
    // the calling thread is worker 0 and the one that talks to the device
    for (int64_t ch = 0; ch < n_chunks && e == cudaSuccess; ch++) {
        const int64_t r0 = ch * rows_per_chunk, nr = std::min<int64_t>(rows_per_chunk, n_rows - r0);
        {
            const size_t bytes = (size_t)nr * row_bytes;
            const size_t hi = (n_threads == 1) ? bytes : bytes / (size_t)n_threads / 64 * 64;
            if (hi > 0) memcpy(c->h_stage[ch % 3], reinterpret_cast<const unsigned char *>(rows) + (size_t)r0 * row_bytes, hi);
            done[(size_t)ch].fetch_add(1, std::memory_order_release);
        }
        while (done[(size_t)ch].load(std::memory_order_acquire) < n_threads) std::this_thread::yield();
        e = queue(r0, nr, reinterpret_cast<const double *>(c->h_stage[ch % 3].get()));
        if (e == cudaSuccess) e = cudaEventRecord(c->stage_ev[ch % 3], st);
        if (e == cudaSuccess && ch >= 1) e = cudaEventSynchronize(c->stage_ev[(ch - 1) % 3]);      // buffer (ch + 2) % 3 is free again
        writable.store(ch + 3, std::memory_order_release);
    }
    if (e != cudaSuccess) abort_flag.store(true);
    writable.store(n_chunks + 3, std::memory_order_release);
    for (auto &t : pool) t.join();
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        return fail(MUSE_ERR_CUDA, "staged host->device copy failed: %s", cudaGetErrorString(e));
    }
    return MUSE_OK;
}

extern "C" int muse_group_append(muse_group *g, const double *rows, int64_t n_series, int64_t series_len,
                                 const int32_t *label_ids) {
    if (!g || (!rows && n_series > 0)) return fail(MUSE_ERR_INVALID_ARG, "muse_group_append: NULL argument");
    if (n_series < 0) return fail(MUSE_ERR_INVALID_ARG, "n_series < 0");
    if (series_len != g->N)   // group.go:45-51
        return fail(MUSE_ERR_LENGTH_MISMATCH, "Timeseries has length %lld, but current group has length %lld",
                    (long long)series_len, (long long)g->N);
    if (g->nkeys > 0 && !label_ids && n_series > 0) return fail(MUSE_ERR_INVALID_ARG, "label_ids is NULL but the group has %d label keys", g->nkeys);
    if (n_series == 0) return MUSE_OK;
    if (g->size + n_series > 0x7fffffffLL) return fail(MUSE_ERR_UNSUPPORTED, "more than 2^31-1 series in one store");
    CU(cudaSetDevice(g->ctx->device));
    int rc = group_reserve(g, g->size + n_series);
    if (rc != MUSE_OK) return rc;
    cudaStream_t st = g->ctx->stream;
    cudaPointerAttributes attr;
    const bool pinned = cudaPointerGetAttributes(&attr, rows) == cudaSuccess &&
                        (attr.type == cudaMemoryTypeHost || attr.type == cudaMemoryTypeManaged);
    (void)cudaGetLastError();
    if (!pinned) {
        // pageable rows (a Go slice, a numpy array): a direct cudaMemcpyAsync stages them through the driver's single
        // bounce buffer at a fraction of the link rate -> chunks are copied into a pinned ring by several host threads
        // while the previous chunk is on the wire
        const size_t row_bytes = sizeof(double) * (size_t)g->N;
        rc = stage_rows(g->ctx, rows, n_series, g->N, [&](int64_t r0, int64_t nr, const double *src) {
            double *dst = g->slab + (size_t)(g->size + r0) * g->ld;
            if (g->ld == g->N) return cudaMemcpyAsync(dst, src, (size_t)nr * row_bytes, cudaMemcpyHostToDevice, st);
            return cudaMemcpy2DAsync(dst, sizeof(double) * (size_t)g->ld, src, row_bytes, row_bytes, (size_t)nr, cudaMemcpyHostToDevice, st);
        });
        if (rc != MUSE_OK) return rc;
    } else if (g->ld == g->N) {   // rows are already at the slab's pitch: one flat copy (a pitched copy of 10^6 rows is not always at DMA rate)
        CU(cudaMemcpyAsync(g->slab + (size_t)g->size * g->ld, rows, sizeof(double) * (size_t)g->N * (size_t)n_series,
                           cudaMemcpyHostToDevice, st));
    } else {
        CU(cudaMemcpy2DAsync(g->slab + (size_t)g->size * g->ld, sizeof(double) * (size_t)g->ld, rows,
                             sizeof(double) * (size_t)g->N, sizeof(double) * (size_t)g->N, (size_t)n_series,
                             cudaMemcpyHostToDevice, st));
    }
    if (g->nkeys > 0) {
        // host [n_series][nkeys] -> device SoA [nkeys][cap]
        std::vector<int32_t> col((size_t)n_series);
        for (int k = 0; k < g->nkeys; k++) {
            int32_t mx = g->max_id[k];
            for (int64_t i = 0; i < n_series; i++) {
                int32_t v = label_ids[(size_t)i * g->nkeys + k];
                if (v < -1) v = -1;
                col[(size_t)i] = v;
                mx = std::max(mx, v);
            }
            g->max_id[k] = mx;
            CU(cudaMemcpyAsync(g->labels + (size_t)k * g->cap + g->size, col.data(), sizeof(int32_t) * (size_t)n_series,
                               cudaMemcpyHostToDevice, st));
            CU(cudaStreamSynchronize(st));   // col is reused
        }
    }
    rc = queue_row_stats(g, g->size, n_series);
    if (rc != MUSE_OK) return rc;
    CU(cudaStreamSynchronize(st));
    g->size += n_series;
    g->stats_upto = g->size;
    return MUSE_OK;
}

__global__ void max_id_kernel(const int32_t *ids, int64_t n, int32_t *out) {
    int32_t m = -1;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) m = max(m, ids[i]);
    for (int off = 16; off > 0; off >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, off));
    if ((threadIdx.x & 31) == 0) atomicMax(out, m);
}

__global__ void transpose_labels_kernel(const int32_t *src, int64_t n, int nkeys, int32_t *dst, int64_t cap, int64_t off) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    for (int k = 0; k < nkeys; k++) dst[(size_t)k * cap + off + i] = max(src[(size_t)i * nkeys + k], -1);
}

static int refresh_max_ids(muse_group *g, int64_t off, int64_t n) {
    if (g->nkeys == 0 || n == 0) return MUSE_OK;
    DevBuf<int32_t> d;
    CU(d.grow(MUSE_MAX_LABEL_KEYS));
    CU(cudaMemsetAsync(d, 0xff, sizeof(int32_t) * MUSE_MAX_LABEL_KEYS, g->ctx->stream));
    for (int k = 0; k < g->nkeys; k++)
        max_id_kernel<<<256, 256, 0, g->ctx->stream>>>(g->labels + (size_t)k * g->cap + off, n, d + k);
    int32_t h[MUSE_MAX_LABEL_KEYS];
    CU(cudaMemcpyAsync(h, d, sizeof(h), cudaMemcpyDeviceToHost, g->ctx->stream));
    CU(cudaStreamSynchronize(g->ctx->stream));
    for (int k = 0; k < g->nkeys; k++) g->max_id[k] = std::max(g->max_id[k], h[k]);
    return MUSE_OK;
}

extern "C" int muse_group_append_device(muse_group *g, const double *d_rows, int64_t n_series, int64_t series_len,
                                        const int32_t *d_label_ids) {
    if (!g || (!d_rows && n_series > 0)) return fail(MUSE_ERR_INVALID_ARG, "muse_group_append_device: NULL argument");
    if (series_len != g->N)
        return fail(MUSE_ERR_LENGTH_MISMATCH, "Timeseries has length %lld, but current group has length %lld",
                    (long long)series_len, (long long)g->N);
    if (g->nkeys > 0 && !d_label_ids && n_series > 0) return fail(MUSE_ERR_INVALID_ARG, "d_label_ids is NULL");
    if (n_series <= 0) return n_series == 0 ? MUSE_OK : fail(MUSE_ERR_INVALID_ARG, "n_series < 0");
    if (g->size + n_series > 0x7fffffffLL) return fail(MUSE_ERR_UNSUPPORTED, "more than 2^31-1 series in one store");
    CU(cudaSetDevice(g->ctx->device));
    int rc = group_reserve(g, g->size + n_series);
    if (rc != MUSE_OK) return rc;
    cudaStream_t st = g->ctx->stream;
    CU(cudaMemcpy2DAsync(g->slab + (size_t)g->size * g->ld, sizeof(double) * (size_t)g->ld, d_rows,
                         sizeof(double) * (size_t)g->N, sizeof(double) * (size_t)g->N, (size_t)n_series,
                         cudaMemcpyDeviceToDevice, st));
    if (g->nkeys > 0) {
        transpose_labels_kernel<<<(unsigned)((n_series + 255) / 256), 256, 0, st>>>(d_label_ids, n_series, g->nkeys, g->labels,
                                                                                  g->cap, g->size);
        CU(cudaGetLastError());
        rc = refresh_max_ids(g, g->size, n_series);
        if (rc != MUSE_OK) return rc;
    }
    rc = queue_row_stats(g, g->size, n_series);
    if (rc != MUSE_OK) return rc;
    CU(cudaStreamSynchronize(st));
    g->size += n_series;
    g->stats_upto = g->size;
    return MUSE_OK;
}

// one block per series row; coalesced 8-byte stores.  The row's RowStat (row_stats_kernel's sums about the first
// sample) is accumulated while the samples are generated: a synthetic store never needs a pass of its own for them.
__global__ void __launch_bounds__(256)
synth_rows_kernel(double *slab, int64_t ld, int64_t N, int64_t row0, int64_t n_series, uint64_t seed,
                  int64_t first_index, int32_t *lab0, int32_t *lab1, RowStat *stat, int variant) {
    __shared__ double red[2][8];
    for (int64_t r = blockIdx.x; r < n_series; r += gridDim.x) {
        const int64_t gi = first_index + r;
        const SynthSeries sp = synth_params(seed, gi, N, variant);
        double *row = slab + (size_t)(row0 + r) * ld;
        const double pivot = synth_value(seed, gi, sp, 0);
        double s1 = 0.0, s2 = 0.0;
        for (int64_t t = threadIdx.x; t < ld; t += blockDim.x) {
            const double v = t < N ? synth_value(seed, gi, sp, t) : 0.0;
            row[t] = v;
            if (t < N) {
                const double x = v - pivot;
                s1 += x;
                s2 = fma(x, x, s2);
            }
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            s1 += __shfl_xor_sync(0xffffffffu, s1, off);
            s2 += __shfl_xor_sync(0xffffffffu, s2, off);
        }
        if ((threadIdx.x & 31) == 0) {
            red[0][threadIdx.x >> 5] = s1;
            red[1][threadIdx.x >> 5] = s2;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            s1 = s2 = 0.0;
            for (int w = 0; w < (int)(blockDim.x >> 5); w++) {
                s1 += red[0][w];
                s2 += red[1][w];
            }
            const RowStat rsr = make_row_stat(pivot, s1, s2, (int)N);
            stat[row0 + r] = rsr;
            if (N & 1) row[N] = rsr.mean;      // odd length: the pad column the screening kernels read with the last sample (RowStat)
            if (lab0) lab0[row0 + r] = (int32_t)(gi / 1000);
            if (lab1) lab1[row0 + r] = (int32_t)(gi % 1000);
        }
        __syncthreads();
    }
}

extern "C" int muse_group_append_synthetic_ex(muse_group *g, int64_t n_series, uint64_t seed, int64_t first_index, int32_t variant);
extern "C" int muse_group_append_synthetic(muse_group *g, int64_t n_series, uint64_t seed, int64_t first_index) {
    return muse_group_append_synthetic_ex(g, n_series, seed, first_index, 0);
}

extern "C" int muse_group_append_synthetic_ex(muse_group *g, int64_t n_series, uint64_t seed, int64_t first_index, int32_t variant) {
    if (!g || n_series < 0 || variant < 0 || variant > 1) return fail(MUSE_ERR_INVALID_ARG, "muse_group_append_synthetic: bad argument");
    if (n_series == 0) return MUSE_OK;
    if (g->size + n_series > 0x7fffffffLL) return fail(MUSE_ERR_UNSUPPORTED, "more than 2^31-1 series in one store");
    CU(cudaSetDevice(g->ctx->device));
    int rc = group_reserve(g, g->size + n_series);
    if (rc != MUSE_OK) return rc;
    int32_t *l0 = g->nkeys >= 1 ? g->labels.get() : nullptr;
    int32_t *l1 = g->nkeys >= 2 ? g->labels + (size_t)g->cap : nullptr;
    if (g->nkeys > 2)
        CU(cudaMemsetAsync(g->labels + (size_t)2 * g->cap, 0, sizeof(int32_t) * (size_t)g->cap * (size_t)(g->nkeys - 2), g->ctx->stream));
    const unsigned grid = (unsigned)std::min<int64_t>(n_series, (int64_t)g->ctx->sm_count * 16);
    synth_rows_kernel<<<grid, 256, 0, g->ctx->stream>>>(g->slab, g->ld, g->N, g->size, n_series, seed, first_index, l0, l1, g->row_stat, variant);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(g->ctx->stream));
    g->stats_upto = g->size + n_series;
    if (g->nkeys >= 1) g->max_id[0] = std::max<int32_t>(g->max_id[0], (int32_t)((first_index + n_series - 1) / 1000));
    if (g->nkeys >= 2) g->max_id[1] = std::max<int32_t>(g->max_id[1], (int32_t)std::min<int64_t>(999, first_index + n_series - 1));
    for (int k = 2; k < g->nkeys; k++) g->max_id[k] = std::max(g->max_id[k], 0);
    g->size += n_series;
    return MUSE_OK;
}

// label id of key k for global series index i: (i / div[k]) % mod[k]
__global__ void synth_labels_kernel(int32_t *labels, int64_t cap, int nkeys, int64_t row0, int64_t n_series, int64_t first_index,
                                    const int64_t d0, const int64_t m0, const int64_t d1, const int64_t m1, const int64_t d2,
                                    const int64_t m2, const int64_t d3, const int64_t m3) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_series) return;
    const int64_t gi = first_index + r;
    const int64_t d[4] = {d0, d1, d2, d3}, m[4] = {m0, m1, m2, m3};
    for (int k = 0; k < nkeys && k < 4; k++) labels[(size_t)k * cap + row0 + r] = (int32_t)((gi / d[k]) % m[k]);
}

extern "C" int muse_group_set_synthetic_labels(muse_group *g, const int64_t *div, const int64_t *mod) {
    if (!g || !div || !mod) return fail(MUSE_ERR_INVALID_ARG, "muse_group_set_synthetic_labels: NULL argument");
    if (g->nkeys > 4) return fail(MUSE_ERR_UNSUPPORTED, "synthetic labels for at most 4 keys");
    if (g->size == 0 || g->nkeys == 0) return MUSE_OK;
    int64_t d[4] = {1, 1, 1, 1}, m[4] = {1, 1, 1, 1};
    for (int k = 0; k < g->nkeys; k++) {
        if (div[k] < 1 || mod[k] < 1 || mod[k] > 0x7fffffffLL) return fail(MUSE_ERR_INVALID_ARG, "label divisor / modulus out of range");
        d[k] = div[k];
        m[k] = mod[k];
    }
    CU(cudaSetDevice(g->ctx->device));
    synth_labels_kernel<<<(unsigned)((g->size + 255) / 256), 256, 0, g->ctx->stream>>>(g->labels, g->cap, g->nkeys, 0, g->size,
                                                                                       g->global_offset, d[0], m[0], d[1], m[1],
                                                                                       d[2], m[2], d[3], m[3]);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(g->ctx->stream));
    for (int k = 0; k < g->nkeys; k++)      // an upper bound is all the group table needs
        g->max_id[k] = (int32_t)std::min<int64_t>(m[k] - 1, (g->global_offset + g->size - 1) / d[k]);
    return MUSE_OK;
}

extern "C" void muse_synth_row(uint64_t seed, int64_t index, int64_t series_len, double *out_row) {
    const SynthSeries sp = synth_params(seed, index, series_len);
    for (int64_t t = 0; t < series_len; t++) out_row[t] = synth_value(seed, index, sp, t);
}

extern "C" void muse_synth_reference(uint64_t seed, int64_t series_len, double *out_row) {
    for (int64_t t = 0; t < series_len; t++) out_row[t] = synth_ref_value(seed, series_len, t);
}

extern "C" int64_t muse_group_size(const muse_group *g) { return g ? g->size : 0; }
extern "C" int64_t muse_group_series_len(const muse_group *g) { return g ? g->N : 0; }

extern "C" int muse_group_set_global_offset(muse_group *g, int64_t first_global_index) {
    if (!g || first_global_index < 0) return fail(MUSE_ERR_INVALID_ARG, "muse_group_set_global_offset: bad argument");
    g->global_offset = first_global_index;
    return MUSE_OK;
}

extern "C" int muse_group_clear(muse_group *g) {
    if (!g) return fail(MUSE_ERR_INVALID_ARG, "group is NULL");
    CU(cudaSetDevice(g->ctx->device));
    CU(cudaStreamSynchronize(g->ctx->stream));
    g->size = 0;
    g->stats_upto = 0;
    for (int k = 0; k < MUSE_MAX_LABEL_KEYS; k++) g->max_id[k] = -1;
    return MUSE_OK;
}

extern "C" int muse_group_read_rows(muse_group *g, int64_t first, int64_t n_rows, double *out_rows) {
    if (!g || !out_rows || first < 0 || n_rows < 0 || first + n_rows > g->size) return fail(MUSE_ERR_INVALID_ARG, "muse_group_read_rows: bad argument");
    if (n_rows == 0) return MUSE_OK;
    CU(cudaSetDevice(g->ctx->device));
    CU(cudaMemcpy2DAsync(out_rows, sizeof(double) * (size_t)g->N, g->slab + (size_t)first * g->ld, sizeof(double) * (size_t)g->ld,
                         sizeof(double) * (size_t)g->N, (size_t)n_rows, cudaMemcpyDeviceToHost, g->ctx->stream));
    CU(cudaStreamSynchronize(g->ctx->stream));
    return MUSE_OK;
}

extern "C" int muse_group_read_row(muse_group *g, int64_t local_index, double *out_row) {
    if (!g || !out_row || local_index < 0 || local_index >= g->size) return fail(MUSE_ERR_INVALID_ARG, "muse_group_read_row: bad argument");
    CU(cudaSetDevice(g->ctx->device));
    CU(cudaMemcpyAsync(out_row, g->slab + (size_t)local_index * g->ld, sizeof(double) * (size_t)g->N, cudaMemcpyDeviceToHost,
                       g->ctx->stream));
    CU(cudaStreamSynchronize(g->ctx->stream));
    return MUSE_OK;
}

// muse_group_roll / muse_group_roll_device: argument errors, reported before any device work.
static int roll_check(const muse_group *g, int64_t first, int64_t n_rows, const double *samples, int64_t k, const char *fn) {
    if (!g) return fail(MUSE_ERR_INVALID_ARG, "%s: group is NULL", fn);
    if (k < 0 || k > g->N) return fail(MUSE_ERR_INVALID_ARG, "%s: k = %lld not in [0, %lld]", fn, (long long)k, (long long)g->N);
    if (first < 0 || n_rows < 0 || first > g->size || n_rows > g->size - first)
        return fail(MUSE_ERR_INVALID_ARG, "%s: rows [%lld, %lld + %lld) not in the store's %lld", fn, (long long)first, (long long)first,
                    (long long)n_rows, (long long)g->size);
    if (!samples && k > 0 && n_rows > 0) return fail(MUSE_ERR_INVALID_ARG, "%s: samples is NULL", fn);
    return MUSE_OK;
}

extern "C" int muse_group_roll_device(muse_group *g, int64_t first, int64_t n_rows, const double *d_samples, int64_t k) {
    int rc = roll_check(g, first, n_rows, d_samples, k, "muse_group_roll_device");
    if (rc != MUSE_OK || k == 0 || n_rows == 0) return rc;
    CU(cudaSetDevice(g->ctx->device));
    CU(launch_roll_rows(g->slab, g->ld, (int)g->N, first, n_rows, d_samples, (int)k, g->row_stat, g->ctx->sm_count, g->ctx->stream));
    CU(cudaStreamSynchronize(g->ctx->stream));
    return MUSE_OK;
}

// The new samples reach the device in chunks of whole rows through ctx->d_roll (one buffer: the copy of chunk c + 1 is queued
// behind the roll of chunk c on the same stream); page-locked samples are copied from where they are, pageable ones through the
// pinned staging ring.
extern "C" int muse_group_roll(muse_group *g, int64_t first, int64_t n_rows, const double *samples, int64_t k) {
    int rc = roll_check(g, first, n_rows, samples, k, "muse_group_roll");
    if (rc != MUSE_OK || k == 0 || n_rows == 0) return rc;
    const size_t row_bytes = sizeof(double) * (size_t)k;
    if (row_bytes > MUSE_STAGE_BYTES) return fail(MUSE_ERR_UNSUPPORTED, "muse_group_roll: %lld new samples per row exceed the %zu-byte staging buffer",
                                                  (long long)k, MUSE_STAGE_BYTES);
    muse_ctx *c = g->ctx;
    CU(cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    const int64_t rows_per_chunk = stage_rows_per_chunk(k);
    const int64_t want = k * std::min<int64_t>(n_rows, rows_per_chunk);
    if (c->d_roll.cap() < want) {
        CU(cudaStreamSynchronize(st));
        CU(c->d_roll.grow(want));
    }
    auto queue = [&](int64_t r0, int64_t nr, const double *src) {
        cudaError_t e = cudaMemcpyAsync(c->d_roll, src, (size_t)nr * row_bytes, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = launch_roll_rows(g->slab, g->ld, (int)g->N, first + r0, nr, c->d_roll, (int)k, g->row_stat, c->sm_count, st);
        return e;
    };
    cudaPointerAttributes attr;
    const bool pinned = cudaPointerGetAttributes(&attr, samples) == cudaSuccess &&
                        (attr.type == cudaMemoryTypeHost || attr.type == cudaMemoryTypeManaged);
    (void)cudaGetLastError();
    if (pinned) {
        for (int64_t r0 = 0; r0 < n_rows; r0 += rows_per_chunk)
            CU(queue(r0, std::min<int64_t>(rows_per_chunk, n_rows - r0), samples + (size_t)r0 * (size_t)k));
    } else {
        rc = stage_rows(c, samples, n_rows, k, queue);
        if (rc != MUSE_OK) return rc;
    }
    CU(cudaStreamSynchronize(st));
    return MUSE_OK;
}

static int refresh_row_stats(muse_group *g);

// Removal moves only as many rows as were removed below the new size m: the removed rows below m ("holes", ascending) take
// the kept rows at or above m ("fillers", ascending), the j-th hole the j-th filler.  Finding them is O(n_rows) on the host
// (the fillers are [m, size) minus the listed rows there).  The pairs reach the device in chunks of MUSE_MOVE_CHUNK through
// ctx->d_moves (one buffer: the copy of chunk c + 1 is queued behind the kernel of chunk c on the same stream).
#define MUSE_MOVE_CHUNK ((int64_t)1 << 20)
extern "C" int muse_group_remove(muse_group *g, const int64_t *rows, int64_t n_rows, int64_t *moved_from, int64_t *moved_to,
                                 int64_t *n_moved) {
    if (!g || !n_moved) return fail(MUSE_ERR_INVALID_ARG, "muse_group_remove: NULL argument");
    *n_moved = 0;
    if (n_rows < 0 || n_rows > g->size)
        return fail(MUSE_ERR_INVALID_ARG, "muse_group_remove: %lld rows of a store of %lld", (long long)n_rows, (long long)g->size);
    if (!rows && n_rows > 0) return fail(MUSE_ERR_INVALID_ARG, "muse_group_remove: rows is NULL");
    if (!moved_from != !moved_to) return fail(MUSE_ERR_INVALID_ARG, "muse_group_remove: one of moved_from / moved_to is NULL");
    for (int64_t i = 0; i < n_rows; i++)
        if (rows[i] < 0 || rows[i] >= g->size || (i > 0 && rows[i] <= rows[i - 1]))
            return fail(MUSE_ERR_INVALID_ARG, "muse_group_remove: rows[%lld] = %lld is outside [0, %lld), repeated or out of order",
                        (long long)i, (long long)rows[i], (long long)g->size);
    if (n_rows == 0) return MUSE_OK;
    const int64_t m = g->size - n_rows;
    const int64_t holes = std::lower_bound(rows, rows + n_rows, m) - rows;
    std::vector<int2> mv((size_t)holes);
    for (int64_t j = 0, k = holes, r = m; j < holes; r++) {
        if (k < n_rows && rows[k] == r) {
            k++;      // a removed row at or above m: not a filler
        } else {
            mv[(size_t)j] = make_int2((int)r, (int)rows[j]);
            j++;
        }
    }
    muse_ctx *c = g->ctx;
    CU(cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    int rc = refresh_row_stats(g);      // the moved rows carry their statistics: all of them must exist first
    if (rc) return rc;
    if (holes > 0) CU(c->d_moves.grow(MUSE_MOVE_CHUNK));
    for (int64_t c0 = 0; c0 < holes; c0 += MUSE_MOVE_CHUNK) {
        const int64_t nc = std::min<int64_t>(MUSE_MOVE_CHUNK, holes - c0);
        CU(cudaMemcpyAsync(c->d_moves, mv.data() + c0, sizeof(int2) * (size_t)nc, cudaMemcpyHostToDevice, st));
        CU(launch_move_rows(g->slab, g->ld, g->row_stat, g->labels, g->nkeys, g->cap, c->d_moves, nc, c->sm_count, st));
    }
    g->size = g->stats_upto = m;
    // max_id over the rows that remain, as a fresh store of them has it (group-key widths depend on it); the old values stay
    // if that fails: they are still upper bounds
    int32_t old[MUSE_MAX_LABEL_KEYS];
    memcpy(old, g->max_id, sizeof(old));
    for (int k = 0; k < MUSE_MAX_LABEL_KEYS; k++) g->max_id[k] = -1;
    rc = refresh_max_ids(g, 0, m);
    if (rc) {
        memcpy(g->max_id, old, sizeof(old));
        return rc;
    }
    CU(cudaStreamSynchronize(st));
    if (moved_from)
        for (int64_t j = 0; j < holes; j++) {
            moved_from[j] = mv[(size_t)j].x;
            moved_to[j] = mv[(size_t)j].y;
        }
    *n_moved = holes;
    return MUSE_OK;
}

// ------------------------------------------------------------------------------------
// batch
// ------------------------------------------------------------------------------------
static int64_t next_pow2(int64_t v) {   // == nextPowOf2 (xcorr.go:19-24) for 1 <= v < 2^29
    int64_t n = 1;
    while (n < v) n <<= 1;
    return n;
}

// fp32 tables of the screening kernel; leaves screen_ok = 0 when the shape has no screening kernel
// n = 128 .. 16384: kernels with the fused fp32 second stage (several series per warp up to 1024, one warp per series at 2048,
// one block per series above)
static int screen_is_fused(int log2m) { return log2m >= 6 && log2m <= 13; }
static int screen_is_big(int log2m) { return log2m >= 11 && log2m <= 13; }      // muse_screen_big.cuh

// The per-reference tables of the fp32 kernels, from Xt on the device: weights of the bound
// A[k] = |Xt[k]| * (1 at DC and Nyquist, else 2) rounded UP (the bound must not shrink), one 16-byte entry per
// mirror pair (k, M-k), k < M/2, with the split twiddle exp(-2*pi*i*k/n); the two reference coefficients of the
// second stage; and A[M/2], Xt[M/2] for the host (kernel parameters).
__device__ __forceinline__ void screen_tables_body(const cd *__restrict__ Xt, int M, const float2 *__restrict__ swtw, float4 *__restrict__ sw,
                                                   float4 *__restrict__ sx, float *__restrict__ sb, float *__restrict__ mid,
                                                   const int32_t *__restrict__ std_zero) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k > M / 2) return;
    if (k == 0) mid[0] = __int_as_float(*std_zero);      // the reference's std-zero flag rides along: one copy to the host
    const cd a = Xt[k], c = Xt[M - k];
    if (k == M / 2) {
        mid[1] = __double2float_ru(hypot(a.x, a.y) * 2.0);
        mid[2] = (float)a.x;
        mid[3] = (float)a.y;
        return;
    }
    const float wa = __double2float_ru(hypot(a.x, a.y) * (k == 0 ? 1.0 : 2.0));
    const float wc = __double2float_ru(hypot(c.x, c.y) * (k == 0 ? 1.0 : 2.0));     // k = 0: M - k is the Nyquist bin
    const float2 w = swtw[k];
    sw[k] = make_float4(w.x, w.y, wa, wc);
    sx[k] = make_float4((float)a.x, (float)a.y, (float)c.x, (float)c.y);
    sb[k] = __double2float_ru(sqrt(2.0 * ((double)wa * (double)wa + (double)wc * (double)wc)) * (1.0 + 1e-15));
}
__global__ void screen_tables_kernel(const cd *__restrict__ Xt, int M, const float2 *__restrict__ swtw, float4 *__restrict__ sw,
                                     float4 *__restrict__ sx, float *__restrict__ sb, float *__restrict__ mid,
                                     const int32_t *__restrict__ std_zero) {
    screen_tables_body(Xt, M, swtw, sw, sx, sb, mid, std_zero);
}

// Twiddle tables of FFT length n (they depend on n alone): filled when the scratch set was last used for another n.
static int ensure_ref_tables(muse_batch *b, int64_t ld) {
    const int64_t n = b->n, M = n / 2;
    cudaStream_t st = bstream(b);
    CU(b->d_ref.grow(ld));
    CU(b->d_mid.grow(4));
    const bool want_screen = screen_is_fused(b->log2m);
    if (b->tab_n == n && (b->tab_screen || !want_screen)) return MUSE_OK;
    b->tab_n = 0;
    b->tab_screen = 0;
    if (b->is_long) {      // the reference's transform has n entries, the twiddles are generated on the device
        CU(b->Xt.grow(n));
        CU(b->twM.grow(n));
        CU(launch_long_twiddles(b->twM, b->log2m + 1, st));
        b->tab_n = n;
        return MUSE_OK;
    }
    const long double PI2 = 6.283185307179586476925286766559005768L;
    const int log2p = exact_log2p(b->log2m);
    std::vector<cd> twM((size_t)M + 16);
    fill_pass_twiddles(b->log2m, log2p, twM.data(), [&](long long num, long long den) {
        return cd{(double)cosl(-PI2 * num / den), (double)sinl(-PI2 * num / den)};
    });
    // twiddle tables, correctly rounded from long double
    std::vector<cd> twn((size_t)(M / 2 + 1));
    for (int64_t k = 0; k <= M / 2; k++) twn[(size_t)k] = cd{(double)cosl(-PI2 * k / n), (double)sinl(-PI2 * k / n)};
    CU(b->Xt.grow(M + 1));
    CU(b->twM.grow((int64_t)twM.size()));
    CU(b->twn.grow(M / 2 + 1));
    CU(cudaMemcpyAsync(b->twM, twM.data(), sizeof(cd) * twM.size(), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(b->twn, twn.data(), sizeof(cd) * (size_t)(M / 2 + 1), cudaMemcpyHostToDevice, st));
    std::vector<cf> twp, twi;
    std::vector<float2> swtw;
    if (want_screen) {
        if (screen_is_big(b->log2m)) {
            twi.resize((size_t)10 * (M / 32) + 31 * (M / 1024) + 1024 + 31 * 32);      // ScreenBigCfg::TW_TOTAL
            fill_big_twiddles(b->log2m, twi.data(), [&](long long num, long long den) {
                return cf{(float)cosl(-PI2 * num / den), (float)sinl(-PI2 * num / den)};
            });
            CU(b->twi_f.grow((int64_t)twi.size()));
            CU(cudaMemcpyAsync(b->twi_f, twi.data(), sizeof(cf) * twi.size(), cudaMemcpyHostToDevice, st));
        }
        twp.resize((size_t)M + 64);
        fill_pass_twiddles(b->log2m, 5, twp.data(), [&](long long num, long long den) {      // radix-32 passes in every screening kernel
            return cf{(float)cosl(-PI2 * num / den), (float)sinl(-PI2 * num / den)};
        });
        swtw.resize((size_t)M / 2);
        for (int64_t k = 0; k < M / 2; k++) swtw[(size_t)k] = make_float2((float)cosl(-PI2 * k / n), (float)sinl(-PI2 * k / n));
        CU(b->twp_f.grow((int64_t)twp.size()));
        CU(b->swtw.grow((int64_t)swtw.size()));
        CU(b->sw_f.grow(M / 2));
        CU(b->sx_f.grow(M / 2));
        CU(b->sb_f.grow(M / 2));
        CU(cudaMemcpyAsync(b->twp_f, twp.data(), sizeof(cf) * twp.size(), cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(b->swtw, swtw.data(), sizeof(float2) * swtw.size(), cudaMemcpyHostToDevice, st));
    }
    CU(cudaStreamSynchronize(st));      // the host vectors go out of scope
    b->tab_n = n;
    b->tab_screen = want_screen ? 1 : 0;
    return MUSE_OK;
}

// NewBatch in two halves, so that the references of a multi-query launch share ONE round trip: queue = everything
// up to the copies of the std-zero flag and the middle-bin values into the batch's pinned mailbox; finish (after the
// stream has been synchronised) = the error of muse_batch.go:38-41 (the caller destroys the batch) or the by-value parameters.
// d_ref_row != NULL: the reference row is already on the device, zero-padded to the slab's row pitch (muse_multi_run
// uploads the references of a launch with one copy).
static int ensure_long_work(muse_batch *b, int64_t count);
static LongParams long_params(const muse_batch *b, const double *slab, int64_t count, const int32_t *idx, int signed_scores);

// The batch object with its pooled scratch, the tables of its FFT length and its small allocations: nothing is launched.
static int batch_alloc(muse_ctx *ctx, muse_group *g, int64_t ref_len, BatchPtr &out) {
    if (!ctx || !g) return fail(MUSE_ERR_INVALID_ARG, "muse_batch_create: NULL argument");
    if (g->ctx != ctx) return fail(MUSE_ERR_INVALID_ARG, "group belongs to another context");
    if (ref_len != g->N)   // muse_batch.go:24-28
        return fail(MUSE_ERR_LENGTH_MISMATCH, "comparison group series (length %lld) does not have the same length as the reference (%lld)",
                    (long long)g->N, (long long)ref_len);
    const int64_t n = next_pow2(ref_len);   // muse_batch.go:35
    if (n > MUSE_MAX_FFT_LEN) return fail(MUSE_ERR_UNSUPPORTED, "FFT length %lld > %d", (long long)n, MUSE_MAX_FFT_LEN);
    CU(cudaSetDevice(ctx->device));
    BatchPtr b(new muse_batch());
    b->is_long = n > MUSE_MAX_FUSED_FFT_LEN;
    b->ctx = ctx;
    b->g = g;
    b->N = ref_len;
    b->n = n;
    const int64_t M = n / 2;
    int l = 0;
    while ((1LL << l) < M) l++;
    b->log2m = l;
    {   // scratch of an earlier batch on this context, if there is one: a set whose tables were filled for this FFT
        // length is preferred, then the largest (it fits most stores)
        std::lock_guard<std::mutex> lk(ctx->mu);
        if (!ctx->pool.empty()) {
            size_t best = 0;
            auto better = [&](const RunScratch &x, const RunScratch &y) {
                if ((x.tab_n == n) != (y.tab_n == n)) return x.tab_n == n;
                return x.scratch_cap > y.scratch_cap;
            };
            for (size_t i = 1; i < ctx->pool.size(); i++)
                if (better(ctx->pool[i], ctx->pool[best])) best = i;
            static_cast<RunScratch &>(*b) = std::move(ctx->pool[best]);
            ctx->pool.erase(ctx->pool.begin() + (long)best);
        }
    }
    CU(b->ev.create());
    int rc = ensure_ref_tables(b.get(), g->ld);
    if (rc) return rc;
    CU(b->d_flag.grow(1));
    CU(b->d_counters.grow(1));
    CU(b->d_sel.grow(1));
    CU(b->d_cut.grow(1));
    CU(b->h_pin.grow(1));
    out = std::move(b);
    return MUSE_OK;
}

static int batch_create_queue(muse_ctx *ctx, muse_group *g, const double *ref, int64_t ref_len, BatchPtr &out,
                              const double *d_ref_row = nullptr) {
    if (!ref) return fail(MUSE_ERR_INVALID_ARG, "muse_batch_create: NULL argument");
    BatchPtr b;
    int rc = batch_alloc(ctx, g, ref_len, b);
    if (rc) return rc;
    cudaStream_t st = ctx->stream;
    const int64_t M = b->n / 2;
    if (!d_ref_row) {      // (the select state is cleared where it is used)
        CU(cudaMemsetAsync(b->d_ref, 0, sizeof(double) * (size_t)g->ld, st));
        CU(cudaMemcpyAsync(b->d_ref, ref, sizeof(double) * (size_t)ref_len, cudaMemcpyHostToDevice, st));
    }
    // X on the device through the same forward path the series take
    ExactParams p;
    memset(&p, 0, sizeof(p));
    p.slab = d_ref_row ? d_ref_row : b->d_ref;
    p.ld = g->ld;
    p.count = 1;
    p.N = (int)ref_len;
    p.twM = b->twM;
    p.twn = b->twn;
    p.out_X = b->Xt;
    p.out_flag = b->d_flag;
    if (b->is_long) {
        rc = ensure_long_work(b.get(), 1);
        if (rc) return rc;
        LongParams lp = long_params(b.get(), p.slab, 1, nullptr, 0);
        lp.out_X = b->Xt;
        CU(launch_long(MODE_REF, lp, b->d_long, b->long_pairs, st));
    } else {
        CU(launch_exact(MODE_REF, b->log2m, p, st));
    }
    b->screen_ok = 0;
    const bool screen = b->tab_screen != 0;
    if (screen) {
        screen_tables_kernel<<<(unsigned)((M / 2 + 1 + 255) / 256), 256, 0, st>>>(b->Xt, (int)M, b->swtw, b->sw_f, b->sx_f, b->sb_f, b->d_mid, b->d_flag);
        CU(cudaGetLastError());
    }
    // one round trip: the std-zero flag of the reference and the two middle-bin values the kernels take by value
    if (screen) CU(cudaMemcpyAsync(b->h_pin->mid, b->d_mid, sizeof(float) * 4, cudaMemcpyDeviceToHost, st));      // [0] carries the flag
    else CU(cudaMemcpyAsync(&b->h_pin->flag, b->d_flag, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    b->screen_ok = screen ? -1 : 0;      // -1: pending until batch_create_finish
    out = std::move(b);
    return MUSE_OK;
}

static int batch_create_finish(muse_batch *b) {
    const float *h_mid = b->h_pin->mid;
    int32_t flag = b->h_pin->flag;
    if (b->screen_ok == -1) memcpy(&flag, &h_mid[0], sizeof(flag));
    if (flag)   // muse_batch.go:38-41
        return fail(MUSE_ERR_STDDEV_ZERO, "Invalid input query, Standard deviation of zero");
    if (b->screen_ok == -1) {
        b->a_mid = h_mid[1];
        b->x_mid = cf{h_mid[2], h_mid[3]};
        b->screen_ok = 1;
    }
    return MUSE_OK;
}

extern "C" int muse_batch_create(muse_ctx *ctx, muse_group *g, const double *ref, int64_t ref_len, muse_batch **out) {
    BatchPtr b;
    int rc = batch_create_queue(ctx, g, ref, ref_len, b);
    if (rc) return rc;
    CU(cudaStreamSynchronize(ctx->stream));
    rc = batch_create_finish(b.get());
    if (rc) return rc;
    *out = b.release();
    return MUSE_OK;
}

extern "C" void muse_batch_destroy(muse_batch *b) {
    if (!b) return;
    cudaSetDevice(b->ctx->device);
    cudaStreamSynchronize(bstream(b));
    {   // the store-sized scratch goes back to the context (at most MUSE_SCRATCH_POOL sets are kept: a multi-query launch
        // group has 256 batches alive at once)
        std::lock_guard<std::mutex> lk(b->ctx->mu);
        if (b->ctx->pool.size() < MUSE_SCRATCH_POOL) b->ctx->pool.push_back(std::move(static_cast<RunScratch &>(*b)));
    }
    delete b;
}

extern "C" int64_t muse_batch_fft_len(const muse_batch *b) { return b ? b->n : 0; }

static int ensure_scratch(muse_batch *b) {
    const int64_t S = b->g->size;
    if (S <= b->scratch_cap) return MUSE_OK;
    const int64_t cap = std::max<int64_t>(S, 1024);
    b->scratch_cap = 0;      // until every array has grown: a failure part way leaves the next call to retry
    CU(b->d_score.grow(cap));
    CU(b->d_lag.grow(cap));
    CU(b->d_slot.grow(cap));
    CU(b->d_ckey.grow(cap));
    CU(b->d_skey.grow(cap));
    CU(b->d_cidx.grow(cap));
    CU(b->d_sidx.grow(cap));
    CU(b->d_clag.grow(cap));
    CU(b->d_slag.grow(cap));
    CU(b->d_U.grow(cap));
    CU(b->d_list.grow(cap));
    CU(b->d_rows.grow(cap));
    b->scratch_cap = cap;
    return MUSE_OK;
}

static int check_batch(muse_batch *b) {
    if (!b) return fail(MUSE_ERR_INVALID_ARG, "batch is NULL");
    if (b->g->N != b->N)
        return fail(MUSE_ERR_LENGTH_MISMATCH, "comparison group length %lld != reference length %lld", (long long)b->g->N, (long long)b->N);
    return MUSE_OK;
}

// n > MUSE_MAX_FUSED_FFT_LEN: the work buffer of launch_long, sized for `count` series or 256 MB worth of pairs
static int ensure_long_work(muse_batch *b, int64_t count) {
    const int log2n = b->log2m + 1;
    const size_t per_pair = long_work_bytes(log2n, 1);
    // both buffers of a chunk together: MUSE_LONG_WORK_MB (default 256)
    static const size_t work_mb = getenv("MUSE_LONG_WORK_MB") ? (size_t)std::max(1, atoi(getenv("MUSE_LONG_WORK_MB"))) : 256;
    long long pairs = std::max<long long>(1, (long long)((work_mb << 20) / per_pair));
    pairs = std::min<long long>(pairs, std::max<long long>(1, (count + 1) / 2));
    if (b->long_pairs >= pairs) return MUSE_OK;
    b->long_pairs = 0;
    CU(b->d_long.grow((int64_t)long_work_bytes(log2n, pairs)));
    b->long_pairs = pairs;
    return MUSE_OK;
}

static LongParams long_params(const muse_batch *b, const double *slab, int64_t count, const int32_t *idx, int signed_scores) {
    LongParams lp;
    memset(&lp, 0, sizeof(lp));
    lp.slab = slab;
    lp.ld = b->g->ld;
    lp.count = count;
    lp.idx = idx;
    lp.N = (int)b->N;
    lp.log2n = b->log2m + 1;
    lp.signed_scores = signed_scores;
    lp.X = b->Xt;
    lp.tw = b->twM;
    lp.out_score = b->d_score;
    lp.out_lag = b->d_lag;
    lp.out_flag = b->d_flag;
    return lp;
}

// All series of the store through the exact kernel -> d_score / d_lag.
static int score_exact_all(muse_batch *b, int signed_scores, const int32_t *idx, int64_t count,
                           const unsigned long long *d_count = nullptr) {
    ExactParams p;
    memset(&p, 0, sizeof(p));
    p.count_ptr = d_count;
    p.slab = b->g->slab;
    p.ld = b->g->ld;
    p.count = count;
    p.idx = idx;
    p.N = (int)b->N;
    p.signed_scores = signed_scores;
    p.Xt = b->Xt;
    p.twM = b->twM;
    p.twn = b->twn;
    p.out_score = b->d_score;
    p.out_lag = b->d_lag;
    if (count > 0 && b->is_long) {
        if (d_count) return fail(MUSE_ERR_UNSUPPORTED, "device-side list lengths do not exist above FFT length %d", MUSE_MAX_FUSED_FFT_LEN);
        int rc = ensure_long_work(b, count);
        if (rc) return rc;
        LongParams lp = long_params(b, b->g->slab, count, idx, signed_scores);
        CU(launch_long(MODE_SCORE, lp, b->d_long, b->long_pairs, bstream(b)));
        b->timing.n_launches++;
    } else if (count > 0) {
        CU(launch_exact(MODE_SCORE, b->log2m, p, bstream(b)));
        b->timing.n_launches++;
    }
    return MUSE_OK;
}

extern "C" int muse_batch_score_all(muse_batch *b, int32_t signed_scores, double *scores, int32_t *lags) {
    int rc = check_batch(b);
    if (rc) return rc;
    if (!scores || !lags) return fail(MUSE_ERR_INVALID_ARG, "muse_batch_score_all: NULL output");
    CU(cudaSetDevice(b->ctx->device));
    rc = ensure_scratch(b);
    if (rc) return rc;
    const int64_t S = b->g->size;
    rc = score_exact_all(b, signed_scores, nullptr, S);
    if (rc) return rc;
    CU(cudaMemcpyAsync(scores, b->d_score, sizeof(double) * (size_t)S, cudaMemcpyDeviceToHost, bstream(b)));
    CU(cudaMemcpyAsync(lags, b->d_lag, sizeof(int32_t) * (size_t)S, cudaMemcpyDeviceToHost, bstream(b)));
    CU(cudaStreamSynchronize(bstream(b)));
    return MUSE_OK;
}

extern "C" int muse_batch_xcorr(muse_batch *b, int64_t local_index, double *cc, int32_t *std_zero) {
    int rc = check_batch(b);
    if (rc) return rc;
    if (!cc || local_index < 0 || local_index >= b->g->size) return fail(MUSE_ERR_INVALID_ARG, "muse_batch_xcorr: bad argument");
    CU(cudaSetDevice(b->ctx->device));
    DevBuf<double> d_cc;
    CU(d_cc.grow(b->n));
    ExactParams p;
    memset(&p, 0, sizeof(p));
    p.slab = b->g->slab + (size_t)local_index * b->g->ld;
    p.ld = b->g->ld;
    p.count = 1;
    p.N = (int)b->N;
    p.Xt = b->Xt;
    p.twM = b->twM;
    p.twn = b->twn;
    p.out_score = d_cc;
    p.out_flag = b->d_flag;
    if (b->is_long) {
        rc = ensure_long_work(b, 1);
        if (rc) return rc;
        LongParams lp = long_params(b, p.slab, 1, nullptr, 0);
        lp.out_score = d_cc;
        CU(launch_long(MODE_CC, lp, b->d_long, b->long_pairs, bstream(b)));
    } else {
        CU(launch_exact(MODE_CC, b->log2m, p, bstream(b)));
    }
    int32_t flag = 0;
    CU(cudaMemcpyAsync(cc, d_cc, sizeof(double) * (size_t)b->n, cudaMemcpyDeviceToHost, bstream(b)));
    CU(cudaMemcpyAsync(&flag, b->d_flag, sizeof(flag), cudaMemcpyDeviceToHost, bstream(b)));
    CU(cudaStreamSynchronize(bstream(b)));
    if (std_zero) *std_zero = flag;
    return MUSE_OK;
}

// ------------------------------------------------------------------------------------
// Run: scores -> group max -> filter -> top-N
// ------------------------------------------------------------------------------------
struct RunArgs {
    const int32_t *key_cols;
    int32_t n_key_cols;
    int64_t max_lag, top_n;
    double threshold;
    int32_t sign_filter, mode, signed_scores;
    int32_t list_only;   // fused runs: the caller reads scores only through the exact list (no NaN fill of the score array)
    int32_t group_cut;   // grouped fused runs whose top-N is final here (one GPU): members below the top_n-th certain group need no exact score
    // The rows the run scores: rows[0 .. count), ascending store rows (a selection), or every row of the store (rows NULL,
    // count = size()).  Everything that depends on the size of the store -- the AUTO rule, launch bounds, what a fallback
    // scores -- uses count, so a filtered run takes the path a store of just its rows would take.
    const int32_t *rows;
    int64_t count;
    int32_t pre_launches;   // launches the caller queued since it recorded ev[0]; -1: the run records ev[0] itself
    int32_t prescreened;    // d_U and the cut-off state come from the tensor-core launch group: the fused run starts at its tail
};

// The arguments of a run over every row of g's store.
static RunArgs run_args(const muse_group *g, const int32_t *key_cols, int32_t n_key_cols, int64_t max_lag, int64_t top_n,
                        double threshold, int32_t sign_filter, int32_t mode, int32_t signed_scores) {
    RunArgs a{key_cols, n_key_cols, max_lag, top_n, threshold, sign_filter, mode, signed_scores};
    a.count = g->size;
    a.pre_launches = -1;
    return a;
}

// The checks of a run entry point's outputs (n_out, top_n records in scores, lags and series_idx) and group-by columns; fn
// names the entry point in the message.
static int check_run_outputs(const char *fn, const int64_t *n_out, int64_t top_n, const double *scores, const int64_t *lags,
                             const int64_t *series_idx, const int32_t *key_cols, int32_t n_key_cols) {
    if (!n_out || (top_n > 0 && (!scores || !lags || !series_idx))) return fail(MUSE_ERR_INVALID_ARG, "%s: NULL output", fn);
    if (n_key_cols < 0 || (n_key_cols > 0 && !key_cols)) return fail(MUSE_ERR_INVALID_ARG, "%s: bad key columns", fn);
    return MUSE_OK;
}

// The fp32 threshold of the screening passes: never above the fp64 threshold.
static float threshold_floor(double threshold) { return threshold > 0 ? (float)threshold * 0.999999f : 0.f; }

struct Rec {
    unsigned long long key;   // |score| bits
    int32_t idx;
    int32_t lagsgn;           // 2*lag + (score < 0)
    double score() const { return cand_score(key, lagsgn); }
    int32_t lag() const { return cand_lag(lagsgn); }
};

// Key bits per group-by column.  64 / ncols each when every column's cardinality fits: that packing does not depend on the
// store, so the shards of a multi-GPU run merge on it.  Otherwise ceil(log2(cardinality)) of THIS store's columns, which
// any number of keys up to MUSE_MAX_KEY_COLS can use as long as the widths sum to at most 64 bits.  A shard (shard = true)
// cannot: the shards merge on the keys, so they must not depend on the store.
static int key_bits(const muse_group *g, const int32_t *key_cols, int n_key_cols, int *bits, bool shard) {
    if (n_key_cols > MUSE_MAX_KEY_COLS) return fail(MUSE_ERR_UNSUPPORTED, "grouping by more than %d label keys", MUSE_MAX_KEY_COLS);
    const int fixed = 64 / n_key_cols;
    bool fits = true;
    int total = 0;
    for (int c = 0; c < n_key_cols; c++) {
        const int col = key_cols[c];
        if (col < 0 || col >= g->nkeys) return fail(MUSE_ERR_INVALID_ARG, "key column %d not in [0,%d)", col, g->nkeys);
        const int64_t card = (int64_t)g->max_id[col] + 2;      // ids -1 .. max_id -> values 0 .. max_id + 1
        int w = 1;
        while (w < 63 && (1LL << w) < card) w++;
        bits[c] = w;
        total += w;
        if (fixed < 64 && card > (1LL << fixed)) fits = false;
    }
    if (fits) {
        for (int c = 0; c < n_key_cols; c++) bits[c] = fixed;
        return MUSE_OK;
    }
    if (total > 64)
        return fail(MUSE_ERR_UNSUPPORTED, "the label cardinalities of the %d group-by keys need %d key bits (at most 64)", n_key_cols, total);
    if (shard)
        return fail(MUSE_ERR_UNSUPPORTED, "shards merge on group keys of at most %d bits per column (64 / %d keys)", fixed, n_key_cols);
    return MUSE_OK;
}

static int setup_group_table(muse_batch *b, const RunArgs &a, bool shard, KeyCols &kc, GroupTable &gt) {
    muse_group *g = b->g;
    int rc = key_bits(g, a.key_cols, a.n_key_cols, kc.bits, shard);
    if (rc) return rc;
    kc.ncols = a.n_key_cols;
    long double prod = 1;
    for (int c = 0; c < a.n_key_cols; c++) {
        const int col = a.key_cols[c];
        kc.col[c] = g->labels + (size_t)col * g->cap;
        const int64_t card = (int64_t)g->max_id[col] + 2;
        gt.radix[c] = card;
        prod *= (long double)card;
    }
    const int64_t S = g->size;
    const int64_t dense_limit = std::max<int64_t>(4 * S, 1 << 20);
    int64_t slots;
    if (prod <= (long double)dense_limit) {
        gt.dense = 1;
        slots = (int64_t)prod;
    } else {
        gt.dense = 0;
        slots = 1;
        while (slots < 2 * S) slots <<= 1;
    }
    CU(b->d_gmax.grow(slots));
    CU(b->d_hkeys.grow(slots));
    CU(b->d_gidx.grow(slots));
    gt.slots = slots;
    gt.gmax = b->d_gmax;
    gt.gidx = b->d_gidx;
    gt.hkeys = b->d_hkeys;
    cudaStream_t st = bstream(b);
    CU(cudaMemsetAsync(gt.gmax, 0, sizeof(unsigned long long) * (size_t)slots, st));
    CU(cudaMemsetAsync(gt.gidx, 0x7f, sizeof(int32_t) * (size_t)slots, st));
    if (!gt.dense) CU(cudaMemsetAsync(gt.hkeys, 0, sizeof(unsigned long long) * (size_t)slots, st));
    return MUSE_OK;
}

// Group max and representative of every series on its exact score (group_max_kernel, group_rep_kernel): d_slot and the
// group table `gt` hold them when the work queued on the stream has run.
static int queue_group_reps(muse_batch *b, const RunArgs &a, bool shard, KeyCols &kc, GroupTable &gt) {
    memset(&gt, 0, sizeof(gt));
    memset(&kc, 0, sizeof(kc));
    int rc = setup_group_table(b, a, shard, kc, gt);
    if (rc) return rc;
    const int64_t S = b->g->size;
    if (S > 0) {
        const unsigned blocks = (unsigned)((S + 255) / 256);
        group_max_kernel<<<blocks, 256, 0, bstream(b)>>>(gt, kc, b->d_score, S, b->d_slot);
        group_rep_kernel<<<blocks, 256, 0, bstream(b)>>>(gt, b->d_score, S, b->d_slot);
    }
    b->timing.n_launches += 2;
    return MUSE_OK;
}

// fused screened runs launch the exact kernel over at most this many listed series without knowing
// the list length on the host; run_fused_overflow finishes a longer list after the fact
#define MUSE_EXACT_UB 32768
static int run_fused_overflow(muse_batch *b, const RunArgs &a, int64_t n_exact, bool refill);

// The run's statistics from its counters (d_counters, read back to the host): a fused run's `listed` is its exact list and
// `refined` its refined count; any other run re-scores listed + refined (screened runs: pilot + second round).
static void settle_counters(muse_batch *b, const RunCounters &c) {
    if (b->fused_run) {
        b->timing.n_rescored = (int64_t)c.listed;
        b->timing.n_refined = (int64_t)c.refined;
    } else {
        b->timing.n_rescored = (int64_t)(c.listed + c.refined);
    }
}

// Produces the selected records on the host (unsorted).  apply_filter == 0 keeps every
// representative (grouped multi-GPU partials, SURVEY F2).
static int run_select(muse_batch *b, const RunArgs &a, int apply_filter, int64_t limit, std::vector<Rec> &recs) {
    muse_group *g = b->g;
    const int64_t S = g->size;
    cudaStream_t st = bstream(b);
    recs.clear();
    if (S == 0) return MUSE_OK;
    const unsigned blocks = (unsigned)((S + 255) / 256);
    GroupTable gt;
    memset(&gt, 0, sizeof(gt));
    const bool grouped = a.n_key_cols > 0;
    if (grouped) {
        KeyCols kc;
        int rc = queue_group_reps(b, a, false, kc, gt);
        if (rc) return rc;
    }
    CU(cudaMemsetAsync(b->d_counters, 0, sizeof(unsigned long long) * 2, st));      // cand, selected
    FilterArgs f{a.max_lag, a.threshold, a.sign_filter, apply_filter};
    Cand cand{b->d_ckey, b->d_cidx, b->d_clag, &b->d_counters->cand};
    emit_candidates_kernel<<<blocks, 256, 0, st>>>(gt, grouped ? b->d_slot.get() : nullptr, b->d_score, b->d_lag, S, f, cand);
    b->timing.n_launches++;
    CU(cudaGetLastError());
    // one round trip: the count and the first CH records together (pinned mailbox)
    const size_t CH = std::min<size_t>((size_t)S, MUSE_SELECT_CHUNK);
    const RunCounters &h_n = b->h_pin->counters;
    auto &h_cand = b->h_pin->cand;
    CU(cudaMemcpyAsync(&b->h_pin->counters, b->d_counters, sizeof(RunCounters), cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(h_cand.key, b->d_ckey, sizeof(unsigned long long) * CH, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(h_cand.idx, b->d_cidx, sizeof(int32_t) * CH, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(h_cand.lagsgn, b->d_clag, sizeof(int32_t) * CH, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    unsigned long long ncand = h_n.cand;
    settle_counters(b, h_n);
    if (b->fused_run == 1 && (int64_t)h_n.listed > std::min<int64_t>(a.count, MUSE_EXACT_UB)) {
        // rare: more exact candidates than the fixed launch covered -> finish them and select again
        const int64_t n_exact = (int64_t)h_n.listed;
        int rc = run_fused_overflow(b, a, n_exact, false);
        if (rc) return rc;
        b->fused_run = 0;
        rc = run_select(b, a, apply_filter, limit, recs);
        b->timing.n_rescored = n_exact;
        return rc;
    }
    if (ncand == 0) return MUSE_OK;
    auto better = [](const Rec &x, const Rec &y) { return key_precedes(x.key, x.idx, y.key, y.idx); };
    if (ncand <= CH) {
        recs.resize((size_t)ncand);
        for (size_t i = 0; i < (size_t)ncand; i++) recs[i] = Rec{h_cand.key[i], h_cand.idx[i], h_cand.lagsgn[i]};
    } else {
        const unsigned long long *src_key = b->d_ckey;
        const int32_t *src_idx = b->d_cidx, *src_lag = b->d_clag;
        unsigned long long nsel = ncand;
        if (limit >= 0 && ncand > (unsigned long long)limit && ncand > 262144ull) {
            // device radix select of the `limit` best by (|score| desc, index asc)
            if (limit == 0) return MUSE_OK;
            CU(cudaMemsetAsync(b->d_sel, 0, sizeof(SelectState), st));
            unsigned long long want = (unsigned long long)limit;
            CU(cudaMemcpyAsync(&b->d_sel.get()->want, &want, sizeof(want), cudaMemcpyHostToDevice, st));
            const unsigned sblocks = (unsigned)((ncand + 1023ull) / 1024ull);
            for (int r = 0; r < 6; r++) select_round_kernel<<<sblocks, 1024, 0, st>>>(b->d_sel, b->d_ckey, b->d_cidx, ncand, r);
            select_gather_kernel<<<sblocks, 1024, 0, st>>>(b->d_sel, b->d_ckey, b->d_cidx, ncand, b->d_clag, b->d_skey, b->d_sidx,
                                                           b->d_slag, &b->d_counters->selected);
            b->timing.n_launches += 7;
            CU(cudaGetLastError());
            CU(cudaMemcpyAsync(&nsel, &b->d_counters->selected, sizeof(nsel), cudaMemcpyDeviceToHost, st));
            CU(cudaStreamSynchronize(st));
            src_key = b->d_skey;
            src_idx = b->d_sidx;
            src_lag = b->d_slag;
        }
        std::vector<unsigned long long> hk((size_t)nsel);
        std::vector<int32_t> hi((size_t)nsel), hl((size_t)nsel);
        CU(cudaMemcpyAsync(hk.data(), src_key, sizeof(unsigned long long) * (size_t)nsel, cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(hi.data(), src_idx, sizeof(int32_t) * (size_t)nsel, cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(hl.data(), src_lag, sizeof(int32_t) * (size_t)nsel, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        recs.resize((size_t)nsel);
        for (size_t i = 0; i < (size_t)nsel; i++) recs[i] = Rec{hk[i], hi[i], hl[i]};
    }
    if (limit >= 0 && recs.size() > (size_t)limit) {
        std::nth_element(recs.begin(), recs.begin() + limit, recs.end(), better);
        recs.resize((size_t)limit);
    }
    std::sort(recs.begin(), recs.end(), better);
    return MUSE_OK;
}

static cudaError_t launch_screen(const muse_batch *b, const ScreenParams &p, cudaStream_t st) {
    if (b->log2m == 10) return launch_screen_warp(p, b->ctx->sm_count, st);
    if (screen_is_big(b->log2m)) return launch_screen_big(b->log2m, p, b->ctx->sm_count, st);
    static cudaError_t (*const sub[])(const ScreenParams &, int, cudaStream_t) = {launch_screen_sub<1>, launch_screen_sub<2>,
                                                                                 launch_screen_sub<3>, launch_screen_sub<4>};
    if (b->log2m >= 6 && b->log2m <= 9) return sub[b->log2m - 6](p, b->ctx->sm_count, st);
    return cudaErrorInvalidValue;
}

static int ensure_lower(muse_batch *b) {
    CU(b->d_L.grow(b->g->size));
    CU(b->d_W.grow(b->g->size));
    return MUSE_OK;
}

// Per-row statistics of the store (RowStat): the ingest paths queue them behind the copy that brings the rows in
// (queue_row_stats, synth_rows_kernel); this is the safety net for rows that arrived any other way.
static int refresh_row_stats(muse_group *g) {
    if (g->stats_upto < g->size) {
        int rc = queue_row_stats(g, g->stats_upto, g->size - g->stats_upto);
        if (rc) return rc;
        g->stats_upto = g->size;
    }
    return MUSE_OK;
}

// The screening parameters of b over the store rows rows[0 .. count) (rows NULL: the first count rows).
static ScreenParams screen_params(muse_batch *b, const int32_t *rows, int64_t count) {
    ScreenParams sp;
    memset(&sp, 0, sizeof(sp));
    sp.slab = b->g->slab;
    sp.ld = b->g->ld;
    sp.count = count;
    sp.rows = rows;
    sp.N = (int)b->N;
    sp.twp = b->twp_f;
    sp.sw = b->sw_f;
    sp.a_mid = b->a_mid;
    sp.out_U = b->d_U;
    sp.sx = b->sx_f;
    sp.sb = b->sb_f;
    sp.twi = b->twi_f;
    sp.x_mid = b->x_mid;
    sp.row_stat = b->g->row_stat;
    sp.cut_bits = &b->d_cut->bits;
    sp.n_refined = &b->d_cut->refined;
    sp.next_claim = &b->d_cut->claims;
    sp.cut_hist = b->d_cut->hist;
    sp.top_n = 1;
    return sp;
}

// Arms the fused refinement of the warp kernel: running cut-off = cut0 (+inf: bounds only),
// counters (series claims, n_refined) and histogram cleared, lag window in the kernel's rotated cc index.
#define MUSE_INIT_CUT_BLOCKS ((MUSE_CUT_WORDS + 255) / 256)
__device__ __forceinline__ void init_cut_body(CutState *state, float cut0) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) {
        state->bits = __float_as_uint(cut0);
        state->claims = 0u;
        state->refined = 0ull;
    }
    if (i < MUSE_CUT_WORDS) state->hist[i] = 0u;
}
__global__ void init_cut_kernel(CutState *state, float cut0) { init_cut_body(state, cut0); }

// the same for the queries of a multi-query launch: blockIdx.y = query
__global__ void init_cut_batch_kernel(CutState *const *__restrict__ states, float cut0) { init_cut_body(states[blockIdx.y], cut0); }

// skip_init: the cut-off state is armed by init_cut_batch_kernel for all the queries of a launch at once
static int arm_refinement(muse_batch *b, ScreenParams &sp, float cut0, int64_t max_lag, int64_t top_n, double threshold, bool skip_init = false) {
    if (!screen_is_fused(b->log2m)) return MUSE_OK;
    int rc = refresh_row_stats(b->g);
    if (rc) return rc;
    sp.row_stat = b->g->row_stat;
    if (!skip_init) {
        init_cut_kernel<<<MUSE_INIT_CUT_BLOCKS, 256, 0, bstream(b)>>>(b->d_cut, cut0);
        CU(cudaGetLastError());
    }
    const int64_t n = b->n, pad = n - b->N;
    if (max_lag < 0) max_lag = -1;                          // nothing passes |lag| <= max_lag
    if (2 * max_lag >= n - 1) {                             // every lag is inside
        sp.win_lo = 0;
        sp.win_len = (int)n;
    } else {
        sp.win_lo = (int)(((pad - max_lag) % n + n) % n);
        sp.win_len = (int)(2 * max_lag);                    // -2 when max_lag < 0: no index qualifies
    }
    sp.top_n = (int)std::min<int64_t>(std::max<int64_t>(top_n, 1), 0x7fffffff);
    float thr = (float)threshold;
    if ((double)thr < threshold) thr = nextafterf(thr, INFINITY);    // round UP: a counted lower bound must really reach the threshold
    sp.thr = thr > 0.f ? thr : 0.f;
    return MUSE_OK;
}

// idx list of every series whose (refined) bound reaches the final cut-off, read from device memory, into n->listed (the
// refined count rides along).  rows: bound i belongs to the store's row rows[i] (a selection), which goes into the list;
// NULL: row i
__device__ __forceinline__ void survivors_cut_body(const float *__restrict__ U, int64_t S, const CutState *__restrict__ cut,
                                                   int32_t *__restrict__ out, RunCounters *n, const int32_t *__restrict__ rows) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) n->refined = cut->refined;
    const float lo = __uint_as_float(cut->bits);
    warp_append(&n->listed, i < S && U[i] >= lo, [&](unsigned long long pos) { out[pos] = rows ? rows[i] : (int32_t)i; });
}
__global__ void survivors_cut_kernel(const float *__restrict__ U, int64_t S, const CutState *__restrict__ cut,
                                     int32_t *__restrict__ out, RunCounters *n) {
    survivors_cut_body(U, S, cut, out, n, nullptr);
}

// the batched tails of muse_multi_run: blockIdx.y = query (MultiTail, muse_select.cuh)
__global__ void tail_reset_kernel(const MultiTail *__restrict__ tails, int nq) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q < nq) *tails[q].counters = RunCounters{0ull, 0ull, 0ull, 0ull};
}
__global__ void survivors_cut_batch_kernel(const MultiTail *__restrict__ tails, int64_t S, const int32_t *__restrict__ rows) {
    const MultiTail t = tails[blockIdx.y];
    survivors_cut_body(t.U, S, t.cut, t.list, t.counters, rows);
}
// reference preparation of a launch's queries: screen_tables_kernel with blockIdx.y = query; the 4 floats of every query
// (std-zero flag, A[M/2], Xt[M/2]) land in ONE array for one copy to the host
struct TablesArgs {
    const cd *Xt;
    float4 *sw, *sx;
    const int32_t *std_zero;
    float *sb;
};
__global__ void screen_tables_batch_kernel(const TablesArgs *__restrict__ args, int M, const float2 *__restrict__ swtw, float *__restrict__ mids) {
    const TablesArgs a = args[blockIdx.y];
    screen_tables_body(a.Xt, M, swtw, a.sw, a.sx, a.sb, mids + 4 * blockIdx.y, a.std_zero);
}

extern "C" int muse_batch_screen_bounds(muse_batch *b, int32_t refine, int64_t max_lag, float *upper, float *lower) {
    int rc = check_batch(b);
    if (rc) return rc;
    if (!upper || (refine && !lower)) return fail(MUSE_ERR_INVALID_ARG, "muse_batch_screen_bounds: NULL output");
    if (!b->screen_ok) return fail(MUSE_ERR_UNSUPPORTED, "no screening kernel for series length %lld", (long long)b->N);
    if (refine && !screen_is_fused(b->log2m)) return fail(MUSE_ERR_UNSUPPORTED, "the fused refinement needs an FFT length of 128 .. 16384");
    CU(cudaSetDevice(b->ctx->device));
    rc = ensure_scratch(b);
    if (rc) return rc;
    const int64_t S = b->g->size;
    if (S == 0) return MUSE_OK;
    cudaStream_t st = bstream(b);
    ScreenParams sp = screen_params(b, nullptr, S);
    if (refine) {
        rc = ensure_lower(b);
        if (rc) return rc;
        sp.out_L = b->d_L;
    }
    // refine: cut-off 0 that never rises (top_n = INT_MAX): every series takes the second stage
    rc = arm_refinement(b, sp, refine ? 0.f : INFINITY, max_lag, 0x7fffffff, 0.0);
    if (rc) return rc;
    CU(launch_screen(b, sp, st));
    CU(cudaMemcpyAsync(upper, b->d_U, sizeof(float) * (size_t)S, cudaMemcpyDeviceToHost, st));
    if (refine) CU(cudaMemcpyAsync(lower, b->d_L, sizeof(float) * (size_t)S, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return MUSE_OK;
}

// Screened scoring with the fused kernel (n = 2048, ungrouped): ONE pass over the slab gives
// every series an upper bound that is either the loose spectral one (below the running cut-off:
// cannot be in the result) or the tight fp32 one; the exact fp64 kernel then scores only the
// series whose bound reaches the final cut-off.  No host round trip before the final one: the
// cut-off and the list length stay on the device, the exact kernel is launched over
// MUSE_EXACT_UB series and skips what the list does not hold.
static int score_fused(muse_batch *b, const RunArgs &a) {
    const int64_t S = b->g->size;
    cudaStream_t st = bstream(b);
    if (!a.prescreened) {      // prescreened (muse_multi_run): the bounds and cut-off came out of the tensor-core launch group
        ScreenParams sp = screen_params(b, a.rows, a.count);
        int rc = arm_refinement(b, sp, threshold_floor(a.threshold), a.max_lag, a.top_n, a.threshold);
        if (rc) return rc;
        CU(launch_screen(b, sp, st));
        b->timing.n_launches += 2;
    }
    CU(cudaEventRecord(b->ev[1], st));
    if (!a.list_only) CU(cudaMemsetAsync(b->d_score, 0xff, sizeof(double) * (size_t)S, st));      // NaN = "cannot be in the result"
    const unsigned blocks = (unsigned)((S + 255) / 256);
    survivors_cut_kernel<<<blocks, 256, 0, st>>>(b->d_U, S, b->d_cut, b->d_list, b->d_counters);
    b->timing.n_launches++;
    return score_exact_all(b, a.signed_scores, b->d_list, std::min<int64_t>(a.count, MUSE_EXACT_UB), &b->d_counters->listed);
}

// Grouped runs on the fused kernels: every series takes the fp32 second stage (bounds on the score
// itself, window ignored), a group's best LOWER bound prunes its members, and only the members whose
// upper bound reaches it -- the representative and whatever ties it within the fp32 slack -- are
// scored in fp64.  The group max / representative / filter / top-N then run on those exact scores
// exactly as in an all-exact run (every other member is provably below its group's representative).
static int score_fused_grouped(muse_batch *b, const RunArgs &a) {
    const int64_t S = b->g->size;
    cudaStream_t st = bstream(b);
    ScreenParams sp = screen_params(b, a.rows, a.count);
    int rc = ensure_lower(b);
    if (rc) return rc;
    sp.out_L = b->d_L;
    sp.grouped = 1;
    // a member below the threshold cannot be the representative of a group that passes results.go:46-52
    const float thr_lo = threshold_floor(a.threshold);
    rc = arm_refinement(b, sp, thr_lo, a.max_lag, 0x7fffffff, 0.0);      // a cut-off that never rises
    if (rc) return rc;
    GroupTable gt;
    memset(&gt, 0, sizeof(gt));
    KeyCols kc;
    memset(&kc, 0, sizeof(kc));
    rc = setup_group_table(b, a, false, kc, gt);
    if (rc) return rc;
    const unsigned blocks = (unsigned)((S + 255) / 256);
    const bool running = screen_is_big(b->log2m);      // the kernel itself keeps each group's best lower bound
    if (running) {
        group_slots_kernel<<<blocks, 256, 0, st>>>(gt, kc, S, b->d_slot);
        sp.slot_of = b->d_slot;
        sp.group_L = gt.gmax;
        sp.out_W = b->d_W;
        b->timing.n_launches++;
    }
    CU(launch_screen(b, sp, st));
    b->timing.n_launches += 2;
    CU(cudaEventRecord(b->ev[1], st));
    CU(cudaMemsetAsync(b->d_score, 0xff, sizeof(double) * (size_t)S, st));      // NaN = "not its group's representative"
    if (!running) {
        group_lower_bound_kernel<<<blocks, 256, 0, st>>>(gt, kc, b->d_L, S, b->d_slot);
        b->timing.n_launches++;
    }
    const unsigned *cut_bits = nullptr;
    if (running && a.group_cut && a.top_n > 0 && a.top_n < 0x7fffffff) {
        group_uncertain_kernel<<<blocks, 256, 0, st>>>(gt, b->d_U, b->d_W, S, b->d_slot);
        group_cut_count_kernel<<<(unsigned)((gt.slots + 255) / 256), 256, 0, st>>>(gt, a.threshold, b->d_cut->hist);
        group_cut_find_kernel<<<1, 32, 0, st>>>(b->d_cut->hist, (int)a.top_n, &b->d_cut->bits);
        b->timing.n_launches += 3;
        cut_bits = &b->d_cut->bits;
    }
    group_contenders_kernel<<<blocks, 256, 0, st>>>(gt, b->d_U, S, b->d_slot, thr_lo, b->d_list, &b->d_counters->listed, cut_bits);
    b->timing.n_launches++;
    CU(cudaGetLastError());
    unsigned long long *h_listed = &b->h_pin->counters.listed;
    CU(cudaMemcpyAsync(h_listed, &b->d_counters->listed, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));                                 // one small round trip: the list length sizes the launch
    const int64_t n_exact = (int64_t)*h_listed;
    rc = score_exact_all(b, a.signed_scores, b->d_list, n_exact);
    if (rc) return rc;
    CU(cudaMemcpyAsync(&b->d_counters->refined, &b->d_cut->refined, sizeof(unsigned long long), cudaMemcpyDeviceToDevice, st));
    return MUSE_OK;
}

// The exact list was longer than the launch bound: score the rest now that its length is known.
// refill: the run skipped the NaN fill of the score array (list_only) and the caller is about to
// read it as a whole -- fill it and score the complete list again.
static int run_fused_overflow(muse_batch *b, const RunArgs &a, int64_t n_exact, bool refill) {
    const int64_t S = b->g->size;
    if (refill) {
        CU(cudaMemsetAsync(b->d_score, 0xff, sizeof(double) * (size_t)S, bstream(b)));
        return score_exact_all(b, a.signed_scores, b->d_list, n_exact);
    }
    if (n_exact <= std::min<int64_t>(a.count, MUSE_EXACT_UB)) return MUSE_OK;
    return score_exact_all(b, a.signed_scores, b->d_list + MUSE_EXACT_UB, n_exact - MUSE_EXACT_UB);
}

// The scores of a run (its scratch grown: ensure_scratch) queued on the stream.
static int run_scores(muse_batch *b, const RunArgs &a) {
    int rc;
    memset(&b->timing, 0, sizeof(b->timing));
    b->fused_run = 0;
    b->timing_pending = 0;
    cudaStream_t st = bstream(b);
    if (a.pre_launches >= 0) b->timing.n_launches = a.pre_launches;      // the run began with the caller's work (ev[0] recorded)
    else CU(cudaEventRecord(b->ev[0], st));
    CU(cudaMemsetAsync(b->d_counters, 0, sizeof(RunCounters), st));
    // screening needs: a kernel for this FFT size, an ungrouped unsigned run, a sign filter that
    // unsigned scores can pass, and a store big enough to be worth two extra round trips
    // grouped runs are screened only by the fused kernels (the bound of a member says nothing about the
    // lag of its group's representative; the fused second stage bounds every member's score tightly)
    // signed scores (Muse.Run, muse.go:72-76): the bounds are bounds on |score|, which is what the filter's threshold and the
    // top-N rank by; the survivors are re-scored signed.  A sign filter on signed scores needs the sign, which no bound has.
    const bool can_screen = b->screen_ok && (a.n_key_cols == 0 || screen_is_fused(b->log2m)) &&
                            (a.signed_scores ? a.sign_filter == MUSE_SIGN_ANY : a.sign_filter != MUSE_SIGN_NEG);
    bool screen = can_screen && (a.mode == MUSE_MODE_SCREEN || (a.mode == MUSE_MODE_AUTO && a.count >= 16384));
    if (screen && a.n_key_cols > 0) {
        b->timing.mode = MUSE_MODE_SCREEN;
        b->fused_run = 2;          // statistics as a fused run; its exact list is already complete
        rc = score_fused_grouped(b, a);
        if (rc) return rc;
        CU(cudaEventRecord(b->ev[2], st));
        return MUSE_OK;
    }
    if (screen) {
        b->timing.mode = MUSE_MODE_SCREEN;
        b->fused_run = 1;
        rc = score_fused(b, a);
        if (rc) return rc;
        CU(cudaEventRecord(b->ev[2], st));
        return MUSE_OK;
    }
    b->timing.mode = MUSE_MODE_EXACT;
    rc = score_exact_all(b, a.signed_scores, a.rows, a.count);
    if (rc) return rc;
    CU(cudaEventRecord(b->ev[1], st));
    CU(cudaEventRecord(b->ev[2], st));
    return MUSE_OK;
}

// Elapsed times between the run's events; a failed query of an event must not stay behind as the runtime's last error.
static void read_timing_events(muse_batch *b) {
    float *out[4] = {&b->timing.total_ms, &b->timing.score_ms, &b->timing.rescore_ms, &b->timing.select_ms};
    const int from[4] = {0, 0, 1, 2}, to[4] = {3, 1, 2, 3};
    for (int i = 0; i < 4; i++)
        if (cudaEventElapsedTime(out[i], b->ev[from[i]], b->ev[to[i]]) != cudaSuccess) {
            (void)cudaGetLastError();
            *out[i] = 0.f;
        }
}

static int finish_timing(muse_batch *b) {
    cudaStream_t st = bstream(b);
    CU(cudaEventRecord(b->ev[3], st));
    CU(cudaEventSynchronize(b->ev[3]));
    read_timing_events(b);
    return MUSE_OK;
}

// A run queued without a final synchronisation (timing_pending): its times and counters once its end-of-run event is complete.
static int finish_pending_timing(muse_batch *b) {
    CU(cudaEventSynchronize(b->ev[3]));
    read_timing_events(b);
    settle_counters(b, b->h_pin->counters);
    b->timing_pending = 0;
    return MUSE_OK;
}

// The records of a padded list up to its first padding record (flags != 0), at most top_n, into the caller's arrays: their count.
static int64_t records_out(const muse_partial *r, int64_t top_n, double *scores, int64_t *lags, int64_t *series_idx) {
    int64_t k = 0;
    for (; k < top_n && r[k].flags == 0; k++) {
        scores[k] = r[k].score;
        lags[k] = r[k].lag;
        series_idx[k] = r[k].series_idx;
    }
    return k;
}

// The same for the host path's sorted records, whose series indices are local to the store.
static int64_t records_out(const muse_batch *b, const std::vector<Rec> &recs, double *scores, int64_t *lags, int64_t *series_idx) {
    for (size_t i = 0; i < recs.size(); i++) {
        scores[i] = recs[i].score();
        lags[i] = recs[i].lag();
        series_idx[i] = b->g->global_offset + recs[i].idx;
    }
    return (int64_t)recs.size();
}

static int queue_topn_records(muse_batch *b, const RunArgs &a, muse_partial *d_out, int64_t capacity);

// Ungrouped runs with a device-side top-N, in two halves: queue = scores, filter, rank, copy of the top_n records into
// the batch's pinned mailbox; finish (after the stream has been synchronised) = read the mailbox, or -- when the
// candidate list was too long for the device-side select, or the fused path's exact launch did not cover its list --
// finish on the host path from the scores already on the device.
static bool device_topn_applies(const muse_batch *b, const RunArgs &a) {
    // a filtered run: as on a store of its rows, whose scratch holds max(rows, 1024) entries (ensure_scratch)
    const int64_t cap = a.rows ? std::max<int64_t>(a.count, 1024) : b->scratch_cap;
    return a.n_key_cols == 0 && a.count > 0 && device_topn_fits(a.top_n, cap);
}

static int device_topn_queue(muse_batch *b, const RunArgs &a) {
    muse_partial *d_rec = reinterpret_cast<muse_partial *>(b->d_skey.get());      // free scratch in this path
    int rc = queue_topn_records(b, a, d_rec, a.top_n);
    if (rc) return rc;
    cudaStream_t st = bstream(b);
    CU(cudaMemcpyAsync(b->h_pin->recs, d_rec, sizeof(muse_partial) * (size_t)a.top_n, cudaMemcpyDeviceToHost, st));
    CU(cudaEventRecord(b->ev[3], st));
    return MUSE_OK;
}

static int device_topn_finish(muse_batch *b, const RunArgs &a, double *scores, int64_t *lags, int64_t *series_idx, int64_t *n_out) {
    const int64_t top_n = a.top_n;
    const muse_partial *h_rec = b->h_pin->recs;
    if (h_rec[0].flags != 2) {
        *n_out = records_out(h_rec, top_n, scores, lags, series_idx);
        return finish_pending_timing(b);
    }
    b->timing_pending = 0;
    int rc;
    if (b->fused_run == 1) {
        rc = run_fused_overflow(b, a, (int64_t)b->h_pin->counters.listed, true);
        if (rc) return rc;
        b->fused_run = 0;
    }
    std::vector<Rec> recs;
    rc = run_select(b, a, 1, top_n, recs);
    if (rc) return rc;
    *n_out = records_out(b, recs, scores, lags, series_idx);
    return finish_timing(b);
}

// The run of b that `a` describes (the device set, the scratch grown: ensure_scratch): its records into the caller's arrays.
static int batch_run(muse_batch *b, const RunArgs &a, double *scores, int64_t *lags, int64_t *series_idx, int64_t *n_out) {
    int rc;
    if (device_topn_applies(b, a)) {
        // ungrouped: filter and top-N on the device, ONE copy of top_n records to the host
        rc = device_topn_queue(b, a);
        if (rc) return rc;
        CU(cudaStreamSynchronize(bstream(b)));
        return device_topn_finish(b, a, scores, lags, series_idx, n_out);
    }
    rc = run_scores(b, a);
    if (rc) return rc;
    std::vector<Rec> recs;
    rc = run_select(b, a, 1, a.top_n, recs);
    if (rc) return rc;
    *n_out = records_out(b, recs, scores, lags, series_idx);
    return finish_timing(b);
}

extern "C" int muse_batch_run_ex(muse_batch *b, const int32_t *key_cols, int32_t n_key_cols, int64_t max_lag, int64_t top_n,
                                 double threshold, int32_t sign_filter, int32_t mode, int32_t signed_scores, double *scores,
                                 int64_t *lags, int64_t *series_idx, int64_t *n_out) {
    int rc = check_batch(b);
    if (rc) return rc;
    rc = check_run_outputs("muse_batch_run", n_out, top_n, scores, lags, series_idx, key_cols, n_key_cols);
    if (rc) return rc;
    if (top_n < 0) top_n = 0;
    CU(cudaSetDevice(b->ctx->device));
    RunArgs a = run_args(b->g, key_cols, n_key_cols, max_lag, top_n, threshold, sign_filter, mode, signed_scores);
    a.group_cut = 1;
    *n_out = 0;
    rc = ensure_scratch(b);
    if (rc) return rc;
    return batch_run(b, a, scores, lags, series_idx, n_out);
}

extern "C" int muse_batch_run(muse_batch *b, const int32_t *key_cols, int32_t n_key_cols, int64_t max_lag, int64_t top_n,
                              double threshold, int32_t sign_filter, double *scores, int64_t *lags, int64_t *series_idx,
                              int64_t *n_out) {
    return muse_batch_run_ex(b, key_cols, n_key_cols, max_lag, top_n, threshold, sign_filter, MUSE_MODE_AUTO, 0, scores, lags,
                             series_idx, n_out);
}

// ------------------------------------------------------------------------------------
// Filtered runs: Batch.Run over the series whose label ids match (Group.FilterByLabelValues, group.go:60-71)
// ------------------------------------------------------------------------------------
#define MUSE_WHERE_MAX 16        // equalities of one predicate
#define MUSE_WHERE_TILE 1024     // rows per block of the selection kernels: 256 threads x 4 rows
struct WherePred {
    const int32_t *col[MUSE_WHERE_MAX];   // label-id column of each equality
    int32_t id[MUSE_WHERE_MAX];
    int n;
};
__device__ __forceinline__ bool where_match(const WherePred &p, int64_t i) {
    for (int j = 0; j < p.n; j++)
        if (p.col[j][i] != p.id[j]) return false;
    return true;
}

// 1. matching rows per tile of MUSE_WHERE_TILE rows
__global__ void __launch_bounds__(256) where_count_kernel(WherePred p, int64_t S, int32_t *__restrict__ block_count) {
    __shared__ int wsum[8];
    const int64_t base = (int64_t)blockIdx.x * MUSE_WHERE_TILE;
    int c = 0;
#pragma unroll
    for (int k = 0; k < MUSE_WHERE_TILE / 256; k++) {
        const int64_t i = base + k * 256 + threadIdx.x;
        c += (i < S && where_match(p, i)) ? 1 : 0;
    }
    c = __reduce_add_sync(0xffffffffu, c);
    if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        int total = 0;
        for (int w = 0; w < 8; w++) total += wsum[w];
        block_count[blockIdx.x] = total;
    }
}

// 2. one block: exclusive scan of the nb tile counts in place, the selection's length into off[nb]
__global__ void __launch_bounds__(1024) where_scan_kernel(int32_t *__restrict__ off, int64_t nb) {
    __shared__ int wsum[32];
    __shared__ int carry;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int64_t base = 0; base < nb; base += 1024) {
        const int64_t i = base + threadIdx.x;
        const int v = i < nb ? off[i] : 0;
        int x = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, x, d);
            if (lane >= d) x += y;
        }
        if (lane == 31) wsum[w] = x;
        __syncthreads();
        if (w == 0) {
            int s = wsum[lane];
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int y = __shfl_up_sync(0xffffffffu, s, d);
                if (lane >= d) s += y;
            }
            wsum[lane] = s;
        }
        __syncthreads();
        const int excl = carry + (w > 0 ? wsum[w - 1] : 0) + x - v;
        if (i < nb) off[i] = excl;
        __syncthreads();                    // every thread has read carry
        if (threadIdx.x == 1023) carry = excl + v;
        __syncthreads();
    }
    if (threadIdx.x == 0) off[nb] = carry;
}

// 3. the matching rows of each tile at the tile's offset, in ascending order (the same list on every run)
__global__ void __launch_bounds__(256) where_write_kernel(WherePred p, int64_t S, const int32_t *__restrict__ off, int32_t *__restrict__ rows) {
    __shared__ int wsum[8];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t base = (int64_t)blockIdx.x * MUSE_WHERE_TILE;
    int out = off[blockIdx.x];
#pragma unroll
    for (int k = 0; k < MUSE_WHERE_TILE / 256; k++) {
        const int64_t i = base + k * 256 + threadIdx.x;
        const bool m = i < S && where_match(p, i);
        const unsigned ball = __ballot_sync(0xffffffffu, m);
        if (lane == 0) wsum[w] = __popc(ball);
        __syncthreads();
        int before = 0, total = 0;
        for (int v = 0; v < 8; v++) {
            before += v < w ? wsum[v] : 0;
            total += wsum[v];
        }
        if (m) rows[out + before + __popc(ball & ((1u << lane) - 1u))] = (int32_t)i;
        out += total;
        __syncthreads();                    // wsum is rewritten by the next slice
    }
}

// Rows outside the selection get the values that already mean "cannot be in the result" to the per-series kernels that
// walk the whole store (survivors_cut, group_*, emit_candidates): score NaN (group max / rep and the candidates skip it),
// upper bound -1 (never a survivor or contender, never marks its group uncertain) and lower bound -1 (never a group's
// bound).  The pass over the selection then overwrites its own rows.
__global__ void where_neutral_kernel(double *__restrict__ score, float *__restrict__ U, float *__restrict__ L, int64_t S) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= S) return;
    score[i] = __longlong_as_double(-1ll);      // all bits set: a NaN, what the NaN fills of the other paths write
    U[i] = -1.f;
    L[i] = -1.f;
}

// The predicate where_cols[j] == where_ids[j] (j < n_where) on the label columns of g, after the argument checks of a
// filtered run (fn names the entry point in the message).
static int where_pred(const muse_group *g, const int32_t *where_cols, const int32_t *where_ids, int32_t n_where, const char *fn,
                      WherePred &p) {
    if (n_where < 0 || n_where > MUSE_WHERE_MAX)
        return fail(MUSE_ERR_INVALID_ARG, "%s: %d where columns (0 .. %d)", fn, (int)n_where, MUSE_WHERE_MAX);
    if (n_where > 0 && (!where_cols || !where_ids)) return fail(MUSE_ERR_INVALID_ARG, "%s: NULL where arrays", fn);
    memset(&p, 0, sizeof(p));
    p.n = n_where;
    for (int j = 0; j < n_where; j++) {
        if (where_cols[j] < 0 || where_cols[j] >= g->nkeys)
            return fail(MUSE_ERR_INVALID_ARG, "%s: where column %d not in [0,%d)", fn, (int)where_cols[j], g->nkeys);
        if (where_ids[j] < 0) return fail(MUSE_ERR_INVALID_ARG, "%s: negative label id %d", fn, (int)where_ids[j]);
        p.col[j] = g->labels + (size_t)where_cols[j] * g->cap;
        p.id[j] = where_ids[j];
    }
    return MUSE_OK;
}

// The selection of a predicate over the store's size() rows into buf (room for size() entries; ascending local rows), queued
// on the context's stream with off as the per-tile scratch: rows = buf and its length m, or rows = NULL when every row matches
// (the run of the whole store).
static int select_where(muse_ctx *ctx, const muse_group *g, const WherePred &p, int32_t *buf, DevBuf<int32_t> &off,
                        const int32_t *&rows, int64_t &m) {
    const int64_t S = g->size;
    cudaStream_t st = ctx->stream;
    const int64_t nb = (S + MUSE_WHERE_TILE - 1) / MUSE_WHERE_TILE;
    CU(off.grow(nb + 1));
    where_count_kernel<<<(unsigned)nb, 256, 0, st>>>(p, S, off);
    where_scan_kernel<<<1, 1024, 0, st>>>(off, nb);
    where_write_kernel<<<(unsigned)nb, 256, 0, st>>>(p, S, off, buf);
    CU(cudaGetLastError());
    int32_t h_m = 0;                      // one small copy: the host sizes the launches and takes the AUTO decision on it
    CU(cudaMemcpyAsync(&h_m, off.get() + nb, sizeof(h_m), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    m = h_m;
    rows = m < S ? buf : nullptr;
    return MUSE_OK;
}

// The run of b over the selection a.rows[0 .. a.count), made on the stream before this call (a.rows NULL: the whole store).
// Its timing starts at ev[0]: recorded by the caller, who queued a.pre_launches launches since, or here (a.pre_launches < 0).
static int run_selected(muse_batch *b, RunArgs a, double *scores, int64_t *lags, int64_t *series_idx, int64_t *n_out) {
    *n_out = 0;
    if (!a.rows) return batch_run(b, a, scores, lags, series_idx, n_out);
    int rc = ensure_lower(b);
    if (rc) return rc;
    cudaStream_t st = bstream(b);
    if (a.pre_launches < 0) {
        CU(cudaEventRecord(b->ev[0], st));
        a.pre_launches = 0;
    }
    if (a.count == 0) {    // nothing matches: no records and nothing scored
        memset(&b->timing, 0, sizeof(b->timing));
        b->timing_pending = 0;
        b->timing.mode = MUSE_MODE_EXACT;
        b->timing.n_launches = a.pre_launches;
        CU(cudaEventRecord(b->ev[1], st));      // no scoring pass, no re-scoring
        CU(cudaEventRecord(b->ev[2], st));
        return finish_timing(b);
    }
    const int64_t S = b->g->size;
    where_neutral_kernel<<<(unsigned)((S + 255) / 256), 256, 0, st>>>(b->d_score, b->d_U, b->d_L, S);
    CU(cudaGetLastError());
    a.pre_launches++;
    return batch_run(b, a, scores, lags, series_idx, n_out);
}

extern "C" int muse_batch_run_where(muse_batch *b, const int32_t *where_cols, const int32_t *where_ids, int32_t n_where,
                                    const int32_t *key_cols, int32_t n_key_cols, int64_t max_lag, int64_t top_n, double threshold,
                                    int32_t sign_filter, int32_t mode, int32_t signed_scores, double *scores, int64_t *lags,
                                    int64_t *series_idx, int64_t *n_out) {
    int rc = check_batch(b);
    if (rc) return rc;
    muse_group *g = b->g;
    WherePred p;
    rc = where_pred(g, where_cols, where_ids, n_where, "muse_batch_run_where", p);
    if (rc) return rc;
    rc = check_run_outputs("muse_batch_run_where", n_out, top_n, scores, lags, series_idx, key_cols, n_key_cols);
    if (rc) return rc;
    if (top_n < 0) top_n = 0;
    CU(cudaSetDevice(b->ctx->device));
    RunArgs a = run_args(g, key_cols, n_key_cols, max_lag, top_n, threshold, sign_filter, mode, signed_scores);
    a.group_cut = 1;
    *n_out = 0;
    rc = ensure_scratch(b);
    if (rc) return rc;
    if (n_where == 0 || g->size == 0) return batch_run(b, a, scores, lags, series_idx, n_out);      // the run of the whole store
    // The timing of a filtered run starts here, before the selection, and counts its launches in every case.
    CU(cudaEventRecord(b->ev[0], bstream(b)));
    rc = select_where(b->ctx, g, p, b->d_rows, b->d_where_off, a.rows, a.count);
    if (rc) return rc;
    a.pre_launches = 3;      // the selection's count, scan, write
    return run_selected(b, a, scores, lags, series_idx, n_out);
}

// ------------------------------------------------------------------------------------
// multi-GPU partials
// ------------------------------------------------------------------------------------
extern "C" int64_t muse_batch_partial_capacity(muse_batch *b, const int32_t *key_cols, int32_t n_key_cols, int64_t top_n) {
    (void)key_cols;
    if (!b) return 0;
    if (n_key_cols <= 0) return std::min<int64_t>(std::max<int64_t>(top_n, 0), b->g->size);
    return b->g->size;   // at most one representative per series
}

// The launch of a device-side top-N (partial_topn_kernel, partial_topn_push_kernel) behind queue_candidates.
struct TopnLaunch {
    long long exact_bound;   // the fused path's exact launch bound (its list must not be longer), else -1
    unsigned blocks;
};

// Queues the filter of an ungrouped run's exact scores into the candidate list (counters.cand).  The candidate and selected
// counts are still zero: run_scores cleared all four counters and ungrouped scoring writes only `listed` and `refined`.
static TopnLaunch queue_candidates(muse_batch *b, const RunArgs &a) {
    const int64_t S = b->g->size;
    cudaStream_t st = bstream(b);
    if (S > 0) {
        FilterArgs f{a.max_lag, a.threshold, a.sign_filter, 1};
        Cand cand{b->d_ckey, b->d_cidx, b->d_clag, &b->d_counters->cand};
        if (b->fused_run == 1) {
            // only the listed series have scores: filter those (the list's length stays on the device)
            const int64_t lim = std::min<int64_t>(a.count, MUSE_EXACT_UB);
            emit_listed_kernel<<<(unsigned)((lim + 255) / 256), 256, 0, st>>>(b->d_list, &b->d_counters->listed, lim, b->d_score, b->d_lag, f, cand);
        } else {
            GroupTable gt;
            memset(&gt, 0, sizeof(gt));
            emit_candidates_kernel<<<(unsigned)((S + 255) / 256), 256, 0, st>>>(gt, nullptr, b->d_score, b->d_lag, S, f, cand);
        }
        b->timing.n_launches++;
    }
    // the grid covers MUSE_PARTIAL_RANK_CAP candidates; blocks past the real count (device side) leave at once
    const long long exact_bound = b->fused_run == 1 ? (long long)std::min<int64_t>(a.count, MUSE_EXACT_UB) : -1;
    const unsigned pblocks = (unsigned)std::min<int64_t>((std::max<int64_t>(a.count, 1) + 7) / 8, (int64_t)b->ctx->sm_count * 8);   // 8 warps per block, one warp per candidate
    return TopnLaunch{exact_bound, pblocks};
}

// Ungrouped shard partials without a host round trip: scores, filter and the shard's top_n stay on
// the device; `d_out` (DEVICE memory, `capacity` >= top_n records) is complete when the work queued
// on the context's stream has run.  Nothing is synchronised here, so a collective enqueued on the
// same stream (ncclAllGather of the records) follows directly.
// Queues (no synchronisation): scores, filter, device-side top_n of an UNGROUPED run as muse_partial
// records in device memory, the counters into the pinned mailbox, and the end-of-run event.
static int queue_topn_records(muse_batch *b, const RunArgs &a_in, muse_partial *d_out, int64_t capacity) {
    static_assert(sizeof(PartialRec) == sizeof(muse_partial), "PartialRec mirrors muse_partial");
    RunArgs a = a_in;
    a.list_only = 1;
    int rc = run_scores(b, a);
    if (rc) return rc;
    cudaStream_t st = bstream(b);
    const TopnLaunch tl = queue_candidates(b, a);
    partial_topn_kernel<<<tl.blocks, 256, 0, st>>>(b->d_ckey, b->d_cidx, b->d_clag, b->d_counters, (long long)a.top_n,
                                                   (long long)b->g->global_offset, tl.exact_bound, reinterpret_cast<PartialRec *>(d_out),
                                                   (long long)capacity);
    b->timing.n_launches++;
    CU(cudaGetLastError());
    // statistics and the end-of-run event are picked up by muse_batch_last_timing
    CU(cudaMemcpyAsync(&b->h_pin->counters, b->d_counters, sizeof(RunCounters), cudaMemcpyDeviceToHost, st));
    CU(cudaEventRecord(b->ev[3], st));
    b->timing_pending = 1;
    return MUSE_OK;
}

extern "C" int muse_batch_run_partial_device(muse_batch *b, int64_t max_lag, int64_t top_n, double threshold, int32_t sign_filter,
                                             int32_t mode, muse_partial *d_out, int64_t capacity) {
    int rc = check_batch(b);
    if (rc) return rc;
    if (!d_out || capacity < 1) return fail(MUSE_ERR_INVALID_ARG, "muse_batch_run_partial_device: no output records");
    if (top_n < 0) top_n = 0;
    if (top_n > capacity) return fail(MUSE_ERR_INVALID_ARG, "partial capacity %lld < top_n %lld", (long long)capacity, (long long)top_n);
    CU(cudaSetDevice(b->ctx->device));
    rc = ensure_scratch(b);
    if (rc) return rc;
    return queue_topn_records(b, run_args(b->g, nullptr, 0, max_lag, top_n, threshold, sign_filter, mode, 0), d_out, capacity);
}

static int host_keys(muse_batch *b, const RunArgs &a, const std::vector<Rec> &recs, std::vector<uint64_t> &keys) {
    // canonical group key of each record's series (labels fetched per record)
    keys.resize(recs.size());
    muse_group *g = b->g;
    int bits[MUSE_MAX_KEY_COLS];
    int rc = key_bits(g, a.key_cols, a.n_key_cols, bits, true);
    if (rc) return rc;
    cudaStream_t st = bstream(b);
    std::vector<int32_t> ids(recs.size() * (size_t)a.n_key_cols);
    if (recs.size() > 4096) {
        std::vector<int32_t> col((size_t)g->size);
        for (int c = 0; c < a.n_key_cols; c++) {
            CU(cudaMemcpyAsync(col.data(), g->labels + (size_t)a.key_cols[c] * g->cap, sizeof(int32_t) * (size_t)g->size, cudaMemcpyDeviceToHost, st));
            CU(cudaStreamSynchronize(st));
            for (size_t i = 0; i < recs.size(); i++) ids[i * a.n_key_cols + c] = col[(size_t)recs[i].idx];
        }
    } else {
        for (size_t i = 0; i < recs.size(); i++)
            for (int c = 0; c < a.n_key_cols; c++)
                CU(cudaMemcpyAsync(&ids[i * a.n_key_cols + c], g->labels + (size_t)a.key_cols[c] * g->cap + recs[i].idx, sizeof(int32_t),
                                   cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
    }
    for (size_t i = 0; i < recs.size(); i++) {
        uint64_t key = 0;
        for (int c = 0; c < a.n_key_cols; c++) {
            const uint64_t v = (uint64_t)(ids[i * a.n_key_cols + c] + 1);
            key = bits[c] >= 64 ? v : ((key << bits[c]) | v);
        }
        keys[i] = key;
    }
    return MUSE_OK;
}

extern "C" int muse_batch_run_partial(muse_batch *b, const int32_t *key_cols, int32_t n_key_cols, int64_t max_lag, int64_t top_n,
                                      double threshold, int32_t sign_filter, int32_t mode, muse_partial *out, int64_t capacity,
                                      int64_t *n_out) {
    int rc = check_batch(b);
    if (rc) return rc;
    if (!out && capacity > 0) return fail(MUSE_ERR_INVALID_ARG, "muse_batch_run_partial: NULL output");
    rc = check_run_outputs("muse_batch_run_partial", n_out, 0, nullptr, nullptr, nullptr, key_cols, n_key_cols);
    if (rc) return rc;
    if (top_n < 0) top_n = 0;
    CU(cudaSetDevice(b->ctx->device));
    const RunArgs a = run_args(b->g, key_cols, n_key_cols, max_lag, top_n, threshold, sign_filter, mode, 0);
    *n_out = 0;
    rc = ensure_scratch(b);
    if (rc) return rc;
    rc = run_scores(b, a);
    if (rc) return rc;
    std::vector<Rec> recs;
    const bool grouped = n_key_cols > 0;
    // grouped: every representative, unfiltered (the filter needs the GLOBAL group max);
    // ungrouped: the shard's own filtered top_n is enough
    rc = run_select(b, a, grouped ? 0 : 1, grouped ? -1 : top_n, recs);
    if (rc) return rc;
    if ((int64_t)recs.size() > capacity) return fail(MUSE_ERR_INVALID_ARG, "partial capacity %lld < %zu records", (long long)capacity, recs.size());
    std::vector<uint64_t> keys;
    if (grouped) {
        rc = host_keys(b, a, recs, keys);
        if (rc) return rc;
    }
    for (size_t i = 0; i < recs.size(); i++) {
        out[i].series_idx = b->g->global_offset + recs[i].idx;
        out[i].group_key = grouped ? keys[i] : (uint64_t)out[i].series_idx;
        out[i].score = recs[i].score();
        out[i].lag = recs[i].lag();
        out[i].flags = 0;
    }
    *n_out = (int64_t)recs.size();
    return finish_timing(b);
}

extern "C" int muse_merge_partials(const muse_partial *parts, int64_t n_parts, int64_t max_lag, int64_t top_n, double threshold,
                                   int32_t sign_filter, double *scores, int64_t *lags, int64_t *series_idx, int64_t *n_out) {
    if (!n_out || (n_parts > 0 && !parts)) return fail(MUSE_ERR_INVALID_ARG, "muse_merge_partials: NULL argument");
    if (top_n < 0) top_n = 0;
    if (top_n > 0 && (!scores || !lags || !series_idx)) return fail(MUSE_ERR_INVALID_ARG, "muse_merge_partials: NULL output");
    // group max across shards first (muse_batch.go:87-89), ties -> lowest global series index
    const PartialRec *recs = reinterpret_cast<const PartialRec *>(parts);
    std::unordered_map<uint64_t, PartialRec> best;
    best.reserve((size_t)n_parts * 2 + 1);
    for (int64_t i = 0; i < n_parts; i++) {
        const PartialRec &p = recs[i];
        if ((p.flags & 1) || p.score != p.score) continue;
        auto it = best.find(p.group_key);
        if (it == best.end()) best.emplace(p.group_key, p);
        else if (rec_precedes(p, it->second)) it->second = p;
    }
    const FilterArgs f{max_lag, threshold, sign_filter, 1};
    std::vector<PartialRec> v;
    v.reserve(best.size());
    for (auto &kv : best)
        if (passed(f, kv.second.score, kv.second.lag)) v.push_back(kv.second);
    auto better = [](const PartialRec &x, const PartialRec &y) { return rec_precedes(x, y); };
    if ((int64_t)v.size() > top_n) {
        std::nth_element(v.begin(), v.begin() + top_n, v.end(), better);
        v.resize((size_t)top_n);
    }
    std::sort(v.begin(), v.end(), better);
    for (size_t i = 0; i < v.size(); i++) {
        scores[i] = v[i].score;
        lags[i] = v[i].lag;
        series_idx[i] = v[i].series_idx;
    }
    *n_out = (int64_t)v.size();
    return MUSE_OK;
}

// ------------------------------------------------------------------------------------
// many reference queries against one resident store (SURVEY 8f rank 2, BASELINE.json configs[4])
// ------------------------------------------------------------------------------------
// The bounds of up to TcCfg::TN queries (batches bs[0 .. nq), FFT length 2048, tables built) against the whole store, as
// one bf16 contraction on the tensor cores: magnitudes of every series -> tiles, the queries' weights -> tiles, GEMM with
// the bound's epilogue into every batch's d_U.  Everything is queued on the context's stream.  rows: the S series are the
// store's rows rows[0 .. S) (a selection; bound s is that of rows[s]), NULL: the store's S = size() rows.
static int tc_bounds_queue(muse_ctx *ctx, muse_group *g, muse_batch **bs, int nq, const int32_t *rows, int64_t S) {
    cudaStream_t st = ctx->stream;
    CU(ctx->mt_ev.create());
    int rc = refresh_row_stats(g);
    if (rc) return rc;
    CU(ctx->tc_a.grow((int64_t)TcCfg::a_bytes(S)));
    CU(ctx->tc_mid.grow(S));
    CU(ctx->tc_b.grow((int64_t)TcCfg::b_bytes()));
    CU(ctx->tc_amid.grow(TcCfg::TN));
    CU(ctx->tc_ptrs.grow(2 * TcCfg::TN));
    void *h_ptrs[2 * TcCfg::TN];
    float h_amid[TcCfg::TN];
    memset(h_ptrs, 0, sizeof(h_ptrs));
    memset(h_amid, 0, sizeof(h_amid));
    for (int q = 0; q < nq; q++) {
        rc = ensure_scratch(bs[q]);
        if (rc) return rc;
        h_ptrs[q] = bs[q]->sw_f;
        h_ptrs[TcCfg::TN + q] = bs[q]->d_U;
        h_amid[q] = bs[q]->a_mid;
    }
    // pageable sources: the copies have left the host buffers when the calls return
    CU(cudaMemcpyAsync(ctx->tc_ptrs, h_ptrs, sizeof(h_ptrs), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(ctx->tc_amid, h_amid, sizeof(h_amid), cudaMemcpyHostToDevice, st));
    const ScreenParams sp = screen_params(bs[0], rows, S);
    CU(cudaEventRecord(ctx->mt_ev[0], st));
    CU(launch_mag_tiles(sp, ctx->tc_a, ctx->tc_mid, ctx->sm_count, st));
    CU(launch_weight_tiles(reinterpret_cast<const float4 *const *>(ctx->tc_ptrs.get()), nq, ctx->tc_b, st));
    CU(cudaEventRecord(ctx->mt_ev[1], st));
    TcBoundsParams tp;
    memset(&tp, 0, sizeof(tp));
    tp.a_tiles = ctx->tc_a;
    tp.b_tiles = ctx->tc_b;
    tp.mid = ctx->tc_mid;
    tp.amid = ctx->tc_amid;
    tp.row_stat = g->row_stat;
    tp.rows = rows;
    tp.out_U = reinterpret_cast<float *const *>(ctx->tc_ptrs + TcCfg::TN);
    tp.S = S;
    tp.nq = nq;
    CU(launch_bounds_tc(tp, st));
    CU(cudaEventRecord(ctx->mt_ev[2], st));
    return MUSE_OK;
}

// ctx->d_multi_refs for rows of the store's length and pitch: MUSE_MULTI_GROUP reference rows, pad columns zero
static int ensure_multi_refs(muse_ctx *ctx, const muse_group *g) {
    if (ctx->d_multi_ld == g->ld && ctx->d_multi_n == g->N) return MUSE_OK;
    ctx->d_multi_ld = ctx->d_multi_n = 0;
    CU(ctx->d_multi_refs.grow(MUSE_MULTI_GROUP * g->ld));
    CU(cudaMemsetAsync(ctx->d_multi_refs, 0, sizeof(double) * (size_t)MUSE_MULTI_GROUP * (size_t)g->ld, ctx->stream));
    ctx->d_multi_ld = g->ld;
    ctx->d_multi_n = g->N;
    return MUSE_OK;
}

static bool tc_shape_ok(const muse_group *g, int64_t ref_len) {
    return ref_len == g->N && next_pow2(ref_len) == 2048;
}

// Layout of the per-launch tables of the tensor-core multi-query path (the same in device memory and in the pinned host
// mirror): parameter blocks of the batched kernels, then the results that come back.
struct MultiTables {
    static constexpr int Q = MUSE_MULTI_GROUP;
    static size_t off_ep() { return 0; }                                                  // ExactParams[Q]: reference spectra
    static size_t off_ta() { return off_ep() + sizeof(ExactParams) * Q; }                 // TablesArgs[Q]
    static size_t off_cut() { return off_ta() + sizeof(TablesArgs) * Q; }                 // CutState*[Q]: cut-off states
    static size_t off_tail() { return off_cut() + sizeof(void *) * Q; }                   // MultiTail[Q]
    static size_t off_ep2() { return off_tail() + sizeof(MultiTail) * Q; }                // ExactParams[Q]: fp64 re-scoring
    static size_t off_mids() { return off_ep2() + sizeof(ExactParams) * Q; }              // float[Q][4]
    static size_t off_cnt() { return off_mids() + sizeof(float) * 4 * Q; }                // RunCounters[Q]
    static size_t off_recs() { return (off_cnt() + sizeof(RunCounters) * Q + 255) / 256 * 256; }      // PartialRec[Q][top_n]
    static size_t bytes(int64_t top_n) { return off_recs() + sizeof(PartialRec) * (size_t)Q * (size_t)std::max<int64_t>(top_n, 1); }
};

// One launch group (<= 256 references) of muse_multi_run on the tensor-core path, with ONE launch per stage for all its
// queries: reference spectra and tables (batched fp64 kernel in MODE_REF, blockIdx.y = query), cut-off states, bounds
// (bf16 contraction), second stages (one pass over the store), survivors, fp64 re-scoring, filter, top-N -- and two
// round trips to the host: the std-zero flags after the preparation, the list lengths before the re-scoring.  A query
// whose lists do not fit the device-side select finishes alone on the single-query path.  The group's batches go into `bs`
// (nq entries), which the caller keeps until the work queued on them has run.  rows: the run covers the S series rows[0 .. S)
// of the store (a selection, muse_multi_run_where): the magnitudes, bounds and second stages are compact over them and the
// survivors' lists carry store rows, so the tails are those of a whole-store run.  NULL: the store's S = size() rows.
static int multi_run_tc_group(muse_ctx *ctx, muse_group *g, const int32_t *rows, int64_t S, const double *refs, int nq, int64_t ref_len,
                              int64_t max_lag, int64_t top_n, double threshold, int32_t sign_filter, double *scores, int64_t *lags,
                              int64_t *series_idx, int64_t *n_out, std::vector<BatchPtr> &bs) {
    using MT = MultiTables;
    cudaStream_t st = ctx->stream;
    CU(ctx->d_mt.grow((int64_t)MT::bytes(top_n)));
    CU(ctx->h_mt.grow((int64_t)MT::bytes(top_n)));
    unsigned char *d = ctx->d_mt, *h = ctx->h_mt;
    int rc = ensure_multi_refs(ctx, g);
    if (rc) return rc;
    CU(cudaMemcpy2DAsync(ctx->d_multi_refs, sizeof(double) * (size_t)g->ld, refs, sizeof(double) * (size_t)ref_len,
                         sizeof(double) * (size_t)ref_len, (size_t)nq, cudaMemcpyHostToDevice, st));

    // ---- reference preparation: one launch per stage ----
    ExactParams *h_ep = reinterpret_cast<ExactParams *>(h + MT::off_ep());
    TablesArgs *h_ta = reinterpret_cast<TablesArgs *>(h + MT::off_ta());
    CutState **h_cut = reinterpret_cast<CutState **>(h + MT::off_cut());
    for (int i = 0; i < nq; i++) {
        rc = batch_alloc(ctx, g, ref_len, bs[(size_t)i]);
        if (rc == MUSE_OK) rc = ensure_scratch(bs[(size_t)i].get());
        if (rc) return rc;
        muse_batch *b = bs[(size_t)i].get();
        ExactParams &p = h_ep[i];
        memset(&p, 0, sizeof(p));
        p.slab = ctx->d_multi_refs + (size_t)i * (size_t)g->ld;
        p.ld = g->ld;
        p.count = 1;
        p.N = (int)ref_len;
        p.twM = b->twM;
        p.twn = b->twn;
        p.out_X = b->Xt;
        p.out_flag = b->d_flag;
        h_ta[i] = TablesArgs{b->Xt, b->sw_f, b->sx_f, b->d_flag, b->sb_f};
        h_cut[i] = b->d_cut;
    }
    const int64_t M = bs[0]->n / 2;
    const float thr_lo = threshold_floor(threshold);
    CU(cudaMemcpyAsync(d, h, MT::off_tail(), cudaMemcpyHostToDevice, st));
    CU(launch_exact_batch(MODE_REF, reinterpret_cast<const ExactParams *>(d + MT::off_ep()), nq, 1, st));
    screen_tables_batch_kernel<<<dim3((unsigned)((M / 2 + 1 + 255) / 256), (unsigned)nq), 256, 0, st>>>(
        reinterpret_cast<const TablesArgs *>(d + MT::off_ta()), (int)M, bs[0]->swtw, reinterpret_cast<float *>(d + MT::off_mids()));
    init_cut_batch_kernel<<<dim3(MUSE_INIT_CUT_BLOCKS, (unsigned)nq), 256, 0, st>>>(reinterpret_cast<CutState *const *>(d + MT::off_cut()), thr_lo);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(h + MT::off_mids(), d + MT::off_mids(), sizeof(float) * 4 * (size_t)nq, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    const float *h_mids = reinterpret_cast<const float *>(h + MT::off_mids());
    std::vector<int> live;
    for (int i = 0; i < nq; i++) {
        int32_t flag;
        memcpy(&flag, &h_mids[4 * i], sizeof(flag));
        if (flag) {      // muse_batch.go:38-41: this query has no Batch; the others do
            n_out[i] = -1;
            continue;
        }
        muse_batch *b = bs[(size_t)i].get();
        b->a_mid = h_mids[4 * i + 1];
        b->x_mid = cf{h_mids[4 * i + 2], h_mids[4 * i + 3]};
        b->screen_ok = 1;
        n_out[i] = 0;
        live.push_back(i);
    }
    const int nl = (int)live.size();
    if (nl == 0) return MUSE_OK;

    // ---- bounds (tensor cores) and second stages (one pass over the store) ----
    std::vector<muse_batch *> lb((size_t)nl);
    std::vector<MultiQuery> hq((size_t)nl);
    ScreenParams sp0;
    for (int k = 0; k < nl; k++) {
        muse_batch *b = lb[(size_t)k] = bs[(size_t)live[(size_t)k]].get();
        ScreenParams sp = screen_params(b, rows, S);
        rc = arm_refinement(b, sp, thr_lo, max_lag, top_n, threshold, true);
        if (rc) return rc;
        if (k == 0) sp0 = sp;
        MultiQuery &m = hq[(size_t)k];
        memset(&m, 0, sizeof(m));
        m.sw = b->sw_f;
        m.sx = b->sx_f;
        m.x_mid = b->x_mid;
        m.a_mid = b->a_mid;
        m.cut = b->d_cut;
        m.out_U = b->d_U;
    }
    CU(ctx->d_multi_q.grow(MUSE_MULTI_GROUP));
    CU(ctx->d_multi_next.grow(1));
    MultiQuery *d_q = ctx->d_multi_q;
    CU(cudaMemcpyAsync(d_q, hq.data(), sizeof(MultiQuery) * (size_t)nl, cudaMemcpyHostToDevice, st));
    rc = tc_bounds_queue(ctx, g, lb.data(), nl, rows, S);
    if (rc) return rc;
    CU(launch_refine_multi(sp0, d_q, nl, ctx->sm_count, ctx->d_multi_next, st));
    CU(cudaEventRecord(ctx->mt_ev[3], st));

    // ---- tails: survivors -> fp64 re-scoring -> filter -> top-N, one launch each ----
    MultiTail *h_tail = reinterpret_cast<MultiTail *>(h + MT::off_tail());
    ExactParams *h_ep2 = reinterpret_cast<ExactParams *>(h + MT::off_ep2());
    RunCounters *d_cnt = reinterpret_cast<RunCounters *>(d + MT::off_cnt());
    PartialRec *d_recs = reinterpret_cast<PartialRec *>(d + MT::off_recs());
    const int64_t lim = std::min<int64_t>(S, MUSE_EXACT_UB);
    for (int k = 0; k < nl; k++) {
        muse_batch *b = lb[(size_t)k];
        h_tail[k] = MultiTail{b->d_U, b->d_cut, b->d_list, d_cnt + k, b->d_score, b->d_lag, b->d_ckey, b->d_cidx, b->d_clag,
                              d_recs + (size_t)k * (size_t)top_n};
        ExactParams &p = h_ep2[k];
        memset(&p, 0, sizeof(p));
        p.slab = g->slab;
        p.ld = g->ld;
        p.count = lim;
        p.count_ptr = &d_cnt[k].listed;
        p.idx = b->d_list;
        p.N = (int)ref_len;
        p.Xt = b->Xt;
        p.twM = b->twM;
        p.twn = b->twn;
        p.out_score = b->d_score;
        p.out_lag = b->d_lag;
    }
    CU(cudaMemcpyAsync(d + MT::off_tail(), h + MT::off_tail(), MT::off_mids() - MT::off_tail(), cudaMemcpyHostToDevice, st));
    const MultiTail *d_tail = reinterpret_cast<const MultiTail *>(d + MT::off_tail());
    tail_reset_kernel<<<(nl + 255) / 256, 256, 0, st>>>(d_tail, nl);
    survivors_cut_batch_kernel<<<dim3((unsigned)((S + 255) / 256), (unsigned)nl), 256, 0, st>>>(d_tail, S, rows);
    CU(cudaGetLastError());
    RunCounters *h_cnt = reinterpret_cast<RunCounters *>(h + MT::off_cnt());
    CU(cudaMemcpyAsync(h_cnt, d_cnt, sizeof(RunCounters) * (size_t)nl, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));      // the list lengths size the next launches
    int64_t max_len = 0;
    for (int k = 0; k < nl; k++) max_len = std::max<int64_t>(max_len, std::min<int64_t>((int64_t)h_cnt[k].listed, lim));
    if (max_len > 0) {
        CU(launch_exact_batch(MODE_SCORE, reinterpret_cast<const ExactParams *>(d + MT::off_ep2()), nl, max_len, st));
        FilterArgs f{max_lag, threshold, sign_filter, 1};
        emit_listed_batch_kernel<<<dim3((unsigned)((max_len + 255) / 256), (unsigned)nl), 256, 0, st>>>(d_tail, (long long)lim, f);
    }
    partial_topn_batch_kernel<<<dim3(16, (unsigned)nl), 256, 0, st>>>(d_tail, (long long)top_n, (long long)g->global_offset, (long long)lim);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(h + MT::off_recs(), d_recs, sizeof(PartialRec) * (size_t)nl * (size_t)top_n, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(h_cnt, d_cnt, sizeof(RunCounters) * (size_t)nl, cudaMemcpyDeviceToHost, st));
    CU(cudaEventRecord(ctx->mt_ev[4], st));
    CU(cudaStreamSynchronize(st));
    const muse_partial *h_recs = reinterpret_cast<const muse_partial *>(h + MT::off_recs());
    for (int k = 0; k < nl; k++) {
        const int i = live[(size_t)k];
        const muse_partial *r = h_recs + (size_t)k * (size_t)top_n;
        double *sc = scores + (size_t)i * (size_t)top_n;
        int64_t *lg = lags + (size_t)i * (size_t)top_n, *ix = series_idx + (size_t)i * (size_t)top_n;
        ctx->multi_rescored += (int64_t)h_cnt[k].listed;
        ctx->multi_refined += (int64_t)h_cnt[k].refined;
        if (r[0].flags == 2) {
            // the list did not fit the device-side select (or the re-scoring launch): this query finishes alone, from its
            // bounds and cut-off on the device (the fused run skips the screening of a prescreened run) -- or, over a
            // selection, whose bounds are compact and not those of the store's rows, screened again as a filtered run
            RunArgs a = run_args(g, nullptr, 0, max_lag, top_n, threshold, sign_filter, MUSE_MODE_SCREEN, 0);
            a.rows = rows;
            a.count = S;
            a.prescreened = rows ? 0 : 1;
            rc = run_selected(lb[(size_t)k], a, sc, lg, ix, n_out + i);
            if (rc) return rc;
            continue;
        }
        n_out[i] = records_out(r, top_n, sc, lg, ix);
    }
    return MUSE_OK;
}

extern "C" int muse_multi_last_stats(const muse_ctx *ctx, int64_t *n_refined, int64_t *n_rescored) {
    if (!ctx || !n_refined || !n_rescored) return fail(MUSE_ERR_INVALID_ARG, "muse_multi_last_stats: NULL argument");
    *n_refined = ctx->multi_refined;
    *n_rescored = ctx->multi_rescored;
    return MUSE_OK;
}

extern "C" int muse_multi_last_timing(const muse_ctx *ctx, float *ms4) {
    if (!ctx || !ms4) return fail(MUSE_ERR_INVALID_ARG, "muse_multi_last_timing: NULL argument");
    for (int i = 0; i < 4; i++) {
        ms4[i] = 0.f;
        if (ctx->mt_ev[i] && ctx->mt_ev[i + 1] && cudaEventElapsedTime(&ms4[i], ctx->mt_ev[i], ctx->mt_ev[i + 1]) != cudaSuccess) {
            (void)cudaGetLastError();
            ms4[i] = 0.f;
        }
    }
    return MUSE_OK;
}

extern "C" int muse_multi_bounds_tc(muse_ctx *ctx, muse_group *g, const double *refs, int64_t n_refs, int64_t ref_len, float *upper) {
    if (!ctx || !g || !refs || !upper) return fail(MUSE_ERR_INVALID_ARG, "muse_multi_bounds_tc: NULL argument");
    if (n_refs < 1 || n_refs > TcCfg::TN) return fail(MUSE_ERR_INVALID_ARG, "muse_multi_bounds_tc: 1 .. %d references", TcCfg::TN);
    if (!tc_shape_ok(g, ref_len)) return fail(MUSE_ERR_UNSUPPORTED, "the tensor-core bounds exist for even series lengths of FFT length 2048");
    CU(cudaSetDevice(ctx->device));
    const int64_t S = g->size;
    if (S == 0) return MUSE_OK;
    std::vector<BatchPtr> own((size_t)n_refs);
    std::vector<muse_batch *> bs((size_t)n_refs);
    for (size_t q = 0; q < bs.size(); q++) {
        const int rc = muse_batch_create(ctx, g, refs + q * (size_t)ref_len, ref_len, &bs[q]);
        if (rc) return rc;
        own[q].reset(bs[q]);
    }
    const int rc = tc_bounds_queue(ctx, g, bs.data(), (int)bs.size(), nullptr, S);
    if (rc) return rc;
    for (size_t q = 0; q < bs.size(); q++)
        CU(cudaMemcpyAsync(upper + q * (size_t)S, bs[q]->d_U, sizeof(float) * (size_t)S, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return MUSE_OK;
}

// The argument checks of muse_multi_run (fn names the entry point in the message).
static int multi_check(const muse_ctx *ctx, const muse_group *g, const double *refs, int64_t n_refs, const int32_t *key_cols,
                       int32_t n_key_cols, int64_t top_n, const double *scores, const int64_t *lags, const int64_t *series_idx,
                       const int64_t *n_out, const char *fn) {
    if (!ctx || !g || (!refs && n_refs > 0) || !n_out) return fail(MUSE_ERR_INVALID_ARG, "%s: NULL argument", fn);
    if (n_refs < 0 || top_n < 0) return fail(MUSE_ERR_INVALID_ARG, "%s: n_refs %lld, top_n %lld", fn, (long long)n_refs, (long long)top_n);
    return check_run_outputs(fn, n_out, top_n, scores, lags, series_idx, key_cols, n_key_cols);
}

// muse_multi_run over the m store rows rows[0 .. m) (ascending; a selection of muse_multi_run_where), or over the whole store
// (rows NULL, m = size()).  Every decision that depends on the size of the store takes m, so the call takes the path, and
// returns the records, of a store that holds only those rows.
static int multi_run(muse_ctx *ctx, muse_group *g, const int32_t *rows, int64_t m, const double *refs, int64_t n_refs, int64_t ref_len,
                     const int32_t *key_cols, int32_t n_key_cols, int64_t max_lag, int64_t top_n, double threshold, int32_t sign_filter,
                     int32_t mode, double *scores, int64_t *lags, int64_t *series_idx, int64_t *n_out) {
    // the tensor-core path (multi_run_tc_group, up to MUSE_MULTI_GROUP queries per pass over the store) exists for the
    // shape the single-query warp kernel serves (FFT length 2048, ungrouped, unsigned scores, a sign filter unsigned
    // scores can pass, a store worth screening, a device-side top-N); everything else -- and a group of one query -- is
    // NewBatch + Run per reference on the resident store: the store, its row statistics and the run scratch (context
    // pool) are shared, and results of query q land in row q of the outputs
    const bool one_pass = n_key_cols == 0 && mode != MUSE_MODE_EXACT && sign_filter != MUSE_SIGN_NEG && ref_len == g->N &&
                          next_pow2(ref_len) == 2048 && device_topn_fits(top_n, m) &&
                          (m >= 16384 || mode == MUSE_MODE_SCREEN) && n_refs > 1;
    ctx->multi_refined = ctx->multi_rescored = 0;
    const int QC = one_pass ? MUSE_MULTI_GROUP : MUSE_MULTI_SEPARATE;
    for (int64_t q0 = 0; q0 < n_refs; q0 += QC) {
        const int nq = (int)std::min<int64_t>(QC, n_refs - q0);
        if (one_pass && nq > 1) {
            std::vector<BatchPtr> bs((size_t)nq);
            const int rc = multi_run_tc_group(ctx, g, rows, m, refs + (size_t)q0 * (size_t)ref_len, nq, ref_len, max_lag, top_n, threshold,
                                              sign_filter, scores + (size_t)q0 * (size_t)top_n, lags + (size_t)q0 * (size_t)top_n,
                                              series_idx + (size_t)q0 * (size_t)top_n, n_out + q0, bs);
            if (rc) {
                cudaStreamSynchronize(ctx->stream);      // work queued on the batches may still be running: it ends before they go
                return rc;
            }
            continue;
        }
        int rc = MUSE_OK;
        // the references of the group: ONE upload (rows at the slab's pitch, pad columns zero), then queued back to
        // back, ONE round trip
        const bool rows_on_device = ref_len == g->N;
        if (rows_on_device) {
            rc = ensure_multi_refs(ctx, g);
            if (rc) return rc;
            CU(cudaMemcpy2DAsync(ctx->d_multi_refs, sizeof(double) * (size_t)g->ld, refs + (size_t)q0 * (size_t)ref_len,
                                 sizeof(double) * (size_t)ref_len, sizeof(double) * (size_t)ref_len, (size_t)nq,
                                 cudaMemcpyHostToDevice, ctx->stream));
        }
        std::vector<BatchPtr> bs((size_t)nq);
        for (int i = 0; i < nq && rc == MUSE_OK; i++)
            rc = batch_create_queue(ctx, g, refs + (size_t)(q0 + i) * (size_t)ref_len, ref_len, bs[(size_t)i],
                                    rows_on_device ? ctx->d_multi_refs + (size_t)i * (size_t)g->ld : nullptr);
        if (cudaStreamSynchronize(ctx->stream) != cudaSuccess && rc == MUSE_OK) rc = fail(MUSE_ERR_CUDA, "cudaStreamSynchronize failed");
        if (rc) return rc;
        for (int i = 0; i < nq; i++) {
            rc = batch_create_finish(bs[(size_t)i].get());
            if (rc == MUSE_ERR_STDDEV_ZERO) {   // muse_batch.go:38-41: this query has no Batch; the others do
                n_out[q0 + i] = -1;
                bs[(size_t)i].reset();
            } else if (rc) {
                return rc;
            }
        }
        RunArgs a = run_args(g, key_cols, n_key_cols, max_lag, top_n, threshold, sign_filter, mode, 0);
        a.group_cut = 1;
        a.rows = rows;      // every query of the call reads the one selection
        a.count = m;
        for (int i = 0; i < nq; i++) {
            if (!bs[(size_t)i]) continue;
            const int64_t q = q0 + i;
            double *sc = scores ? scores + (size_t)q * (size_t)top_n : nullptr;
            int64_t *lg = lags ? lags + (size_t)q * (size_t)top_n : nullptr, *ix = series_idx ? series_idx + (size_t)q * (size_t)top_n : nullptr;
            rc = ensure_scratch(bs[(size_t)i].get());
            if (rc == MUSE_OK) rc = run_selected(bs[(size_t)i].get(), a, sc, lg, ix, n_out + q);
            bs[(size_t)i].reset();
            if (rc) return rc;
        }
    }
    return MUSE_OK;
}

extern "C" int muse_multi_run(muse_ctx *ctx, muse_group *g, const double *refs, int64_t n_refs, int64_t ref_len,
                              const int32_t *key_cols, int32_t n_key_cols, int64_t max_lag, int64_t top_n, double threshold,
                              int32_t sign_filter, int32_t mode, double *scores, int64_t *lags, int64_t *series_idx,
                              int64_t *n_out) {
    const int rc = multi_check(ctx, g, refs, n_refs, key_cols, n_key_cols, top_n, scores, lags, series_idx, n_out, "muse_multi_run");
    if (rc) return rc;
    CU(cudaSetDevice(ctx->device));
    return multi_run(ctx, g, nullptr, g->size, refs, n_refs, ref_len, key_cols, n_key_cols, max_lag, top_n, threshold, sign_filter, mode,
                     scores, lags, series_idx, n_out);
}

extern "C" int muse_multi_run_where(muse_ctx *ctx, muse_group *g, const double *refs, int64_t n_refs, int64_t ref_len,
                                    const int32_t *where_cols, const int32_t *where_ids, int32_t n_where, const int32_t *key_cols,
                                    int32_t n_key_cols, int64_t max_lag, int64_t top_n, double threshold, int32_t sign_filter,
                                    int32_t mode, double *scores, int64_t *lags, int64_t *series_idx, int64_t *n_out) {
    int rc = multi_check(ctx, g, refs, n_refs, key_cols, n_key_cols, top_n, scores, lags, series_idx, n_out, "muse_multi_run_where");
    if (rc) return rc;
    WherePred p;
    rc = where_pred(g, where_cols, where_ids, n_where, "muse_multi_run_where", p);
    if (rc) return rc;
    if (n_where == 0 || g->size == 0 || n_refs == 0)
        return muse_multi_run(ctx, g, refs, n_refs, ref_len, key_cols, n_key_cols, max_lag, top_n, threshold, sign_filter, mode, scores,
                              lags, series_idx, n_out);
    if (g->ctx != ctx) return fail(MUSE_ERR_INVALID_ARG, "muse_multi_run_where: group belongs to another context");
    CU(cudaSetDevice(ctx->device));
    // ONE selection for every reference of the call
    CU(ctx->d_where_rows.grow(g->size));
    const int32_t *rows = nullptr;
    int64_t m = 0;
    rc = select_where(ctx, g, p, ctx->d_where_rows, ctx->d_where_off, rows, m);
    if (rc) return rc;
    return multi_run(ctx, g, rows, m, refs, n_refs, ref_len, key_cols, n_key_cols, max_lag, top_n, threshold, sign_filter, mode, scores,
                     lags, series_idx, n_out);
}

// ------------------------------------------------------------------------------------
// generic xCorr (xcorr.go:102-153): any n, optional z-normalisation
// ------------------------------------------------------------------------------------
extern "C" int muse_xcorr(muse_ctx *ctx, const double *x, int64_t x_len, const double *y, int64_t y_len, int64_t n,
                          int32_t normalize, double *cc, int64_t cc_capacity, int64_t *n_out, int64_t *lag, double *value,
                          int32_t *std_zero) {
    if (!ctx || !x || !y || !n_out || !lag || !value) return fail(MUSE_ERR_INVALID_ARG, "muse_xcorr: NULL argument");
    if (x_len < 1 || y_len < 1) return fail(MUSE_ERR_INVALID_ARG, "muse_xcorr: empty input (x %lld, y %lld samples)", (long long)x_len, (long long)y_len);
    const int64_t nn = std::max(n, std::max(x_len, y_len));   // xcorr.go:104-106
    // up to 4096 lags: direct evaluation, n^2 fp64 FMAs (the reference's own vectors are n = 5).  Above: the FFT passes of
    // kernels_long.cu -- one transform of length n when n is a power of two (the reference's benchmark shape, n = 32768),
    // else the linear correlation at a power of two >= 2n, folded
    if (nn > (1ll << 26)) return fail(MUSE_ERR_UNSUPPORTED, "muse_xcorr: n = %lld above 2^26", (long long)nn);
    const bool by_fft = nn > 4096;
    long long L = nn;
    if (by_fft && (nn & (nn - 1))) L = next_pow2(2 * nn);
    const size_t work_bytes = by_fft ? long_xcorr_work_bytes(L) : 0;
    if (cc && cc_capacity < nn) return fail(MUSE_ERR_INVALID_ARG, "muse_xcorr: cc holds %lld values, n = %lld", (long long)cc_capacity, (long long)nn);
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    *n_out = nn;
    *lag = 0;
    *value = 0.0;
    if (std_zero) *std_zero = 0;
    // one allocation: x, y, xp, yp, cc (doubles), then lag, value, flag
    const size_t nd = (size_t)x_len + (size_t)y_len + 3 * (size_t)nn;
    DevBuf<unsigned char> d;
    CU(d.grow((int64_t)(nd * sizeof(double) + 32 + 256 + work_bytes)));
    void *d_work = d + ((nd * sizeof(double) + 32 + 255) / 256) * 256;
    double *dx = reinterpret_cast<double *>(d.get()), *dy = dx + x_len, *dxp = dy + y_len, *dyp = dxp + nn, *dcc = dyp + nn;
    long long *dlag = reinterpret_cast<long long *>(dcc + nn);
    double *dval = reinterpret_cast<double *>(dlag + 1);
    int *dflag = reinterpret_cast<int *>(dval + 1);
    struct Tail { long long lag; double val; int flag; int pad; } tail;
    CU(cudaMemcpyAsync(dx, x, sizeof(double) * (size_t)x_len, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(dy, y, sizeof(double) * (size_t)y_len, cudaMemcpyHostToDevice, st));
    CU(cudaMemsetAsync(dlag, 0, 32, st));
    xcorr_prepare_kernel<<<2, 256, 0, st>>>(dx, x_len, dy, y_len, nn, normalize ? 1 : 0, dxp, dyp, dflag);
    // xcorr.go:139-142: gonum's inverse transform is unnormalised (n x the correlation); the reference scales
    // by 1/(n(n-1)) for z-normalised inputs and by 1/n otherwise -> 1/(n-1) and 1 on a direct sum
    const double scale = normalize ? 1.0 / (double)(nn - 1) : 1.0;
    if (by_fft) CU(launch_long_xcorr(dxp, dyp, nn, L, scale, dcc, d_work, st));
    else xcorr_direct_kernel<<<(unsigned)((nn + XC_LAGS - 1) / XC_LAGS), XC_LAGS, 0, st>>>(dxp, dyp, nn, scale, dcc);
    xcorr_argmax_kernel<<<1, 256, 0, st>>>(dcc, nn, dlag, dval);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(&tail, dlag, sizeof(tail), cudaMemcpyDeviceToHost, st));
    if (cc) CU(cudaMemcpyAsync(cc, dcc, sizeof(double) * (size_t)nn, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (normalize && tail.flag) {   // xcorr.go:109-126: (nil, 0, 0)
        if (std_zero) *std_zero = 1;
        *n_out = 0;
        return MUSE_OK;
    }
    *lag = tail.lag;
    *value = tail.val;
    return MUSE_OK;
}

// ------------------------------------------------------------------------------------
// multi-GPU exchange over NVLink peer memory (one process per GPU)
// ------------------------------------------------------------------------------------
struct muse_exchange {
    muse_ctx *ctx = nullptr;
    int rank = 0, world = 0;
    int64_t capacity = 0;                 // records per rank per step
    DevBuf<unsigned char> base;           // local buffer: recs[2][world][capacity] then flags[2][world] (IPC-exported)
    size_t recs_bytes = 0;                // bytes of ONE parity's records
    unsigned char *peer_base[MUSE_EXCHANGE_MAX_RANKS] = {};   // every rank's buffer as seen from here (own: base)
    bool opened = false;
    unsigned long long epoch = 0;
    DevBuf<unsigned> d_done;
    DevBuf<int> d_status;
    PinnedBuf h_recs;                     // pinned: the merged top_n records of one step, then the status word
    // device-side merge of the gathered records (group max across shards, filter, top-N), all in merge_buf
    DevBuf<unsigned char> merge_buf;
    MergeState merge = {};
    size_t merge_bytes = 0;               // the hash table at the front of merge_buf: merge.hkeys, gmax, gidx
    unsigned long long *d_nlocal = nullptr;   // grouped runs: representatives of this shard
    PartialRec *d_out = nullptr;          // [capacity] merged top_n
    // muse_multi_run_exchange, allocated on its first call: this rank's per-query lists of one step, device and pinned host
    // ([capacity] records, [MUSE_MULTI_GROUP] counts; the host copy then receives the [world] flag words of the step)
    DevBuf<unsigned char> d_send;
    PinnedBuf h_send;
};

// Opens the next step of the exchange: a new epoch, and every rank's receive records and flags of the epoch's parity.
static ExchangePeers exchange_step(muse_exchange *x) {
    x->epoch++;
    const int par = (int)(x->epoch & 1ull);
    ExchangePeers ex;
    memset(&ex, 0, sizeof(ex));
    for (int r = 0; r < x->world; r++) {
        ex.recs[r] = reinterpret_cast<PartialRec *>(x->peer_base[r] + (size_t)par * x->recs_bytes);
        ex.flags[r] = reinterpret_cast<unsigned long long *>(x->peer_base[r] + 2 * x->recs_bytes) + (size_t)par * x->world;
    }
    ex.world = x->world;
    ex.rank = x->rank;
    ex.epoch = x->epoch;
    ex.done_blocks = x->d_done;
    return ex;
}

// exchange_wait_kernel's limit, ~10 s at ~2 GHz: ranks may be a whole host->device upload apart, but a peer that never
// arrives must not hang the box
#define MUSE_EXCHANGE_TIMEOUT_CYCLES 20000000000ll

static size_t exchange_bytes(int world, int64_t capacity) {
    return 2 * (size_t)world * (size_t)capacity * sizeof(muse_partial) + 2 * (size_t)world * sizeof(unsigned long long);
}

extern "C" int muse_exchange_create(muse_ctx *ctx, int32_t rank, int32_t world, int64_t capacity, muse_exchange **out) {
    if (!ctx || !out) return fail(MUSE_ERR_INVALID_ARG, "muse_exchange_create: NULL argument");
    if (world < 1 || world > MUSE_EXCHANGE_MAX_RANKS || rank < 0 || rank >= world || capacity < 1)
        return fail(MUSE_ERR_INVALID_ARG, "muse_exchange_create: rank %d of %d, capacity %lld", rank, world, (long long)capacity);
    CU(cudaSetDevice(ctx->device));
    std::unique_ptr<muse_exchange> x(new muse_exchange());
    x->ctx = ctx;
    x->rank = rank;
    x->world = world;
    x->capacity = capacity;
    x->recs_bytes = (size_t)world * (size_t)capacity * sizeof(muse_partial);
    const size_t bytes = exchange_bytes(world, capacity);
    CU(x->base.grow((int64_t)bytes));
    CU(cudaMemset(x->base, 0, bytes));
    CU(x->d_done.grow(1));
    CU(cudaMemset(x->d_done, 0, sizeof(unsigned)));
    CU(x->d_status.grow(1));
    CU(cudaMemset(x->d_status, 0, sizeof(int)));
    CU(x->h_recs.grow((int64_t)((size_t)capacity * sizeof(muse_partial) + 64)));
    {   // merge scratch: hash table of 2 x (records of all shards) slots, candidate arrays, counters, output records
        const long long total = (long long)world * capacity;
        long long slots = 1;
        while (slots < 2 * total) slots <<= 1;
        const size_t tab = sizeof(unsigned long long) * (size_t)slots;
        const size_t bytes_m = 3 * tab + (size_t)total * (8 + 8 + 4) + 64 + (size_t)capacity * sizeof(PartialRec) + 64;
        CU(x->merge_buf.grow((int64_t)bytes_m));
        CU(cudaMemset(x->merge_buf, 0, bytes_m));
        x->merge_bytes = 3 * tab;
        x->merge.hkeys = reinterpret_cast<unsigned long long *>(x->merge_buf.get());
        x->merge.gmax = x->merge.hkeys + slots;
        x->merge.gidx = x->merge.gmax + slots;
        x->merge.slots = slots;
        x->merge.ckey = x->merge.gidx + slots;
        x->merge.cidx = reinterpret_cast<long long *>(x->merge.ckey + total);
        x->merge.clag = reinterpret_cast<int32_t *>(x->merge.cidx + total);
        unsigned char *tail = reinterpret_cast<unsigned char *>(x->merge.clag + total);
        tail = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(tail) + 31) & ~(uintptr_t)31);
        x->merge.counters = reinterpret_cast<unsigned long long *>(tail);
        x->d_nlocal = x->merge.counters + 4;
        x->d_out = reinterpret_cast<PartialRec *>(tail + 64);
    }
    x->peer_base[rank] = x->base;
    x->opened = (world == 1);
    CU(cudaDeviceSynchronize());
    *out = x.release();
    return MUSE_OK;
}

extern "C" int muse_exchange_ipc_handle(muse_exchange *x, void *handle64) {
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    if (!x || !handle64) return fail(MUSE_ERR_INVALID_ARG, "muse_exchange_ipc_handle: NULL argument");
    if (getenv("MUSE_B200_NO_IPC"))      // test hook: behave like a box where CUDA IPC is closed (callers fall back to the all-gather path)
        return fail(MUSE_ERR_UNSUPPORTED, "CUDA IPC disabled by MUSE_B200_NO_IPC");
    CU(cudaSetDevice(x->ctx->device));
    cudaIpcMemHandle_t h;
    CU(cudaIpcGetMemHandle(&h, x->base));
    memcpy(handle64, &h, sizeof(h));
    return MUSE_OK;
}

extern "C" int muse_exchange_open_peers(muse_exchange *x, const void *handles) {
    if (!x || !handles) return fail(MUSE_ERR_INVALID_ARG, "muse_exchange_open_peers: NULL argument");
    CU(cudaSetDevice(x->ctx->device));
    for (int r = 0; r < x->world; r++) {
        if (r == x->rank) continue;
        cudaIpcMemHandle_t h;
        memcpy(&h, (const unsigned char *)handles + (size_t)r * sizeof(h), sizeof(h));
        void *p = nullptr;
        CU(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
        x->peer_base[r] = (unsigned char *)p;
    }
    x->opened = true;
    return MUSE_OK;
}

extern "C" void muse_exchange_destroy(muse_exchange *x) {
    if (!x) return;
    cudaSetDevice(x->ctx->device);
    cudaStreamSynchronize(x->ctx->stream);
    for (int r = 0; r < x->world; r++)
        if (r != x->rank && x->peer_base[r]) cudaIpcCloseMemHandle(x->peer_base[r]);
    delete x;
}

// One multi-GPU step: scores, then the shard's records stored straight into every rank's receive buffer over NVLink peer
// memory by the kernel that produces them -- ungrouped: the filtered local top_n (partial_topn_push_kernel); grouped: every
// group representative, unfiltered (group_records_push_kernel, SURVEY F2) --, wait for all the peers' flags, merge ON THE
// DEVICE (group max across shards, filter, top-N) and copy only the top_n records to the host.  Every rank returns the same
// global result.  MUSE_ERR_UNSUPPORTED ("host path needed") when a shard's list was too long for the device-side select or
// for its slot: every rank sees the same marker and can fall back together.
extern "C" int muse_batch_run_exchange_ex(muse_batch *b, muse_exchange *x, const int32_t *key_cols, int32_t n_key_cols, int64_t max_lag,
                                          int64_t top_n, double threshold, int32_t sign_filter, int32_t mode, double *scores, int64_t *lags,
                                          int64_t *series_idx, int64_t *n_out) {
    int rc = check_batch(b);
    if (rc) return rc;
    if (!x) return fail(MUSE_ERR_INVALID_ARG, "muse_batch_run_exchange: NULL argument");
    if (x->ctx != b->ctx) return fail(MUSE_ERR_INVALID_ARG, "exchange belongs to another context");
    if (!x->opened) return fail(MUSE_ERR_INVALID_ARG, "muse_exchange_open_peers has not been called");
    rc = check_run_outputs("muse_batch_run_exchange", n_out, top_n, scores, lags, series_idx, key_cols, n_key_cols);
    if (rc) return rc;
    if (top_n < 0) top_n = 0;
    if (top_n > x->capacity) return fail(MUSE_ERR_INVALID_ARG, "exchange capacity %lld < top_n %lld", (long long)x->capacity, (long long)top_n);
    CU(cudaSetDevice(b->ctx->device));
    *n_out = 0;
    const bool grouped = n_key_cols > 0;
    RunArgs a = run_args(b->g, key_cols, n_key_cols, max_lag, top_n, threshold, sign_filter, mode, 0);
    a.list_only = grouped ? 0 : 1;
    rc = ensure_scratch(b);
    if (rc) return rc;
    rc = run_scores(b, a);
    if (rc) return rc;
    const int64_t S = b->g->size;
    cudaStream_t st = bstream(b);
    const ExchangePeers ex = exchange_step(x);
    if (grouped) {
        // group max and representative of THIS shard on the exact scores (as run_select does), then the push
        GroupTable gt;
        KeyCols kc;
        rc = queue_group_reps(b, a, true, kc, gt);
        if (rc) return rc;
        // one block even for an empty shard: its last block releases the shard's flag, which the peers wait for
        const unsigned blocks = (unsigned)((std::max<int64_t>(S, 1) + 255) / 256);
        group_records_push_kernel<<<blocks, 256, 0, st>>>(gt, kc, b->d_slot, b->d_score, b->d_lag, (long long)S, (long long)b->g->global_offset,
                                                          (long long)x->capacity, x->d_nlocal, ex);
    } else {
        const TopnLaunch tl = queue_candidates(b, a);
        partial_topn_push_kernel<<<tl.blocks, 256, 0, st>>>(b->d_ckey, b->d_cidx, b->d_clag, b->d_counters, (long long)top_n,
                                                            (long long)b->g->global_offset, tl.exact_bound, (long long)x->capacity, ex);
    }
    b->timing.n_launches++;
    exchange_wait_kernel<<<1, 32, 0, st>>>(ex.flags[x->rank], x->world, x->epoch, MUSE_EXCHANGE_TIMEOUT_CYCLES, x->d_status);
    // merge on the device: the hash table, candidate counter and status start from zero
    CU(cudaMemsetAsync(x->merge.hkeys, 0, x->merge_bytes / 3 * 2, st));                       // keys and maxima
    CU(cudaMemsetAsync(x->merge.gidx, 0xff, x->merge_bytes / 3, st));                         // representatives: +inf
    CU(cudaMemsetAsync(x->merge.counters, 0, sizeof(unsigned long long) * 4, st));
    const long long total = (long long)x->world * x->capacity;
    const unsigned mblocks = (unsigned)((total + 255) / 256);
    const PartialRec *recs_local = ex.recs[x->rank];
    FilterArgs f{a.max_lag, a.threshold, a.sign_filter, 1};
    merge_max_kernel<<<mblocks, 256, 0, st>>>(x->merge, recs_local, ex.flags[x->rank], x->world, (long long)x->capacity);
    merge_rep_kernel<<<mblocks, 256, 0, st>>>(x->merge, recs_local, ex.flags[x->rank], x->world, (long long)x->capacity);
    merge_emit_kernel<<<mblocks, 256, 0, st>>>(x->merge, recs_local, ex.flags[x->rank], x->world, (long long)x->capacity, f);
    merged_topn_kernel<<<(unsigned)std::min<long long>((total + 7) / 8, (long long)b->ctx->sm_count * 8), 256, 0, st>>>(x->merge, (long long)top_n, x->d_out);
    b->timing.n_launches += 5;
    CU(cudaGetLastError());
    int *h_status = reinterpret_cast<int *>(x->h_recs + (size_t)x->capacity * sizeof(muse_partial));
    if (top_n > 0) CU(cudaMemcpyAsync(x->h_recs, x->d_out, sizeof(muse_partial) * (size_t)top_n, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(h_status, x->d_status, sizeof(int), cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(&b->h_pin->counters, b->d_counters, sizeof(RunCounters), cudaMemcpyDeviceToHost, st));
    CU(cudaEventRecord(b->ev[3], st));
    b->timing_pending = 1;
    CU(cudaStreamSynchronize(st));
    if (*h_status) {
        CU(cudaMemsetAsync(x->d_status, 0, sizeof(int), st));
        return fail(MUSE_ERR_CUDA, "muse_batch_run_exchange: a peer did not deliver its records within the time limit");
    }
    const muse_partial *recs = reinterpret_cast<const muse_partial *>(x->h_recs.get());
    if (top_n > 0 && recs[0].flags == 2)
        return fail(MUSE_ERR_UNSUPPORTED, "host path needed: a shard's record list was too long for the device-side select or merge");
    *n_out = records_out(recs, top_n, scores, lags, series_idx);
    return MUSE_OK;
}

extern "C" int muse_batch_run_exchange(muse_batch *b, muse_exchange *x, int64_t max_lag, int64_t top_n, double threshold,
                                       int32_t sign_filter, int32_t mode, double *scores, int64_t *lags, int64_t *series_idx,
                                       int64_t *n_out) {
    return muse_batch_run_exchange_ex(b, x, nullptr, 0, max_lag, top_n, threshold, sign_filter, mode, scores, lags, series_idx, n_out);
}

// ---- many references against a sharded store (ungrouped) ----------------------------------------------------------------
// Send table of one step: [MUSE_MULTI_GROUP] record counts, then [capacity] records (q * top_n + j), so that the counts and
// the step's records go to the device in ONE copy.  The pinned copy has [world] flag words behind it (read back per step).
static size_t multi_send_bytes(const muse_exchange *x) {
    return (size_t)MUSE_MULTI_GROUP * sizeof(long long) + (size_t)x->capacity * sizeof(PartialRec);
}

static int multi_send_alloc(muse_exchange *x) {
    CU(x->d_send.grow((int64_t)multi_send_bytes(x)));
    CU(x->h_send.grow((int64_t)(multi_send_bytes(x) + (size_t)x->world * sizeof(unsigned long long))));
    return MUSE_OK;
}

// Steps of q_step = min(MUSE_MULTI_GROUP, capacity / top_n) queries, one epoch each: muse_multi_run on the shard, this rank's
// lists into the send table, push to every rank, wait for every rank's flag, per-query merge on the device, merged lists back.
// The number of steps depends only on n_refs, top_n and the capacity, which every rank shares.  Every check that could fail
// on one rank alone comes before the first epoch; a local failure after that still takes part in its step, with the failure
// marker instead of records, so that every rank leaves in that same step.
extern "C" int muse_multi_run_exchange(muse_group *g, muse_exchange *x, const double *refs, int64_t n_refs, int64_t ref_len,
                                       int64_t max_lag, int64_t top_n, double threshold, int32_t sign_filter, int32_t mode,
                                       double *scores, int64_t *lags, int64_t *series_idx, int64_t *n_out) {
    if (!g || !x || (!refs && n_refs > 0) || !n_out) return fail(MUSE_ERR_INVALID_ARG, "muse_multi_run_exchange: NULL argument");
    if (n_refs < 0 || top_n < 0)
        return fail(MUSE_ERR_INVALID_ARG, "muse_multi_run_exchange: n_refs %lld, top_n %lld", (long long)n_refs, (long long)top_n);
    int rc = check_run_outputs("muse_multi_run_exchange", n_out, top_n, scores, lags, series_idx, nullptr, 0);
    if (rc) return rc;
    if (x->ctx != g->ctx) return fail(MUSE_ERR_INVALID_ARG, "muse_multi_run_exchange: exchange and store belong to different contexts");
    if (!x->opened) return fail(MUSE_ERR_INVALID_ARG, "muse_exchange_open_peers has not been called");
    if (top_n > x->capacity) return fail(MUSE_ERR_INVALID_ARG, "exchange capacity %lld < top_n %lld", (long long)x->capacity, (long long)top_n);
    if (ref_len != g->N)      // muse_batch.go:24-28
        return fail(MUSE_ERR_LENGTH_MISMATCH, "reference has length %lld, the comparison group %lld", (long long)ref_len, (long long)g->N);
    muse_ctx *ctx = x->ctx;
    if (top_n == 0)           // nothing to exchange: every rank's answer (no records; -1 for a std-zero reference) is the same
        return muse_multi_run(ctx, g, refs, n_refs, ref_len, nullptr, 0, max_lag, 0, threshold, sign_filter, mode, scores, lags,
                              series_idx, n_out);
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const int64_t q_step = std::min<int64_t>(MUSE_MULTI_GROUP, x->capacity / top_n);
    int local_rc = multi_send_alloc(x);          // a failure from here on is this rank's failure in the current step
    for (int64_t q0 = 0; q0 < n_refs; q0 += q_step) {
        const int nq = (int)std::min<int64_t>(q_step, n_refs - q0);
        double *sc = scores + (size_t)q0 * (size_t)top_n;
        int64_t *lg = lags + (size_t)q0 * (size_t)top_n, *ix = series_idx + (size_t)q0 * (size_t)top_n, *no = n_out + q0;
        long long *h_cnt = reinterpret_cast<long long *>(x->h_send.get());
        PartialRec *h_tab = reinterpret_cast<PartialRec *>(x->h_send + (size_t)MUSE_MULTI_GROUP * sizeof(long long));
        const unsigned long long *h_flags = reinterpret_cast<const unsigned long long *>(x->h_send + multi_send_bytes(x));
        if (local_rc == MUSE_OK)
            local_rc = muse_multi_run(ctx, g, refs + (size_t)q0 * (size_t)ref_len, nq, ref_len, nullptr, 0, max_lag, top_n, threshold,
                                      sign_filter, mode, sc, lg, ix, no);
        if (local_rc == MUSE_OK) {
            for (int q = 0; q < nq; q++) {
                h_cnt[q] = std::max<int64_t>(no[q], 0);
                for (int64_t k = 0; k < h_cnt[q]; k++) {
                    const size_t i = (size_t)q * (size_t)top_n + (size_t)k;
                    h_tab[i] = PartialRec{(unsigned long long)ix[i], sc[i], (long long)ix[i], (int)lg[i], 0};
                }
            }
            const cudaError_t e = cudaMemcpyAsync(x->d_send, x->h_send, (size_t)MUSE_MULTI_GROUP * sizeof(long long) + (size_t)nq * (size_t)top_n * sizeof(PartialRec),
                                                  cudaMemcpyHostToDevice, st);
            if (e != cudaSuccess) {
                (void)cudaGetLastError();
                local_rc = fail(MUSE_ERR_CUDA, "muse_multi_run_exchange: send table: %s", cudaGetErrorString(e));
            }
        }
        const ExchangePeers ex = exchange_step(x);
        const long long total = (long long)nq * top_n;
        const unsigned pblocks = (unsigned)std::max<long long>(1, std::min<long long>((total + 255) / 256, (long long)ctx->sm_count * 4));
        const long long *d_cnt = reinterpret_cast<const long long *>(x->d_send.get());
        const PartialRec *d_tab = reinterpret_cast<const PartialRec *>(x->d_send + (size_t)MUSE_MULTI_GROUP * sizeof(long long));
        multi_records_push_kernel<<<pblocks, 256, 0, st>>>(d_tab, d_cnt, nq, (long long)top_n, (long long)x->capacity,
                                                           local_rc != MUSE_OK ? 1 : 0, ex);
        exchange_wait_kernel<<<1, 32, 0, st>>>(ex.flags[x->rank], x->world, x->epoch, MUSE_EXCHANGE_TIMEOUT_CYCLES, x->d_status);
        multi_merge_kernel<<<(unsigned)nq, 256, 0, st>>>(ex.recs[x->rank], x->world, (long long)x->capacity, (long long)top_n, x->d_out, nullptr);
        CU(cudaGetLastError());
        int *h_status = reinterpret_cast<int *>(x->h_recs + (size_t)x->capacity * sizeof(muse_partial));
        CU(cudaMemcpyAsync(x->h_recs, x->d_out, sizeof(muse_partial) * (size_t)total, cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(h_status, x->d_status, sizeof(int), cudaMemcpyDeviceToHost, st));
        if (x->h_send)      // (absent only when its allocation was this rank's failure)
            CU(cudaMemcpyAsync((void *)h_flags, ex.flags[x->rank], sizeof(unsigned long long) * (size_t)x->world, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        if (local_rc != MUSE_OK) return local_rc;
        if (*h_status) {
            CU(cudaMemsetAsync(x->d_status, 0, sizeof(int), st));
            return fail(MUSE_ERR_CUDA, "muse_multi_run_exchange: a peer did not deliver its records within the time limit");
        }
        for (int r = 0; r < x->world; r++)
            if ((h_flags[r] & 0xffffffffull) == MUSE_EXCHANGE_RANK_FAILED)
                return fail(MUSE_ERR_CUDA, "muse_multi_run_exchange: rank %d failed", r);
        const muse_partial *recs = reinterpret_cast<const muse_partial *>(x->h_recs.get());
        for (int q = 0; q < nq; q++) {
            if (no[q] < 0) continue;      // std(ref) == 0 on every rank (muse_batch.go:38-41)
            const size_t row = (size_t)q * (size_t)top_n;
            no[q] = records_out(recs + row, top_n, sc + row, lg + row, ix + row);
        }
    }
    return MUSE_OK;
}

// The merge of muse_multi_run_exchange on lists already gathered into device memory (e.g. by an NCCL all-gather).
extern "C" int muse_merge_partials_many(muse_ctx *ctx, const muse_partial *d_parts, int32_t world, int64_t n_refs, int64_t top_n,
                                        double *scores, int64_t *lags, int64_t *series_idx, int64_t *n_out) {
    if (!ctx || !n_out) return fail(MUSE_ERR_INVALID_ARG, "muse_merge_partials_many: NULL argument");
    if (world < 1 || n_refs < 0 || top_n < 0)
        return fail(MUSE_ERR_INVALID_ARG, "muse_merge_partials_many: world %d, n_refs %lld, top_n %lld", world, (long long)n_refs, (long long)top_n);
    if (n_refs > 0 && top_n > 0 && (!d_parts || !scores || !lags || !series_idx))
        return fail(MUSE_ERR_INVALID_ARG, "muse_merge_partials_many: NULL records or output");
    if (n_refs > 0x7fffffffll) return fail(MUSE_ERR_INVALID_ARG, "muse_merge_partials_many: n_refs %lld", (long long)n_refs);
    for (int64_t q = 0; q < n_refs; q++) n_out[q] = 0;
    if (n_refs == 0 || top_n == 0) return MUSE_OK;
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const size_t n_rec = (size_t)n_refs * (size_t)top_n;
    DevBuf<unsigned char> d;
    CU(d.grow((int64_t)(n_rec * sizeof(PartialRec) + (size_t)n_refs * sizeof(long long))));
    PartialRec *d_out = reinterpret_cast<PartialRec *>(d.get());
    long long *d_n = reinterpret_cast<long long *>(d_out + n_rec);
    std::vector<muse_partial> h(n_rec);
    multi_merge_kernel<<<(unsigned)n_refs, 256, 0, st>>>(reinterpret_cast<const PartialRec *>(d_parts), world, (long long)(n_refs * top_n),
                                                         (long long)top_n, d_out, d_n);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(h.data(), d_out, n_rec * sizeof(PartialRec), cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(n_out, d_n, (size_t)n_refs * sizeof(long long), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    for (size_t i = 0; i < n_rec; i++) {
        scores[i] = h[i].score;
        lags[i] = h[i].lag;
        series_idx[i] = h[i].series_idx;
    }
    return MUSE_OK;
}

extern "C" int muse_batch_last_timing(const muse_batch *cb, muse_timing *out) {
    if (!cb || !out) return fail(MUSE_ERR_INVALID_ARG, "muse_batch_last_timing: NULL argument");
    muse_batch *b = const_cast<muse_batch *>(cb);
    if (b->timing_pending) {     // a device-side run (muse_batch_run_partial_device): finish its bookkeeping now
        CU(cudaSetDevice(b->ctx->device));
        const int rc = finish_pending_timing(b);
        if (rc) return rc;
    }
    *out = b->timing;
    return MUSE_OK;
}
