/*
 * muse_b200.h -- C ABI of the B200-native go-muse Batch.Run hot path.
 *
 * This is the drop-in boundary: a Go facade that keeps go-muse's exported API
 * (NewSeries / NewGroup / Group.Add / NewBatch / Batch.Run / Results.Fetch) binds
 * exactly these entry points through cgo (INTEGRATION.md shows the stub).  The
 * reference has no FFI of its own -- it is a pure-Go package -- so every entry
 * point cites the Go function (file:line in aouyang1/go-muse) whose work it
 * takes over.
 *
 * Conventions
 *   - plain pointers and sizes only; opaque handles; no C++/torch types.
 *   - every call returns an int status (MUSE_OK == 0); muse_last_error() gives
 *     the message of the calling thread's last failure.  Nothing throws.
 *   - host buffers passed in are COPIED before the call returns (cgo may not
 *     retain Go pointers); host output buffers are owned by the caller.
 *   - calls may come from any OS thread (the library selects the device on
 *     entry); calls on ONE group/batch must not overlap in time.
 *   - strings never cross the boundary: label values are dictionary-encoded to
 *     int32 ids by the host facade (id < 0 == "series does not have this key").
 *   - there is no CPU fallback: without a CUDA device muse_ctx_create fails.
 */
#ifndef MUSE_B200_H
#define MUSE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MUSE_OK                  0
#define MUSE_ERR_INVALID_ARG     1
#define MUSE_ERR_CUDA            2
#define MUSE_ERR_LENGTH_MISMATCH 3  /* muse_batch.go:24-28, group.go:45-51 */
#define MUSE_ERR_STDDEV_ZERO     4  /* muse_batch.go:38-41 "Invalid input query" */
#define MUSE_ERR_NO_DEVICE       5
#define MUSE_ERR_UNSUPPORTED     6  /* e.g. nextPowOf2(len) > MUSE_MAX_FFT_LEN, group-by keys that need more than 64 key bits */
#define MUSE_ERR_OUT_OF_MEMORY   7

#define MUSE_MAX_FFT_LEN (1 << 24)        /* n = nextPowOf2(series length), xcorr.go:19-24: 16 M samples per series */
#define MUSE_MAX_FUSED_FFT_LEN 16384      /* up to here one fused kernel per run; above, FFT passes through global memory */

/* results.go:20-26 */
#define MUSE_SIGN_ANY  0
#define MUSE_SIGN_POS  1
#define MUSE_SIGN_NEG -1

/* muse_batch_run_ex() modes: how the per-series scores are produced */
#define MUSE_MODE_AUTO   0  /* screened when the shape has a screening kernel, else exact */
#define MUSE_MODE_EXACT  1  /* every series through the fp64 kernel */
#define MUSE_MODE_SCREEN 2  /* fp32 spectral upper bound for all + fp64 re-score of survivors;
                               results are identical to MUSE_MODE_EXACT */

typedef struct muse_ctx   muse_ctx;    /* one device, its streams and scratch */
typedef struct muse_group muse_group;  /* series store: group.go:7-12 Group.registry */
typedef struct muse_batch muse_batch;  /* muse_batch.go:13-19 Batch (n, x, Comparison) */

/* One (group, representative) record; the unit exchanged between GPUs.
 * muse_batch.go:79-89: the Score a scoreSingle goroutine sends for its group. */
typedef struct muse_partial {
    uint64_t group_key;   /* packed label-id key of the group (series index when ungrouped) */
    double   score;       /* min(|peak|, 1), muse_batch.go:74-77 */
    int64_t  series_idx;  /* GLOBAL index of the representative series */
    int32_t  lag;         /* xcorr.go:189-194 */
    int32_t  flags;       /* bit0: score is NaN (never passes results.go:46-52) */
} muse_partial;

/* Per-run device timings (CUDA events on the library's own stream). */
typedef struct muse_timing {
    float total_ms;        /* first launch -> results on host */
    float score_ms;        /* the dominant full-slab kernel (exact or screening pass) */
    float rescore_ms;      /* fp64 re-scoring of screened survivors (0 in exact mode) */
    float select_ms;       /* group max + filter + top-N */
    int64_t n_rescored;    /* series that went through the fp64 kernel after screening */
    int64_t n_refined;     /* series that took the fused fp32 second stage (inverse transform) */
    int32_t mode;          /* MUSE_MODE_EXACT or MUSE_MODE_SCREEN actually used */
    int32_t n_launches;    /* kernels launched by this run */
} muse_timing;

const char *muse_last_error(void);
const char *muse_version(void);

/* ---- context --------------------------------------------------------------- */
int  muse_ctx_create(int device, muse_ctx **out);
void muse_ctx_destroy(muse_ctx *ctx);
int  muse_ctx_synchronize(muse_ctx *ctx);
/* Run all of this context's work on the caller's CUDA stream (a cudaStream_t, e.g. the
 * host framework's current stream) instead of the context's own; NULL restores it. */
int  muse_ctx_set_stream(muse_ctx *ctx, void *cuda_stream);
/* Page-locked host memory for rows handed to muse_group_append (full-rate DMA). */
int  muse_host_alloc(void **out, int64_t bytes);
void muse_host_free(void *p);
/* Bytes of device and of page-locked host memory the library holds right now, in this process, over every context
 * (memory of muse_host_alloc belongs to the caller and is not counted).  When every handle is destroyed both are 0. */
int  muse_held_bytes(int64_t *device_bytes, int64_t *pinned_bytes);

/* ---- series store ----------------------------------------------------------
 * Replaces Group{registry} + Series{y, labels} (group.go:7-56, series.go:8-42):
 * a device-resident fp64 slab, one 128-byte-aligned row per series, plus an
 * int32 label-id table [n_label_keys][capacity] (SoA).  Duplicate-UID and
 * empty-label checks (group.go:33-41) stay in the host facade, which owns the
 * strings.  capacity_hint is a reservation, the store grows on demand. */
int  muse_group_create(muse_ctx *ctx, int64_t series_len, int32_t n_label_keys,
                       int64_t capacity_hint, muse_group **out);
void muse_group_destroy(muse_group *g);

/* Group.Add (group.go:31-56): append n_series rows (row-major [n_series][series_len]
 * fp64, HOST memory) and their label ids ([n_series][n_label_keys], may be NULL
 * when n_label_keys == 0).  series_len must equal the group's (group.go:45-51 ->
 * MUSE_ERR_LENGTH_MISMATCH).  Rows in page-locked memory (muse_host_alloc, cudaHostRegister) are copied by one DMA; rows in
 * pageable memory (a Go slice, a numpy array) go through the context's ring of three pinned 64 MB buffers, filled by several
 * host threads (MUSE_STAGE_THREADS, default min(cores, 12)) while the previous chunk is on the wire.  The row statistics of the
 * new rows (mean, 1/std: the z-normalisation of xcorr.go:84-95, once per row instead of once per Run) are computed by a kernel
 * queued behind the copy.  Everything is complete when the call returns. */
int  muse_group_append(muse_group *g, const double *rows, int64_t n_series, int64_t series_len,
                       const int32_t *label_ids);

/* Same, from DEVICE memory already on the context's device (row-major rows). */
int  muse_group_append_device(muse_group *g, const double *d_rows, int64_t n_series,
                              int64_t series_len, const int32_t *d_label_ids);

/* Synthetic siggen-style rows generated on the device (benchmarks at sizes that do
 * not fit in host memory; SURVEY section 8d config C3/C4).  Series i (global index
 * first_index + k) is kind i%3: rect+noise / line+noise / noise, from a counter-based
 * generator keyed (seed, i, t); muse_synth_row() gives the identical row on the host.
 * Label ids: key 0 = i / 1000 ("graph"), key 1 = i % 1000 ("host") when the group has
 * >= 2 label keys. */
int  muse_group_append_synthetic(muse_group *g, int64_t n_series, uint64_t seed, int64_t first_index);
/* variant 0: the mix above; variant 1: every series a rect of the reference's width (10 samples) at a random position -- the
 * adversarial store for the screening (nearly every score within the slack of the top-N cut-off). */
int  muse_group_append_synthetic_ex(muse_group *g, int64_t n_series, uint64_t seed, int64_t first_index, int32_t variant);
/* Replace the label ids of every series in the store by the synthetic scheme
 * id(key k, global index i) = (i / div[k]) % mod[k], i = global offset + local index (benchmarks:
 * SURVEY section 8d config C4 = {graph: i/10000 % 1000, host: i/100 % 100, colo: i % 100}). */
int  muse_group_set_synthetic_labels(muse_group *g, const int64_t *div, const int64_t *mod);
void muse_synth_row(uint64_t seed, int64_t index, int64_t series_len, double *out_row);
void muse_synth_reference(uint64_t seed, int64_t series_len, double *out_row);

int64_t muse_group_size(const muse_group *g);        /* number of series, len(registry) */
int64_t muse_group_series_len(const muse_group *g);  /* Group.Length(), group.go:24-26 */
/* Global index of this store's first series (multi-GPU shards); default 0. */
int  muse_group_set_global_offset(muse_group *g, int64_t first_global_index);
/* Forget every series but keep the allocation (refill with muse_group_append). */
int  muse_group_clear(muse_group *g);
/* Read rows back to the host: one row, or n_rows consecutive rows (dense [n_rows][len]). */
int  muse_group_read_row(muse_group *g, int64_t local_index, double *out_row);
int  muse_group_read_rows(muse_group *g, int64_t first, int64_t n_rows, double *out_rows);

/* Slide rows [first, first + n_rows) of the store forward by k samples, in place (a window of the last N samples of every
 * series, advanced without sending the store over the link again):
 *     row_i <- row_i[k .. N) ++ samples[i - first][0 .. k)
 * samples: dense [n_rows][k] fp64 HOST rows (pageable or page-locked) / DEVICE rows on the context's device.
 * 0 <= k <= N (k == 0: nothing to do; k == N replaces the rows).  Row statistics (and, for odd N, the pad column) are
 * recomputed, bit-identical to what muse_group_append computes for the same rows; labels, size and global offset are
 * unchanged.  Batches created earlier stay valid and see the new rows.  Everything is complete when the call returns (as
 * muse_group_append).  Argument errors (NULL g; NULL samples with k > 0 and n_rows > 0; k < 0 or k > N; a row range outside
 * [0, size)) return MUSE_ERR_INVALID_ARG before any device work and leave the store untouched.  Host samples reach the device
 * in chunks of whole rows of at most 64 MB (page-locked: copied directly; pageable: through the pinned staging ring of
 * muse_group_append), so k may not exceed 8 M samples there (MUSE_ERR_UNSUPPORTED). */
int  muse_group_roll(muse_group *g, int64_t first, int64_t n_rows, const double *samples, int64_t k);
int  muse_group_roll_device(muse_group *g, int64_t first, int64_t n_rows, const double *d_samples, int64_t k);

/* ---- batch -----------------------------------------------------------------
 * NewBatch (muse_batch.go:23-52): checks ref_len against the group
 * (MUSE_ERR_LENGTH_MISMATCH), n = nextPowOf2(ref_len), computes on the device
 * X = rfft(zeroPad(zNormalize(ref)/(N-1), n)); std(ref)==0 -> MUSE_ERR_STDDEV_ZERO.
 * The reference row is copied; unlike go-muse nothing is mutated in place.
 * n <= MUSE_MAX_FUSED_FFT_LEN: one fused kernel scores a series from its row (fp32 screening for n = 128 .. 16384).
 * Above (go-muse has no limit; BenchmarkXCorrWithX is n = 32768, xcorr_test.go:330-348): every series is scored in fp64 by
 * FFT passes through global memory, two series per complex transform, 256 MB of work space at a time. */
int  muse_batch_create(muse_ctx *ctx, muse_group *g, const double *ref, int64_t ref_len,
                       muse_batch **out);
void muse_batch_destroy(muse_batch *b);
int64_t muse_batch_fft_len(const muse_batch *b);     /* Batch.n */

/* Batch.Run + Results filter/top-N for one Run on a fresh Results
 * (muse_batch.go:99-130, results.go:46-87).
 *   key_cols[n_key_cols]: label-key columns to group by (Group.indexLabelValues,
 *       group.go:76-104); n_key_cols == 0: every series is its own group.  Up to 16
 *       columns whose cardinalities fit 64 key bits together (else MUSE_ERR_UNSUPPORTED);
 *       a store holds up to 64 label-key columns.
 *   per group the member with the highest min(|peak|,1) is kept BEFORE the filter
 *   (muse_batch.go:87-89, lowest series index wins ties), then |lag| <= max_lag,
 *   score >= threshold and the sign filter are applied (results.go:46-52) and the
 *   top_n by score are returned in DESCENDING order (results.go:81-85), ties by
 *   ascending series index.
 * Outputs (host, capacity top_n each): scores, lags, series_idx (global index of
 * the representative series -> the facade maps it to that series' *Labels,
 * muse_batch.go:80); *n_out = number written. */
int  muse_batch_run(muse_batch *b, const int32_t *key_cols, int32_t n_key_cols,
                    int64_t max_lag, int64_t top_n, double threshold, int32_t sign_filter,
                    double *scores, int64_t *lags, int64_t *series_idx, int64_t *n_out);

/* As muse_batch_run with an explicit scoring mode (MUSE_MODE_*) and signed scores:
 * signed_scores != 0 keeps the sign and clamps to [-1, 1] as Muse.Run does
 * (muse.go:72-76, group max by |score| :86) instead of abs+clamp. */
int  muse_batch_run_ex(muse_batch *b, const int32_t *key_cols, int32_t n_key_cols,
                       int64_t max_lag, int64_t top_n, double threshold, int32_t sign_filter,
                       int32_t mode, int32_t signed_scores,
                       double *scores, int64_t *lags, int64_t *series_idx, int64_t *n_out);

/* Per-series (score, lag) of every series in the store, exact fp64 path
 * (xCorrWithX + abs/clamp per series; what scoreSingle's loop computes,
 * muse_batch.go:68-77).  Host outputs of muse_group_size() entries. */
int  muse_batch_score_all(muse_batch *b, int32_t signed_scores, double *scores, int32_t *lags);

/* Diagnostic: the fp32 screening pass alone.  upper[i] >= series i's score from
 * muse_batch_score_all (a value > 1, e.g. 2.0, means "undecided: ask the fp64 kernel").
 * refine != 0 (FFT lengths 128 .. 16384) sends EVERY series through the fused second stage
 * (fp32 inverse transform) for the lag window max_lag: upper[i] = -1 when the peak is
 * certainly outside the window (the series fails results.go:46-48), else a tight bound;
 * lower[i] >= 0 is a certain lower bound on the score of a series whose lag is certainly
 * inside the window, -1 otherwise.  MUSE_ERR_UNSUPPORTED when the shape has no such kernel. */
int  muse_batch_screen_bounds(muse_batch *b, int32_t refine, int64_t max_lag, float *upper, float *lower);

/* The full cross-correlation vector cc[n] of one series (xcorr.go:160-197's first
 * return value; KAT support).  *std_zero is set when xcorr.go:165-168 applies. */
int  muse_batch_xcorr(muse_batch *b, int64_t local_index, double *cc, int32_t *std_zero);

/* Many reference queries against ONE resident store: what n_refs x (NewBatch + Batch.Run) (muse_batch.go:23-52,
 * :99-130) return, in one call.  refs: host rows [n_refs][ref_len]; outputs: row q of scores / lags / series_idx
 * (capacity top_n each row) and n_out[q] = results of query q, or -1 when reference q has std == 0
 * (muse_batch.go:38-41: NewBatch fails for that query only).  Arguments as muse_batch_run_ex.
 * For FFT length 2048, ungrouped, unsigned runs over >= 16384 series (any size in MUSE_MODE_SCREEN; more than one
 * reference, top_n <= series / 4)
 * the screening bounds of up to 256 references at a time are ONE bf16 contraction on the tensor cores (tcgen05.mma,
 * muse_multi_bounds_tc), the second stages of all of them one launch over the store, and each query then finishes
 * on the exact fp64 kernel like a single run -- results identical to the separate runs.  Other shapes are served as
 * separate batches on the resident store. */
int  muse_multi_run(muse_ctx *ctx, muse_group *g, const double *refs, int64_t n_refs, int64_t ref_len,
                    const int32_t *key_cols, int32_t n_key_cols, int64_t max_lag, int64_t top_n, double threshold,
                    int32_t sign_filter, int32_t mode,
                    double *scores, int64_t *lags, int64_t *series_idx, int64_t *n_out);

/* Totals of the context's last muse_multi_run over all its queries: (series, query) pairs that took the fp32 second stage and
 * pairs re-scored by the fp64 kernel (tensor-core path only; 0 otherwise). */
int  muse_multi_last_stats(const muse_ctx *ctx, int64_t *n_refined, int64_t *n_rescored);

/* Device times (ms) of the last launch group of the tensor-core multi-query path: [0] magnitudes of the store, [1] the bounds
 * contraction (tcgen05), [2] the second stages, [3] the tails (survivors, fp64 re-scoring, filter, top-N). */
int  muse_multi_last_timing(const muse_ctx *ctx, float *ms4);

/* Diagnostic: the screening bounds of n_refs <= 256 reference queries against the whole store as ONE bf16 contraction on the
 * tensor cores (tcgen05.mma, fp32 accumulation in TMEM; the first stage of muse_multi_run for FFT length 2048):
 * upper[q * muse_group_size() + i] >= the score muse_batch_score_all gives series i against reference q (2.0 = undecided).
 * What go-muse computes per reference with one Batch each (muse_batch.go:23-52, :56-93) is bounded here for all of them
 * from one transform of every series. */
int  muse_multi_bounds_tc(muse_ctx *ctx, muse_group *g, const double *refs, int64_t n_refs, int64_t ref_len, float *upper);

/* xCorr(x, y, n, normalize) of xcorr.go:102-153 for ANY n (the FFT kernels above exist for powers of
 * two; the reference's own KATs use n = 5): n' = max(n, x_len, y_len) (:104-106), optional z-normalisation
 * of both inputs (:108-127), LEADING zero pads (:128-129), cc[k] = sum_t xp[(t+k) mod n'] * yp[t], divided
 * by n'-1 when normalised (:139-140 on gonum's unnormalised inverse), arg-max of |cc| with the first index winning and the wrap to
 * (-n'/2, n'/2] (:145-151).  In fp64 on the device, one pair per call: up to 4096 lags by direct evaluation of that sum; above, by
 * FFT passes through global memory -- one transform of length n' when n' is a power of two (BenchmarkXCorr's n = 32768,
 * xcorr_test.go:310-326), else the linear correlation at a power of two >= 2n', folded.  n' <= 2^26.
 * x, y: host rows.  cc (host, may be NULL): n' values when cc_capacity >= n'.  *n_out = n', or 0 with
 * *std_zero = 1, *lag = 0, *value = 0 when a normalised input has std == 0 (:109-126, the reference returns
 * (nil, 0, 0)). */
int  muse_xcorr(muse_ctx *ctx, const double *x, int64_t x_len, const double *y, int64_t y_len, int64_t n,
                int32_t normalize, double *cc, int64_t cc_capacity, int64_t *n_out, int64_t *lag, double *value,
                int32_t *std_zero);

/* ---- multi-GPU: shard-local partials and their merge -------------------------
 * One store per GPU holds a contiguous block of the series (global offset set with
 * muse_group_set_global_offset).  run_partial produces this shard's group
 * representatives BEFORE the filter (SURVEY F2), or -- ungrouped -- its local top_n
 * AFTER the filter; the caller all-gathers the records (NCCL) and every rank calls
 * muse_merge_partials on the concatenation. */
int  muse_batch_run_partial(muse_batch *b, const int32_t *key_cols, int32_t n_key_cols,
                            int64_t max_lag, int64_t top_n, double threshold, int32_t sign_filter,
                            int32_t mode, muse_partial *out, int64_t capacity, int64_t *n_out);
/* Ungrouped shard partials WITHOUT a host round trip: the shard's filtered top_n are written to
 * d_out in DEVICE memory (capacity >= top_n records; the rest padded with flags = 1) by work queued
 * on the context's stream; the call does not synchronise, so an all-gather of the records enqueued
 * on the same stream (muse_ctx_set_stream) follows directly and muse_merge_partials runs on the
 * gathered host copy.  flags == 2 in record 0: the candidate list was too long for the device-side
 * select -- call muse_batch_run_partial instead.  Timings: muse_batch_last_timing. */
int  muse_batch_run_partial_device(muse_batch *b, int64_t max_lag, int64_t top_n, double threshold,
                                   int32_t sign_filter, int32_t mode, muse_partial *d_out, int64_t capacity);
/* ---- multi-GPU exchange over NVLink peer memory (one process per GPU, one box) ------------
 * The shard's top_n records are stored by the selection kernel itself into the receive buffer of EVERY
 * rank (peer pointers from CUDA IPC handles), followed by a system-scope flag; a step is then ONE call:
 * scores, filter, push, wait for the peers, merge -- no library collective and no host code between
 * the kernels.  Setup: every rank creates an exchange, the ranks swap the 64-byte handles of
 * muse_exchange_ipc_handle (any out-of-band channel, e.g. an all-gather of bytes), and each calls
 * muse_exchange_open_peers with the world_size x 64 bytes in rank order.  Ranks must call
 * muse_batch_run_exchange the same number of times (the steps are matched by an epoch counter).
 * MUSE_ERR_UNSUPPORTED: some shard's candidate list was too long for the device-side select -- every
 * rank gets the same answer and can take muse_batch_run_partial + an all-gather instead. */
typedef struct muse_exchange muse_exchange;
int  muse_exchange_create(muse_ctx *ctx, int32_t rank, int32_t world_size, int64_t capacity, muse_exchange **out);
int  muse_exchange_ipc_handle(muse_exchange *x, void *handle64);
int  muse_exchange_open_peers(muse_exchange *x, const void *handles);
void muse_exchange_destroy(muse_exchange *x);
int  muse_batch_run_exchange(muse_batch *b, muse_exchange *x, int64_t max_lag, int64_t top_n, double threshold,
                             int32_t sign_filter, int32_t mode,
                             double *scores, int64_t *lags, int64_t *series_idx, int64_t *n_out);
/* The same step for GROUPED runs (n_key_cols > 0; n_key_cols == 0 is muse_batch_run_exchange): every group representative of the
 * shard, unfiltered (the filter needs the global group max, muse_batch.go:87-89 before results.go:46-52), is pushed to every
 * rank, and the group max across shards, the filter and the top-N run on the device; only top_n records reach the host.  The
 * exchange's capacity must hold the shard's group representatives (at most min(series, groups) of the shard). */
int  muse_batch_run_exchange_ex(muse_batch *b, muse_exchange *x, const int32_t *key_cols, int32_t n_key_cols, int64_t max_lag,
                                int64_t top_n, double threshold, int32_t sign_filter, int32_t mode,
                                double *scores, int64_t *lags, int64_t *series_idx, int64_t *n_out);
/* Many references against a sharded store (ungrouped): what muse_multi_run writes on ONE store holding every shard -- row q
 * of scores / lags / series_idx (capacity top_n each row, global series indices), n_out[q] results or -1 when reference q has
 * std == 0 -- identical on every rank.  The queries go in steps of min(256, capacity / top_n), one exchange epoch each:
 * muse_multi_run on this shard, its per-query top_n lists pushed into every rank's receive buffer, then a per-query merge on
 * the device.  Contract: every rank passes the same references and arguments, and every rank's exchange has the same
 * capacity (the number of steps follows from n_refs, top_n and the capacity alone).  Argument errors (NULLs, top_n > capacity,
 * an exchange whose peers are not open, store and exchange on different contexts, ref_len) are reported before any step
 * begins.  A rank whose local run fails during a step still completes the step with a failure marker and returns its own
 * error; its peers return MUSE_ERR_CUDA ("rank r failed") in that same step.  A sticky CUDA error (a faulted context) cannot
 * be published this way: the peers then return MUSE_ERR_CUDA after the exchange's time limit.  A shard with no series
 * takes part and contributes no records. */
int  muse_multi_run_exchange(muse_group *g, muse_exchange *x, const double *refs, int64_t n_refs, int64_t ref_len,
                             int64_t max_lag, int64_t top_n, double threshold, int32_t sign_filter, int32_t mode,
                             double *scores, int64_t *lags, int64_t *series_idx, int64_t *n_out);
/* The merge of muse_multi_run_exchange for lists gathered by the caller (e.g. an NCCL all-gather, where CUDA IPC is closed).
 * d_parts: DEVICE memory on the context's device, [world][n_refs][top_n] records -- every rank's muse_multi_run rows as
 * muse_partial records (group_key = series_idx, flags 0), each row sorted as muse_multi_run returns it and padded with
 * flags = 1.  Outputs (host) as muse_multi_run; n_out[q] = merged records (a std-zero reference has none: its -1 comes from
 * the caller's own muse_multi_run).  Runs on the context's stream and synchronises it. */
int  muse_merge_partials_many(muse_ctx *ctx, const muse_partial *d_parts, int32_t world, int64_t n_refs, int64_t top_n,
                              double *scores, int64_t *lags, int64_t *series_idx, int64_t *n_out);
/* Upper bound on the records run_partial can emit for these arguments. */
int64_t muse_batch_partial_capacity(muse_batch *b, const int32_t *key_cols, int32_t n_key_cols,
                                    int64_t top_n);
int  muse_merge_partials(const muse_partial *parts, int64_t n_parts,
                         int64_t max_lag, int64_t top_n, double threshold, int32_t sign_filter,
                         double *scores, int64_t *lags, int64_t *series_idx, int64_t *n_out);

/* Timings of the batch's most recent run. */
int  muse_batch_last_timing(const muse_batch *b, muse_timing *out);

#ifdef __cplusplus
}
#endif
#endif /* MUSE_B200_H */
