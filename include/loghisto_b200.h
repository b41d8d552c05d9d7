/*
 * loghisto_b200.h -- C ABI of the B200-native loghisto ingest/reduction engine.
 *
 * This is the drop-in boundary for ONE path of spacejam/loghisto: the bodies of
 *   MetricSystem.Histogram      (metrics.go:273-295)  + compress (metrics.go:316-322)
 *   MetricSystem.Counter        (metrics.go:251-269)
 *   TimerToken.Stop             (metrics.go:242-246)   (its Histogram() call)
 *   collectRawMetrics           (metrics.go:420-479)   (cache swap = snapshot)
 *   processHistograms/percentile(metrics.go:336-418)   + decompress (metrics.go:326-332)
 * The reference has no FFI of its own (it is pure Go); these entry points are
 * what a cgo shim that keeps loghisto's exported Go API binds (INTEGRATION.md).
 *
 * Conventions (mirroring the reference's: ingest never fails loudly, never
 * blocks on consumers, metrics.go:570-573/632-636):
 *   - every function returns an lh_status (0 = LH_OK, negative = error); nothing
 *     throws, nothing calls back into the caller;
 *   - all functions are thread-safe; ingest may run concurrently with a
 *     snapshot (double-buffered bucket arrays);
 *   - `stream` arguments are a cudaStream_t passed as void* (NULL = the
 *     context's own ingest stream); device pointers are plain pointers;
 *   - names never cross the boundary: the caller interns name -> dense id.
 *
 * Bucket layout: one dense uint64[65536] per histogram, indexed by
 * (uint16_t)key where key is the reference's int16 bucket.  Samples whose id is
 * >= max_histograms are dropped and counted (lh_stats.dropped).
 *
 * There is NO CPU fallback: without a CUDA device lh_create fails with
 * LH_ERR_NO_DEVICE.
 */
#ifndef LOGHISTO_B200_H_
#define LOGHISTO_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define LH_API __attribute__((visibility("default")))
#else
#define LH_API
#endif

#define LH_ABI_VERSION 2
#define LH_KEYS_PER_HISTOGRAM 65536
#define LH_MAX_PERCENTILES 32
#define LH_MAX_PRECISION 250     /* buckets per unit of ln(1+|v|); the reference's constant is 100 (metrics.go:40-43) */
#define LH_MAX_RANKS 16          /* GPUs one lh_comm group may span (one node) */
#define LH_PEER_HANDLE_BYTES 1024

typedef int32_t lh_status;
enum {
    LH_OK = 0,
    LH_ERR_INVALID = -1,    /* bad argument */
    LH_ERR_CUDA = -2,       /* a CUDA runtime call failed; see lh_last_error */
    LH_ERR_NOMEM = -3,      /* host or device allocation failed */
    LH_ERR_NO_DEVICE = -4,  /* no usable CUDA device: there is no CPU fallback */
    LH_ERR_STATE = -5,      /* call out of order (e.g. reduce without a snapshot) */
    LH_ERR_RANGE = -6       /* id / size out of the configured range */
};

typedef struct lh_ctx lh_ctx;

typedef struct lh_config {
    uint32_t struct_size;     /* = sizeof(lh_config) */
    int32_t device;           /* CUDA ordinal */
    uint32_t max_histograms;  /* H >= 1: ids 0..H-1 */
    uint32_t max_counters;    /* C >= 1: ids 0..C-1 */
    uint64_t staging_bytes;   /* bytes per pinned staging slot (0 = 32 MiB) */
    uint32_t staging_slots;   /* slots in the ring (0 = 3) */
    uint32_t flags;           /* reserved, 0 */
    uint32_t precision;       /* `precision` of compress/decompress (metrics.go:40-43, 316-332): key =
                               * int16(precision*ln(1+|v|)+0.5).  0 = the reference's 100; 1..LH_MAX_PRECISION */
    uint32_t reserved[3];     /* 0 */
} lh_config;

/* ---- lifecycle ------------------------------------------------------- */
LH_API lh_status lh_create(const lh_config *cfg, lh_ctx **out);
LH_API lh_status lh_destroy(lh_ctx *ctx);
LH_API const char *lh_strerror(lh_status st);
/* Last error detail recorded on this context (thread-unsafe snapshot, for logs). */
LH_API const char *lh_last_error(const lh_ctx *ctx);
LH_API uint32_t lh_abi_version(void);

/* ---- ingest, device-resident inputs ------------------------------------
 * Replaces compress + the map lookup + atomic.AddUint64 of metrics.go:273-295.
 * All launches are asynchronous on `stream`. */

/* n samples of ONE histogram (the single-name loop of print_benchmark.go:59-67). */
LH_API lh_status lh_ingest_f64(lh_ctx *ctx, uint32_t histogram_id, const double *d_values, size_t n,
                        void *stream);
/* (id,value) pairs, the name->histogram dispatch path.  ids are dense ids. */
LH_API lh_status lh_ingest_keyed_f64_u16(lh_ctx *ctx, const uint16_t *d_ids, const double *d_values,
                                  size_t n, void *stream);
LH_API lh_status lh_ingest_keyed_f64_u32(lh_ctx *ctx, const uint32_t *d_ids, const double *d_values,
                                  size_t n, void *stream);
/* Timer samples: value = float64(duration.Nanoseconds()), metrics.go:242-246. */
LH_API lh_status lh_ingest_keyed_i64ns_u16(lh_ctx *ctx, const uint16_t *d_ids, const int64_t *d_nanos,
                                    size_t n, void *stream);

/* A batch of Histogram samples AND a batch of Timer samples (metrics.go:242-246 then :273-295) in one call: above a few
 * million pairs both are binned by ONE launch of the write-combining kernel, so its fixed costs are paid once per batch
 * (configs[4]: 50 % Histogram / 25 % Timer ops).  Same semantics as lh_ingest_keyed_f64_u16 followed by
 * lh_ingest_keyed_i64ns_u16; either count may be 0. */
LH_API lh_status lh_ingest_keyed_pair_u16(lh_ctx *ctx, const uint16_t *d_ids_f64, const double *d_values, size_t n_f64,
                                          const uint16_t *d_ids_ns, const int64_t *d_nanos, size_t n_ns, void *stream);
/* Counter(name, amount), metrics.go:251-269: wrapping uint64 adds. */
LH_API lh_status lh_counter_add_u16(lh_ctx *ctx, const uint16_t *d_ids, const uint64_t *d_amounts,
                             size_t n, void *stream);
LH_API lh_status lh_counter_add_u32(lh_ctx *ctx, const uint32_t *d_ids, const uint64_t *d_amounts,
                             size_t n, void *stream);

/* ---- ingest, host-resident inputs ----------------------------------------
 * Same semantics, inputs in host memory.  Copies are chunked and overlapped
 * with the kernels.  On return the host buffers may be reused; the work may
 * still be in flight on the context's ingest stream. */
LH_API lh_status lh_ingest_f64_host(lh_ctx *ctx, uint32_t histogram_id, const double *h_values, size_t n);
LH_API lh_status lh_ingest_keyed_f64_u16_host(lh_ctx *ctx, const uint16_t *h_ids, const double *h_values,
                                       size_t n);
LH_API lh_status lh_ingest_keyed_i64ns_u16_host(lh_ctx *ctx, const uint16_t *h_ids, const int64_t *h_nanos,
                                         size_t n);
LH_API lh_status lh_counter_add_u16_host(lh_ctx *ctx, const uint16_t *h_ids, const uint64_t *h_amounts,
                                  size_t n);

/* ---- merging snapshots --------------------------------------------------
 * Adds n sparse (histogram id, int16 key, uint64 count) triples -- the format lh_snapshot_export returns -- into
 * the ACTIVE bucket arrays.  Bucket counts are a commutative monoid, so snapshots taken on other hosts or GPUs
 * merge exactly (SURVEY.md section 8f rank 3); it also lets a caller re-reduce a RawMetricSet it holds. */
LH_API lh_status lh_merge_counts_host(lh_ctx *ctx, const uint32_t *h_ids, const int16_t *h_keys,
                                      const uint64_t *h_counts, size_t n);

/* ---- pinned staging ring (the cgo-friendly feed) ------------------------
 * cgo forbids C code from keeping Go pointers after a call returns, so the
 * shim fills C-owned pinned memory instead.  A slot of `staging_bytes` is laid
 * out by the caller as it likes and committed with one of the calls below,
 * which enqueue H2D + kernel and recycle the slot when the copy has landed.
 * lh_staging_acquire blocks only when every slot is still in flight. */
typedef struct lh_staging {
    void *host;        /* pinned host memory, `bytes` long, 256-byte aligned */
    uint64_t bytes;
    uint32_t slot;
    uint32_t reserved;
} lh_staging;
LH_API lh_status lh_staging_acquire(lh_ctx *ctx, lh_staging *out);
/* slot holds n float64 values of one histogram */
LH_API lh_status lh_staging_commit_f64(lh_ctx *ctx, const lh_staging *s, uint32_t histogram_id, size_t n);
/* slot holds n float64 values at offset 0 followed, at byte offset
 * ids_offset (multiple of 16), by n uint16 ids */
LH_API lh_status lh_staging_commit_keyed_f64_u16(lh_ctx *ctx, const lh_staging *s, size_t n,
                                          uint64_t ids_offset);
/* slot holds n uint64 amounts at offset 0 and n uint16 ids at ids_offset */
LH_API lh_status lh_staging_commit_counter_u16(lh_ctx *ctx, const lh_staging *s, size_t n,
                                        uint64_t ids_offset);
/* give a slot back unused */
LH_API lh_status lh_staging_abandon(lh_ctx *ctx, const lh_staging *s);

/* ---- snapshot = collectRawMetrics' cache swap (metrics.go:425-428, 460-463)
 *
 * lh_snapshot_begin   freezes the active bucket/counter arrays and makes the
 *                     spare (zeroed) pair active; ingest continues unblocked.
 * lh_snapshot_device  exposes the frozen device arrays so a multi-GPU caller
 *                     can all-reduce them in place (sum of uint64) before
 *                     reducing; work must be ordered on the returned stream.
 * lh_snapshot_reduce  processHistograms for every histogram (count, sum, avg,
 *                     percentiles), results copied to caller arrays.
 * lh_snapshot_export  sparse (key,count) lists + counter deltas, enough to
 *                     rebuild RawMetricSet.Histograms / Rates exactly.
 * lh_snapshot_end     zeroes the frozen arrays and returns them to the pool.
 */
typedef struct lh_device_view {
    uint64_t *d_buckets;   /* [max_histograms][65536] */
    uint64_t *d_counters;  /* [max_counters] interval deltas */
    uint64_t n_bucket_words;
    uint64_t n_counter_words;
    void *stream;          /* cudaStream_t the snapshot work is ordered on */
    uint32_t *d_flags;     /* [max_histograms] 0 = untouched this interval, 1 = counts inside the fast window only,
                            * 3 = also outside it.  A caller that reduces d_buckets in place across GPUs must reduce
                            * these with MAX (= bitwise OR) too: the reduction / export kernels scan only what the
                            * flags cover */
    uint64_t n_flag_words;
} lh_device_view;

LH_API lh_status lh_snapshot_begin(lh_ctx *ctx);
LH_API lh_status lh_snapshot_device(lh_ctx *ctx, lh_device_view *out);

/* Output arrays are caller-allocated host memory:
 *   counts[H]           exact uint64 totals (0 => histogram absent this interval)
 *   sums[H], avgs[H]    as the reference's float64 map values (avg NaN when count==0)
 *   pkeys[H*np]         chosen bucket key per percentile, INT32_MIN where the
 *                       reference's percentile() returns its error (p>1, NaN)
 *   pvals[H*np]         decompress(key); NaN where pkeys is INT32_MIN
 * Any output pointer may be NULL to skip it. */
LH_API lh_status lh_snapshot_reduce(lh_ctx *ctx, const double *percentiles, uint32_t np,
                             uint64_t *counts, double *sums, double *avgs, int32_t *pkeys,
                             double *pvals);

/* Asynchronous form for pipelined callers (the reaper overlaps the next interval's ingest with this
 * interval's reduction): enqueue the reduction of the open snapshot and get a ticket.  The frozen
 * arrays may be released with lh_snapshot_end right away; lh_snapshot_result waits for the ticket and
 * copies its results out.  Two tickets may be in flight; a ticket expires when the second-next is issued. */
LH_API lh_status lh_snapshot_reduce_async(lh_ctx *ctx, const double *percentiles, uint32_t np, uint64_t *ticket);
LH_API lh_status lh_snapshot_result(lh_ctx *ctx, uint64_t ticket, uint64_t *counts, double *sums, double *avgs,
                                    int32_t *pkeys, double *pvals);

typedef struct lh_sparse {
    const uint32_t *offsets;   /* [H+1] prefix offsets into keys/counts */
    const int16_t *keys;       /* ascending per histogram */
    const uint64_t *counts;
    const uint64_t *counter_deltas; /* [max_counters] */
    uint64_t total_entries;
} lh_sparse;
/* Pointers stay valid until the next lh_snapshot_export / lh_destroy. */
LH_API lh_status lh_snapshot_export(lh_ctx *ctx, lh_sparse *out);
/* Dense copy of one frozen histogram into host memory (uint64[65536]). */
LH_API lh_status lh_snapshot_copy_histogram(lh_ctx *ctx, uint32_t histogram_id, uint64_t *h_out65536);
LH_API lh_status lh_snapshot_end(lh_ctx *ctx);

/* ---- multi-GPU: sharded sample stream, bucket arrays summed at snapshot time (SURVEY.md section 8e) -------------
 * One context per GPU (one process per GPU, or one thread per GPU in one process).  Each rank ingests its shard
 * into its own arrays; between lh_snapshot_begin and the reduction, lh_snapshot_allreduce sums the live window of
 * every rank's frozen arrays into this rank's view of the snapshot with ONE small kernel that reads the peers'
 * memory directly over NVLink (peer mappings: CUDA IPC between processes, peer access inside one process) -- no
 * library collective, nothing to link.  uint64 sums are associative, so every rank ends with exactly the bucket
 * counts a single GPU would have produced (metrics.go:273-295 over the whole stream).
 *
 *   lh_comm_export   opaque handle describing this context's arrays; the host exchanges the handles of all ranks
 *                    by any means it has (a file, a pipe, MPI, torch.distributed, Go channels in one process)
 *   lh_comm_import   maps every peer; handles[rank] must be this context's own.  Collective: every rank calls it
 *                    before any rank calls lh_snapshot_allreduce
 *   lh_snapshot_allreduce  collective, between lh_snapshot_begin and lh_snapshot_reduce/_export: ranks must take
 *                    their snapshots in lock-step (same number, same order).  Enqueued on the snapshot stream; the
 *                    kernel waits on the device for the peers' frozen arrays (no host synchronisation) and returns
 *                    LH_OK immediately.  A peer that never arrives makes the kernel give up after 10 s; that is
 *                    reported by lh_comm_info.status != 0 (the snapshot's counts are then this rank's own only)
 *   lh_comm_allreduce_ms   device time of all-reduce `seq` (CUDA events around the kernel on the snapshot stream)
 */
typedef struct lh_peer_handle { uint8_t bytes[LH_PEER_HANDLE_BYTES]; } lh_peer_handle;
typedef struct lh_comm_stats {
    uint32_t rank, world;
    uint32_t status;                 /* 0 ok, 1 a peer did not arrive in time, 2 peers froze different buffers */
    uint32_t reserved;
    uint64_t allreduces;
    uint64_t last_bytes_from_peers;  /* bytes read over NVLink by the most recent all-reduce */
} lh_comm_stats;
LH_API lh_status lh_comm_export(lh_ctx *ctx, lh_peer_handle *out);
LH_API lh_status lh_comm_import(lh_ctx *ctx, uint32_t rank, uint32_t world, const lh_peer_handle *handles);
LH_API lh_status lh_snapshot_allreduce(lh_ctx *ctx, uint32_t include_counters, uint64_t *seq);
LH_API lh_status lh_comm_allreduce_ms(lh_ctx *ctx, uint64_t seq, float *ms);
LH_API lh_status lh_comm_info(lh_ctx *ctx, lh_comm_stats *out);

/* ---- windows: statistics over more than one interval, kept on the device ------------------------------------------
 * One optional accumulator per context, off until lh_window_configure.  It holds the uint64 bucket sums (and counter
 * sums) of
 *   intervals = K (1..LH_MAX_WINDOW_INTERVALS)  the last K folded snapshots (sliding window), or
 *   intervals = 0                               every snapshot folded since it was configured (lifetime).
 *
 *   lh_window_configure  (re)allocate and zero; LH_ERR_STATE while a snapshot is open.  The dense accumulator takes
 *                        H * 512 KiB of device memory.
 *   lh_window_release    free it; window calls then return LH_ERR_STATE until the next configure
 *   lh_window_fold       between lh_snapshot_begin (+ lh_snapshot_allreduce, or an in-place reduction through
 *                        lh_snapshot_device) and lh_snapshot_end, at most once per snapshot: adds what the open
 *                        snapshot's reduction reads (the all-ranks sums after lh_snapshot_allreduce) and, when the
 *                        window is full, subtracts the snapshot folded K folds earlier.  uint64 adds and subtracts are
 *                        exact mod 2^64: a histogram that leaves the window comes back to all-zero cells.  One
 *                        snapshot-stream synchronisation (the size of the sparse copy kept for the eviction).
 *   lh_window_reduce     processHistograms over the window, with or without an open snapshot; same outputs and
 *                        conventions as lh_snapshot_reduce (a histogram absent from every held interval is absent)
 *   lh_window_export     the window as sparse lists; counter_deltas = counter sums over the window.  Pointers stay
 *                        valid until the next lh_window_export / lh_window_release / lh_window_configure / lh_destroy
 * Window calls never touch the snapshot's own results: outstanding lh_snapshot_reduce_async tickets and the buffers
 * of lh_snapshot_export stay as they were. */
#define LH_MAX_WINDOW_INTERVALS 1024
typedef struct lh_window_stats {
    uint32_t intervals;      /* configured K; 0 = lifetime */
    uint32_t held;           /* snapshots currently inside the window (<= K) */
    uint64_t folds;          /* lh_window_fold calls since the last configure */
    uint64_t entries_held;   /* sparse (key,count) entries kept for eviction */
    uint64_t device_bytes;   /* device memory the window holds */
} lh_window_stats;
LH_API lh_status lh_window_configure(lh_ctx *ctx, uint32_t intervals);
LH_API lh_status lh_window_release(lh_ctx *ctx);
LH_API lh_status lh_window_fold(lh_ctx *ctx);
LH_API lh_status lh_window_reduce(lh_ctx *ctx, const double *percentiles, uint32_t np, uint64_t *counts,
                                  double *sums, double *avgs, int32_t *pkeys, double *pvals);
LH_API lh_status lh_window_export(lh_ctx *ctx, lh_sparse *out);
LH_API lh_status lh_window_info(lh_ctx *ctx, lh_window_stats *out);

/* ---- scalar helpers, evaluated ON THE DEVICE (parity probes for tests) --- */
/* out[i] = compress(values[i]) exactly as the ingest kernels compute it
 * (mode 0: production fast path + exact fallback; mode 1: exact path only) */
LH_API lh_status lh_compress_f64(lh_ctx *ctx, const double *d_values, size_t n, int16_t *d_out, int mode,
                          void *stream);
/* copy of the device decompress table: out[(uint16)key] = decompress(key) */
LH_API lh_status lh_decompress_table(lh_ctx *ctx, double *h_out65536);
/* max |fast-path estimate - exact 100*ln(1+|v|)| over the inputs, in bucket
 * units, restricted to samples the fast path accepts; margin evidence for EPS */
LH_API lh_status lh_fastpath_margin(lh_ctx *ctx, const double *d_values, size_t n, double *h_max_err,
                             uint64_t *h_n_slow, void *stream);
/* the same per estimator (1: fast_candidate, 2: the packed-FP32 form of the single-histogram kernels), for the
 * inputs of the last lh_fastpath_margin call */
LH_API lh_status lh_fastpath_margin_detail(lh_ctx *ctx, double *h_err_estimator1, double *h_err_estimator2);

/* ---- synthetic streams (bench / tests; SURVEY.md section 8d) ------------- */
/* kind: 0=U log-uniform, 1=L latency-like, 2=S signed/edge mix, 3=C constant, 4=Z heavy hitter,
 *       6=timer durations (int64 ns bit patterns), 7=counter amounts 1..16, 8=N (stream U with a random sign) */
LH_API lh_status lh_gen_stream_f64(lh_ctx *ctx, int kind, uint64_t seed, uint64_t start, size_t n,
                            double *d_out, void *stream);
LH_API lh_status lh_gen_ids_u16(lh_ctx *ctx, int kind, uint64_t seed, uint64_t start, size_t n,
                         uint32_t n_ids, uint16_t *d_out, void *stream);

/* ---- misc ---------------------------------------------------------------- */
typedef struct lh_stats {
    uint64_t samples;        /* samples accepted by ingest calls (host-side tally) */
    uint64_t counter_ops;
    uint64_t dropped;        /* samples with id out of range (device-side tally) */
    uint64_t kernel_launches;
    uint64_t h2d_bytes;
    uint64_t d2h_bytes;
    uint64_t snapshots;
} lh_stats;
LH_API lh_status lh_get_stats(lh_ctx *ctx, lh_stats *out);
/* wait for all work issued through this context */
LH_API lh_status lh_sync(lh_ctx *ctx);
/* cudaStream_t of the context's own ingest stream, as void* */
LH_API void *lh_ingest_stream(lh_ctx *ctx);
/* device allocation helpers so non-CUDA hosts (ctypes, cgo) can own device buffers */
LH_API lh_status lh_device_alloc(lh_ctx *ctx, size_t bytes, void **d_out);
LH_API lh_status lh_device_free(lh_ctx *ctx, void *d_ptr);
LH_API lh_status lh_host_alloc_pinned(lh_ctx *ctx, size_t bytes, void **h_out);
LH_API lh_status lh_host_free_pinned(lh_ctx *ctx, void *h_ptr);
LH_API lh_status lh_memcpy_h2d(lh_ctx *ctx, void *d_dst, const void *h_src, size_t bytes);
LH_API lh_status lh_memcpy_d2h(lh_ctx *ctx, void *h_dst, const void *d_src, size_t bytes);
/* kernel-variant selection for profiling: key "k1" -> variant number,
 * "k1_grid_mult", "k1_reserve_sms" (SMs the ingest kernels leave free so that a concurrent
 * snapshot / all-reduce kernel can run beside them), "keyed_blocks_per_sm", "keyed_mode" (0 auto, 1 L2-atomic
 * kernel, 2 owner-partitioned write-combining kernel whatever the batch size), and that kernel's knobs: "kp_chunk"
 * (samples per chunk, default 256 M), "wc_spt" (tile shape code: 6 = 896 threads x 4 samples (default), 4 = 1024 x 4,
 * 3 = 768 x 4, 8 = 512 x 8), "wc_flush" (samples a CTA bins between two flushes of its owner buffers, default 24576),
 * "wc_pf" (L2 prefetch distance of its input in tiles, default 1, 0 = off) */
LH_API lh_status lh_tune(lh_ctx *ctx, const char *key, int64_t value);
LH_API int32_t lh_k1_variant_count(void);
LH_API int32_t lh_k1_variant_current(lh_ctx *ctx);
LH_API const char *lh_k1_variant_name(lh_ctx *ctx, int32_t i);
/* name of the kernel the most recent keyed ingest dispatched to */
LH_API const char *lh_keyed_kernel_name(lh_ctx *ctx);
/* time the last `lh_ingest_*` launch range on its stream: CUDA events bracket
 * every ingest kernel; returns the device time of the most recent one in ms */
LH_API lh_status lh_last_kernel_ms(lh_ctx *ctx, float *ms);
/* lh_ingest_seq = number of ingest calls issued so far (1-based sequence number of the latest);
 * lh_kernel_ms = device time of ingest call `seq` (its events stay available for the next 15 calls) */
LH_API uint64_t lh_ingest_seq(lh_ctx *ctx);
LH_API lh_status lh_kernel_ms(lh_ctx *ctx, uint64_t seq, float *ms);

#ifdef __cplusplus
}
#endif
#endif /* LOGHISTO_B200_H_ */
