// lh_api.cu -- C ABI (include/loghisto_b200.h) over the sm_100a kernels.
//
// Host-side bookkeeping only: double-buffered bucket/counter arrays, stream
// and event ordering between ingest and snapshot, the pinned staging ring,
// kernel-variant dispatch.  No bucket arithmetic happens on the CPU.
#include "../../include/loghisto_b200.h"
#include "lh_kernels.cuh"

#include <algorithm>
#include <cmath>
#include <condition_variable>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <vector>
#include <unistd.h>

using namespace lh;

namespace {

struct WriterEvent { cudaStream_t stream; cudaEvent_t ev; };

struct Buffer {
    unsigned long long *d_buckets = nullptr;   // [H][65536]
    unsigned long long *d_counters = nullptr;  // [C]
    uint32_t *d_flags = nullptr;               // [H] 0 untouched / 1 window only / 3 also outside the window
    unsigned int *d_hot = nullptr;             // [hot_replicas][H][2*win] uint32 window of the keyed path
    unsigned long long hot_pending = 0;        // samples added to d_hot since it was last drained
    cudaEvent_t cleared = nullptr;             // zeroing finished
    std::vector<WriterEvent> writers;          // last ingest per stream
};

enum SlotState { SLOT_FREE = 0, SLOT_ACQUIRED = 1 /* handed to the caller (lh_staging_acquire) */, SLOT_INFLIGHT = 2,
                 SLOT_WAITED = 3 /* a thread is waiting for its kernel, mutex released */,
                 SLOT_FILLING = 4 /* lh_*_host is copying pageable memory into it, mutex released */ };
struct Slot {
    void *h = nullptr; void *d = nullptr;
    cudaEvent_t done = nullptr;      // kernel that consumed the slot has finished
    cudaEvent_t copied = nullptr;    // H2D copy into the slot has landed
    int state = SLOT_FREE;
    uint64_t seq = 0;
};

struct K1Variant {
    const char *name;
    void (*launch)(int grid, size_t smem, cudaStream_t s, const double *v32, size_t nvec,
                   const double *head, int nhead, const double *tail, int ntail, unsigned long long *counts,
                   uint32_t *flag, const Prec &pc);
    const void *func;
    int threads;
    size_t smem_fixed;   // bytes besides the sub-histogram (ring + barriers)
    int blocks_per_sm;   // filled at create
    size_t smem;         // filled at create: smem_fixed + sub-histogram for the context's precision
};

template <int THREADS, int UNROLL, int MINB>
void launch_ldg(int grid, size_t smem, cudaStream_t s, const double *v32, size_t nvec, const double *head, int nhead,
                const double *tail, int ntail, unsigned long long *counts, uint32_t *flag, const Prec &pc) {
    k_ingest_single_ldg<THREADS, UNROLL, MINB><<<grid, THREADS, smem, s>>>(v32, nvec, head, nhead, tail, ntail, counts, flag, pc);
}
template <int CW, int STAGES, int STAGE_BYTES, int MINB, bool FOLD>
void launch_bulk(int grid, size_t smem, cudaStream_t s, const double *v32, size_t nvec, const double *head, int nhead,
                 const double *tail, int ntail, unsigned long long *counts, uint32_t *flag, const Prec &pc) {
    k_ingest_single_bulk<CW, STAGES, STAGE_BYTES, MINB, FOLD><<<grid, (CW + 1) * 32, smem, s>>>(v32, nvec, head, nhead, tail, ntail, counts, flag, pc);
}
void launch_probe(int grid, size_t, cudaStream_t s, const double *v32, size_t nvec, const double *head, int nhead,
                  const double *tail, int ntail, unsigned long long *counts, uint32_t *flag, const Prec &pc) {
    k_stream_probe<512, 4><<<grid, 512, 0, s>>>(v32, nvec, head, nhead, tail, ntail, counts, flag, pc);
}

#define LDG_VARIANT(T, U, M) \
    { "ldg256_t" #T "_u" #U "_b" #M, launch_ldg<T, U, M>, (const void *)k_ingest_single_ldg<T, U, M>, T, 0, 0, 0 }
#define BULK_VARIANT(W, S, B, M, F) \
    { "bulk2_w" #W "_s" #S "_" #B "_b" #M "_sign" #F, launch_bulk<W, S, B, M, F != 0>, (const void *)k_ingest_single_bulk<W, S, B, M, F != 0>, (W + 1) * 32, \
      (size_t)S * B + (size_t)S * 16, 0, 0 }

// The shipped kernel plus what the parity tests and profiles/ compare it with (the round-1 sweep of 27 shapes is
// archived in profiles/r01/k1_variants_sustained.txt; only the winners and the independent first version remain).
K1Variant g_k1_variants[] = {
    BULK_VARIANT(16, 4, 32768, 1, 1),   // 0: default (sign folded into the slot)
    BULK_VARIANT(16, 3, 65536, 1, 1),   // 1
    BULK_VARIANT(8, 4, 16384, 2, 1),    // 2
    LDG_VARIANT(512, 2, 2),             // 3: first version (scalar fast_candidate, register double-buffering)
    // 4: read-only diagnostic, produces no counts (never selected by default)
    { "probe_read_only_t512_u4", launch_probe, (const void *)k_stream_probe<512, 4>, 512, 0, 0, 0 },
    BULK_VARIANT(16, 4, 32768, 1, 0),   // 5: negatives flagged to the fix-up instead of folded (2 instructions less per sample)
    BULK_VARIANT(16, 3, 65536, 1, 0),   // 6
};
constexpr int kNumK1Variants = (int)(sizeof(g_k1_variants) / sizeof(g_k1_variants[0]));
constexpr int kDefaultK1Variant = 6;   // 3 x 64 KB stages, negatives through the fix-up: best sustained time on streams U and N (profiles/r02/k1_sustained_r02c.txt)

// Everything the kernels derive from `precision` (metrics.go:40-43), see lh_device.cuh.
Prec make_prec(uint32_t precision) {
    Prec pc{};
    const double P = (double)precision;
    const double c1 = P * 0.6931471805599453094172321;
    pc.precision = P;
    pc.a_int = (uint32_t)std::floor(c1);
    pc.c1 = (float)c1;
    pc.c2 = (float)(c1 - (double)pc.a_int);
    pc.kb = (float)(-1023.0 * (double)pc.c2);
    const float eps = 0.000244140625f * (precision > 100 ? (float)P / 100.0f : 1.0f);
    pc.thresh = 0.5f - eps;
    pc.win = (uint32_t)std::floor(P * 63.0 * 0.6931471805599453094172321 + 0.5) + 1u;
    pc.a4 = pc.a_int * 4u;
    pc.coff = 0u - 1023u * pc.a4 - (0x4B400000u << 2);
    pc.coff0 = 0u - 1023u * pc.a_int - 0x4B400000u;
    return pc;
}

constexpr int kMaxRanks = LH_MAX_RANKS;
constexpr int kCommWords = 2 * LH_MAX_RANKS;       // arrive[16], depart[16]
constexpr uint32_t kPeerMagic = 0x4C485052u;       // "LHPR"

// what lh_comm_export hands to the peers (fits lh_peer_handle)
struct PeerWire {
    uint32_t magic, abi, H, C;
    uint32_t precision, device;
    int64_t pid;
    uint64_t ctx_id;                               // distinguishes contexts of one process
    uint64_t ptr_buckets[2], ptr_flags[2], ptr_counters[2], ptr_comm, ptr_red;
    cudaIpcMemHandle_t ipc_buckets[2], ipc_flags[2], ipc_counters[2], ipc_comm, ipc_red;
};
static_assert(sizeof(PeerWire) <= LH_PEER_HANDLE_BYTES, "lh_peer_handle too small");

struct PeerMap {                                   // one remote rank as mapped into this process
    unsigned long long *buckets[2] = {nullptr, nullptr};
    uint32_t *flags[2] = {nullptr, nullptr};
    unsigned long long *counters[2] = {nullptr, nullptr};
    unsigned long long *comm = nullptr;
    unsigned long long *red = nullptr;             // the rank's REDUCED bucket array: owners of a slice push their sums into it
    bool ipc = false;                              // pointers came from cudaIpcOpenMemHandle (must be closed)
};

// Sparse lists of one view (k_reduce's non-empty counts -> k_scan_nnz -> k_export) and their pinned host mirrors.
// The snapshot and the window each own one set, so neither disturbs what the other handed out.
struct ExportBufs {
    uint32_t *d_nnz = nullptr, *d_offsets = nullptr;   // [H], [H+1]
    uint32_t *h_offsets = nullptr;
    unsigned long long *h_counters = nullptr;          // [C]
    short *d_keys = nullptr, *h_keys = nullptr;
    unsigned long long *d_counts = nullptr, *h_counts = nullptr;
    size_t cap = 0;                                    // entries the key / count buffers hold
};

// One folded snapshot as the window keeps it until it leaves the window (device memory only).
struct WinSlot {
    uint32_t *d_offsets = nullptr;            // [H+1]
    uint32_t *d_flags = nullptr;              // [H]
    unsigned long long *d_counters = nullptr; // [C]
    short *d_keys = nullptr;
    unsigned long long *d_counts = nullptr;
    size_t cap = 0;
    uint64_t entries = 0;
};

struct Window {
    uint32_t intervals = 0;                   // K; 0 = lifetime
    uint64_t folds = 0;
    uint64_t folded_snapshot = 0;             // lh_stats.snapshots of the snapshot folded last (one fold per snapshot)
    unsigned long long *d_acc = nullptr;      // [H][65536]
    uint32_t *d_flags = nullptr;              // [H] 0 / 1 / 3, as a snapshot's
    uint32_t *d_levels = nullptr;             // [2][H] held intervals that touched h at level >= 1, at level 3
    unsigned long long *d_counters = nullptr; // [C]
    // sliding: K + 1 slots, so the capture of fold f never lands on fold f - K before k_window_apply has subtracted
    // it; lifetime: one slot, overwritten by every fold
    std::vector<WinSlot> ring;
    uint32_t *h_total = nullptr;              // pinned: entries of the slot being captured
    double *d_ps = nullptr;
    char *d_res = nullptr, *h_res = nullptr;  // one result slot, laid out as the snapshot's
    bool nnz_valid = false;                   // x.d_nnz holds the accumulator's non-empty counts
    ExportBufs x;
};

}  // namespace

struct lh_ctx {
    lh_config cfg{};
    int device = 0;
    int sm_count = 0;
    uint32_t H = 0, C = 0;
    Prec pc{};
    Buffer buf[2];
    int active = 0;
    bool frozen = false;
    bool nnz_valid = false;
    cudaStream_t ingest_stream = nullptr, snap_stream = nullptr, copy_stream = nullptr;
    double *d_decomp = nullptr;
    unsigned long long *d_dropped = nullptr;
    // reduce / export scratch
    // two result slots (ticket & 1): packed [count H][sum H][avg H][pvals H*np][pkeys H*np]; slot 2 is scratch for
    // lh_snapshot_export when no reduction has produced the non-empty-bucket counts yet (never holds a ticket)
    double *d_ps[3] = {nullptr, nullptr, nullptr};
    char *d_res[3] = {nullptr, nullptr, nullptr};
    char *h_res[3] = {nullptr, nullptr, nullptr};
    cudaEvent_t res_done[3] = {nullptr, nullptr, nullptr};
    uint32_t res_np[3] = {0, 0, 0};
    uint64_t res_ticket[2] = {0, 0};
    uint64_t next_ticket = 1;
    ExportBufs x;                       // lh_snapshot_export's lists (d_nnz also takes every snapshot reduction's counts)
    Window *win = nullptr;              // lh_window_*; null until lh_window_configure
    // staging ring
    std::vector<Slot> slots;
    uint64_t slot_seq = 0;
    size_t staging_bytes = 0;
    // tuning
    unsigned long long last_margin[2] = {0, 0};
    int k1_variant = kDefaultK1Variant;
    int k1_grid_mult = 1;
    int k1_reserve_sms = 0;   // SMs left free for concurrent snapshot / collective kernels
    int keyed_blocks_per_sm = 8;
    uint32_t hot_replicas = 1;          // copies of the hot window (all L2-resident); only the vector RED kernel spreads over them
    int keyed_mode = 0;                 // 0 auto, 1 force L2-atomic kernel, 2 force the write-combining owner kernel
    int64_t kp_chunk = 256 << 20;       // samples per chunk of the owner-partitioned kernel (16 / 32 / 64 / 128 / 256 M: 319 / 339 / 354 / 363 / 368 G samples/s, keyed_pf_probe_r02q/r.txt)
    uint32_t wc_pf_tiles = 1;           // L2 prefetch distance of that kernel's input, in tiles past the one being loaded (0 = off; 1: +12 %)
    uint32_t wc_flush_samples = 24576;  // samples a CTA bins between two flushes of its owner buffers
    int wc_spt = 6;                     // tile shape of that kernel (6: 896 threads x 4 samples; 4: 1024 x 4; 3: 768 x 4; 8: 512 x 8)
    // owner-partitioned keyed kernel scratch (allocated on first use)
    unsigned short *d_kp_queues = nullptr;
    unsigned int *d_kp_cnt = nullptr;     // per-(owner, writer) record counts, then the grid-barrier word
    uint4 *d_kp_rare = nullptr;           // per-CTA lists of samples set aside for the exact path
    size_t kp_cap = 0;
    int kp_parts = 0;
    const char *keyed_kernel = "";       // kernel the last keyed launch used
    // multi-GPU (lh_comm_*): peer mappings of every rank's arrays + this rank's reduced output arrays
    uint32_t comm_rank = 0, comm_world = 0;
    unsigned long long *d_comm = nullptr;         // this rank's comm block (uint64[kCommWords])
    unsigned int *d_comm_aux = nullptr;           // [0] block counter, [1] status
    PeerMap peers[kMaxRanks];
    unsigned long long *d_red_buckets = nullptr;  // [H][65536] sums over ranks (valid for the open snapshot after lh_snapshot_allreduce)
    uint32_t *d_red_flags = nullptr;
    unsigned long long *d_red_counters = nullptr;
    bool view_reduced = false;                    // the open snapshot's reduce/export read the reduced arrays
    bool view_counters_reduced = false;
    uint64_t comm_seq = 0;
    bool comm_two_shot = false;                    // form of the last all-reduce (lh_comm_info's byte count)
    static constexpr int kCommRing = 8;
    cudaEvent_t comm_t0[kCommRing] = {}, comm_t1[kCommRing] = {};
    uint64_t ctx_id = 0;
    K1Variant k1[kNumK1Variants];
    // timing of the most recent ingest kernel
    // CUDA events bracket every ingest launch; a ring keeps the last kTimingRing of them
    static constexpr int kTimingRing = 16;
    cudaEvent_t ev_t0s[kTimingRing] = {}, ev_t1s[kTimingRing] = {};
    cudaEvent_t ev_t0 = nullptr, ev_t1 = nullptr;   // the pair of the launch being issued
    uint64_t ingest_seq = 0;                         // launches issued so far
    bool timing_valid = false;
    // stats
    lh_stats stats{};
    std::mutex mu;
    std::condition_variable slot_cv;     // a staging slot came back (see slot_wait_free)
    std::string last_error;
};

namespace {

lh_status fail(lh_ctx *ctx, lh_status st, const char *what, cudaError_t e = cudaSuccess) {
    if (ctx) {
        char buf[512];
        if (e != cudaSuccess) snprintf(buf, sizeof buf, "%s: %s (%s)", what, cudaGetErrorName(e), cudaGetErrorString(e));
        else snprintf(buf, sizeof buf, "%s", what);
        ctx->last_error = buf;
    }
    return st;
}

#define LH_CUDA(ctx, call)                                                      \
    do {                                                                        \
        cudaError_t _e = (call);                                                \
        if (_e != cudaSuccess) return fail((ctx), LH_ERR_CUDA, #call, _e);      \
    } while (0)

// order `s` after the zeroing of buffer b, and remember `s` as a writer of b
lh_status before_write(lh_ctx *ctx, int b, cudaStream_t s) {
    LH_CUDA(ctx, cudaStreamWaitEvent(s, ctx->buf[b].cleared, 0));
    return LH_OK;
}
lh_status after_write(lh_ctx *ctx, int b, cudaStream_t s) {
    for (auto &w : ctx->buf[b].writers)
        if (w.stream == s) { LH_CUDA(ctx, cudaEventRecord(w.ev, s)); return LH_OK; }
    WriterEvent w{s, nullptr};
    LH_CUDA(ctx, cudaEventCreateWithFlags(&w.ev, cudaEventDisableTiming));
    LH_CUDA(ctx, cudaEventRecord(w.ev, s));
    ctx->buf[b].writers.push_back(w);
    return LH_OK;
}

void next_timing_slot(lh_ctx *ctx) {
    const int i = (int)(ctx->ingest_seq % lh_ctx::kTimingRing);
    ctx->ev_t0 = ctx->ev_t0s[i];
    ctx->ev_t1 = ctx->ev_t1s[i];
    ctx->ingest_seq++;
}

cudaStream_t pick_stream(lh_ctx *ctx, void *stream) { return stream ? (cudaStream_t)stream : ctx->ingest_stream; }

int grid_1d(lh_ctx *ctx, size_t n, int threads, int per_thread, int blocks_per_sm) {
    size_t need = (n + (size_t)threads * per_thread - 1) / ((size_t)threads * per_thread);
    size_t cap = (size_t)ctx->sm_count * blocks_per_sm;
    return (int)std::max<size_t>(1, std::min(need, cap));
}

// ---- K1 dispatch (locked) ----
lh_status launch_single(lh_ctx *ctx, uint32_t hid, const double *d_values, size_t n, cudaStream_t s) {
    if (hid >= ctx->H) return fail(ctx, LH_ERR_RANGE, "histogram_id >= max_histograms");
    if (((uintptr_t)d_values & 7u) != 0) return fail(ctx, LH_ERR_INVALID, "d_values must be 8-byte aligned");
    const int b = ctx->active;
    lh_status st = before_write(ctx, b, s);
    if (st != LH_OK) return st;
    unsigned long long *counts = ctx->buf[b].d_buckets + (size_t)hid * 65536u;
    uint32_t *flag = ctx->buf[b].d_flags + hid;
    const K1Variant &kv = ctx->k1[ctx->k1_variant];
    // a CTA's uint32 sub-histogram must not overflow: tiles are dealt round-robin, so bounding a launch to
    // 2^31 samples per CTA keeps every cell below 2^32 whatever the grid size (reserved SMs shrink it)
    const int grid = std::max(1, ctx->sm_count - ctx->k1_reserve_sms) * kv.blocks_per_sm * ctx->k1_grid_mult;
    const size_t kMaxPerLaunch = std::min((size_t)1 << 36, (size_t)grid << 31);
    size_t done = 0;
    next_timing_slot(ctx);
    LH_CUDA(ctx, cudaEventRecord(ctx->ev_t0, s));
    while (done < n) {
        size_t m = std::min(n - done, kMaxPerLaunch);
        const double *p = d_values + done;
        // peel up to 3 samples so the body is 32-byte aligned (256-bit loads, 16-byte bulk copies)
        int nhead = (int)(((32u - ((uintptr_t)p & 31u)) & 31u) / 8u);
        if ((size_t)nhead > m) nhead = (int)m;
        const double *head = p;
        const double *body = p + nhead;
        size_t nvec = (m - nhead) >> 2;
        const double *tail = body + nvec * 4;
        int ntail = (int)(m - nhead - nvec * 4);
        kv.launch(grid, kv.smem, s, body, nvec, head, nhead, tail, ntail, counts, flag, ctx->pc);
        LH_CUDA(ctx, cudaGetLastError());
        ctx->stats.kernel_launches++;
        done += m;
    }
    LH_CUDA(ctx, cudaEventRecord(ctx->ev_t1, s));
    ctx->timing_valid = true;
    ctx->stats.samples += n;
    return after_write(ctx, b, s);
}

lh_status fold_hot(lh_ctx *ctx, int b, cudaStream_t s) {
    const size_t cells = (size_t)ctx->H * 2u * ctx->pc.win;
    int grid = (int)std::min<size_t>((cells + 255) / 256, (size_t)ctx->sm_count * 16);
    k_fold_hot<<<grid, 256, 0, s>>>(ctx->buf[b].d_hot, ctx->buf[b].d_buckets, ctx->buf[b].d_flags, cells, ctx->hot_replicas, ctx->pc.win);
    LH_CUDA(ctx, cudaGetLastError());
    ctx->stats.kernel_launches++;
    ctx->buf[b].hot_pending = 0;
    return LH_OK;
}

KeyedOut keyed_out(lh_ctx *ctx, int b) {
    KeyedOut o{};
    o.hot = ctx->buf[b].d_hot; o.buckets = ctx->buf[b].d_buckets; o.flags = ctx->buf[b].d_flags;
    o.dropped = ctx->d_dropped; o.H = ctx->H;
    return o;
}

// How many histograms' positive windows one pass of k_ingest_keyed_small can privatise.
uint32_t ks_ids_per_pass(const lh_ctx *ctx) { return std::max<uint32_t>(1, (uint32_t)(KS_SMEM_BYTES / ((size_t)ctx->pc.win * 4))); }

// Owner-partitioned write-combining kernel: used when the histograms cannot be privatised per CTA in a few
// passes but P owner CTAs (one per SM) can hold them all, and the batch is big enough to amortise the
// cooperative launch.
constexpr size_t kSmemBudget = 227 * 1024;
// Processes the first *taken samples (whole tiles only); the caller sends the rest to the scalar kernel.
// Optional second segment (ids2, vals2, n2): int64 nanosecond samples binned by the SAME launch (ValT = double only).
template <typename IdT, typename ValT, int SPT>
lh_status launch_keyed_wc_spt(lh_ctx *ctx, int b, const IdT *ids, const ValT *vals, size_t n4x4, cudaStream_t s, bool *used, size_t *taken,
                              const IdT *ids2 = nullptr, const long long *vals2 = nullptr, size_t n2 = 0, size_t *taken2 = nullptr) {
    *used = false;
    *taken = 0;
    if (taken2) *taken2 = 0;
    const int P = std::min(ctx->sm_count - ctx->k1_reserve_sms, (int)WC_MAX_PARTS);
    if (P < 8 || n4x4 + n2 == 0) return LH_OK;
    const uint32_t ids_per = (ctx->H + P - 1) / P;
    using S = WcShape<SPT>;
    const size_t hist_bytes = (((size_t)ids_per * ctx->pc.win + 3) & ~(size_t)3) * 4;
    // the owners' windows first, then the largest per-owner buffers that still fit (fewer SMs for ingest = more ids per
    // owner = less room: 256 records at P = 147, 192 at P = 140 for H = 1024)
    uint32_t row_cap = 0;
    size_t smem = 0;
    for (uint32_t cap_try : {256u, 192u, 128u}) {
        smem = hist_bytes + 2 * WC_MAX_PARTS * 4 + (size_t)(P + 1) * (cap_try + WC_ROW_EXTRA) * 2;
        if (smem <= kSmemBudget) { row_cap = cap_try; break; }
    }
    if (!row_cap || (size_t)ids_per * ctx->pc.win > 65535) return LH_OK;               // records are 16-bit (lid*win + slot)
    if (ctx->keyed_mode != 2 && n4x4 + n2 < ((size_t)1 << 22)) return LH_OK;           // small batches: the L2-atomic kernel
    n4x4 = n4x4 / S::TILE * S::TILE;
    n2 = n2 / S::TILE * S::TILE;
    if (n4x4 + n2 == 0) return LH_OK;
    // chunks of about kp_chunk samples, EQUAL in size: with the nominal slice a short last chunk would be binned by a
    // few CTAs at full slice length while the others idle (it cost a whole chunk time per launch: 50 M pairs ran at 211
    // instead of 260 G samples/s, profiles/r02/keyed_batch_probe_r02l.txt)
    const size_t slice_max = std::max<size_t>(1, ((size_t)ctx->kp_chunk + (size_t)P * S::TILE - 1) / ((size_t)P * S::TILE));
    const size_t tiles_all = n4x4 / S::TILE + n2 / S::TILE;
    const size_t nchunks = (tiles_all + slice_max * P - 1) / (slice_max * P);
    const size_t slice_tiles = std::max<size_t>(1, (tiles_all + nchunks * P - 1) / (nchunks * P));
    // every (owner, writer) pair has its own sub-queue: 1.25x the expected records per pair per chunk, plus slack
    // (records that do not fit take the exact L2 route, so this only trades speed on heavily skewed ids)
    const size_t expect = slice_max * S::TILE / P;       // sized for the nominal slice: the allocation does not follow the batch size
    const size_t cap = ((expect * 5 / 4 + 3 * WC_LINE + WC_LINE - 1) / WC_LINE) * WC_LINE;
    if (!ctx->d_kp_queues || ctx->kp_cap != cap || ctx->kp_parts != P) {
        cudaFree(ctx->d_kp_queues); cudaFree(ctx->d_kp_cnt); cudaFree(ctx->d_kp_rare);
        ctx->d_kp_queues = nullptr; ctx->d_kp_cnt = nullptr; ctx->d_kp_rare = nullptr;
        LH_CUDA(ctx, cudaMalloc(&ctx->d_kp_rare, (size_t)P * WC_RARE_CAP * sizeof(uint4)));
        LH_CUDA(ctx, cudaMalloc(&ctx->d_kp_queues, (size_t)2 * P * P * cap * sizeof(unsigned short)));
        LH_CUDA(ctx, cudaMalloc(&ctx->d_kp_cnt, ((size_t)2 * P * P + 1) * sizeof(unsigned int)));
        ctx->kp_cap = cap; ctx->kp_parts = P;
    }
    const void *fn = (const void *)k_ingest_keyed_wc<IdT, ValT, SPT, false>;
    if constexpr (std::is_same<ValT, double>::value) {
        if (n2) fn = (const void *)k_ingest_keyed_wc<IdT, double, SPT, true>;
    }
    LH_CUDA(ctx, cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    unsigned int *d_barrier = ctx->d_kp_cnt + (size_t)2 * P * P;
    LH_CUDA(ctx, cudaMemsetAsync(d_barrier, 0, sizeof(unsigned int), s));
    WcParams prm{};
    prm.ids = ids; prm.vals = vals; prm.n = n4x4; prm.ids_per = ids_per; prm.cap = (uint32_t)cap;
    prm.ids2 = ids2; prm.vals2 = vals2; prm.n2 = n2;
    prm.inv_p = (uint32_t)(((uint64_t)1 << 32) / (uint64_t)P) + 1u;
    // samples between two flushes of the shared-memory owner buffers: the flush costs about the same whatever it moves,
    // so as many as the buffers hold at 4 sigma (wc_flush_samples; default 24576)
    // ... and an owner's expected share m of one interval must leave room for the carried-over remainder (< 64) and the
    // binomial spread: m + 3.5 sqrt(m) + 63 <= row_cap
    const double room = (double)row_cap - 63.0;
    const double m_max = std::pow((-3.5 + std::sqrt(3.5 * 3.5 + 4.0 * room)) / 2.0, 2.0);
    const uint32_t flush_samples = std::min<uint32_t>(ctx->wc_flush_samples, (uint32_t)(m_max * P));
    prm.flush_tiles = std::max<uint32_t>(1u, flush_samples / S::TILE);
    prm.pf_tiles = ctx->wc_pf_tiles;
    prm.row_cap = row_cap;
    prm.row_stride = row_cap + WC_ROW_EXTRA;
    prm.slice_tiles = (uint32_t)slice_tiles; prm.queues = ctx->d_kp_queues; prm.q_cnt = ctx->d_kp_cnt;
    prm.barrier = d_barrier; prm.rare = ctx->d_kp_rare; prm.o = keyed_out(ctx, b);
    Prec pc = ctx->pc;
    void *args[] = {&prm, &pc};
    LH_CUDA(ctx, cudaLaunchCooperativeKernel(fn, dim3(P), dim3(S::THREADS), args, smem, s));
    ctx->stats.kernel_launches++;
    *used = true;
    *taken = n4x4;
    if (taken2) *taken2 = n2;
    return LH_OK;
}
template <typename IdT, typename ValT>
lh_status launch_keyed_wc(lh_ctx *ctx, int b, const IdT *ids, const ValT *vals, size_t n4x4, cudaStream_t s, bool *used, size_t *taken,
                          const IdT *ids2 = nullptr, const long long *vals2 = nullptr, size_t n2 = 0, size_t *taken2 = nullptr) {
#define LH_WC_SHAPE(code) case code: return launch_keyed_wc_spt<IdT, ValT, code>(ctx, b, ids, vals, n4x4, s, used, taken, ids2, vals2, n2, taken2);
    switch (ctx->wc_spt) {
        LH_WC_SHAPE(6) LH_WC_SHAPE(4) LH_WC_SHAPE(3)
        default: return launch_keyed_wc_spt<IdT, ValT, 8>(ctx, b, ids, vals, n4x4, s, used, taken, ids2, vals2, n2, taken2);
    }
#undef LH_WC_SHAPE
}

template <typename IdT, typename ValT>
lh_status launch_keyed(lh_ctx *ctx, const IdT *d_ids, const ValT *d_vals, size_t n, cudaStream_t s) {
    if (((uintptr_t)d_vals & 7u) || ((uintptr_t)d_ids & (sizeof(IdT) - 1)))
        return fail(ctx, LH_ERR_INVALID, "ids / values are not naturally aligned");
    const int b = ctx->active;
    lh_status st = before_write(ctx, b, s);
    if (st != LH_OK) return st;
    constexpr int T = 256;
    const KeyedOut ko = keyed_out(ctx, b);
    next_timing_slot(ctx);
    LH_CUDA(ctx, cudaEventRecord(ctx->ev_t0, s));
    size_t done = 0;
    while (done < n) {
        // no uint32 cell of the hot window may wrap: drain it before 2^32 samples have gone in
        const unsigned long long kCap = 0xFFFFFFFFull;
        if (ctx->buf[b].hot_pending >= kCap - (1ull << 30)) { st = fold_hot(ctx, b, s); if (st != LH_OK) return st; }
        size_t m = (size_t)std::min<unsigned long long>(n - done, kCap - ctx->buf[b].hot_pending);
        const IdT *ids = d_ids + done;
        const ValT *vals = d_vals + done;
        // scalar head until the values are 32-byte aligned; the vector body also needs ids aligned to 4 ids
        size_t head = std::min<size_t>(m, ((32u - ((uintptr_t)vals & 31u)) & 31u) / 8u);
        bool vec_ok = (((uintptr_t)(ids + head)) & (4 * sizeof(IdT) - 1)) == 0;
        size_t n4 = vec_ok ? (m - head) / 4 : 0;
        size_t tail_off = head + n4 * 4;
        if (!vec_ok) { head = 0; tail_off = 0; }
        if (head) {
            k_ingest_keyed<IdT, ValT, T><<<1, T, 0, s>>>(ids, vals, head, ko, ctx->pc);
            ctx->stats.kernel_launches++;
        }
        size_t hot_used = 0;
        if (n4) {
            bool used = false;
            // few histograms: their windows fit in shared memory (K1-style privatisation).  Up to KS_MAX_PASSES
            // passes over id sub-ranges match or beat the L2-atomic kernel (each pass is HBM-bound at 10 B/sample) and,
            // unlike it, do not depend on how clustered the values are.
            constexpr uint32_t KS_MAX_PASSES = 4;
            const uint32_t per_max = ks_ids_per_pass(ctx);
            const uint32_t passes = (ctx->H + per_max - 1) / per_max;
            if (passes <= KS_MAX_PASSES && ctx->keyed_mode == 0 && n4 >= 4096) {
                const uint32_t per = (ctx->H + passes - 1) / passes;
                const size_t smem = ((size_t)per * ctx->pc.win + 4) * 4;
                const void *fn = (const void *)k_ingest_keyed_small<IdT, ValT>;
                LH_CUDA(ctx, cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                // one CTA per SM; fewer when the batch is small, so that the per-CTA flush stays negligible
                int grid = (int)std::max<size_t>(1, std::min<size_t>((size_t)(ctx->sm_count - ctx->k1_reserve_sms),
                                                                      n4 / (KS_THREADS * 16)));
                for (uint32_t lo = 0; lo < ctx->H; lo += per) {
                    const uint32_t cnt = std::min(per, ctx->H - lo);
                    k_ingest_keyed_small<IdT, ValT><<<grid, KS_THREADS, smem, s>>>(ids + head, vals + head, n4, lo, cnt, ko, ctx->pc);
                    ctx->stats.kernel_launches++;
                }
                used = true;
                hot_used = n4 * 4;
                ctx->keyed_kernel = "k_ingest_keyed_small";
            }
            if (!used && ctx->keyed_mode != 1) {
                size_t taken = 0;
                st = launch_keyed_wc<IdT, ValT>(ctx, b, ids + head, vals + head, n4 * 4, s, &used, &taken);
                if (st != LH_OK) return st;
                if (used) {
                    ctx->keyed_kernel = "k_ingest_keyed_wc";
                    tail_off = head + taken;          // whole tiles only: the ragged remainder goes through the scalar kernel below
                }
            }
            if (!used) {
                int grid = grid_1d(ctx, n4, T, 1, ctx->keyed_blocks_per_sm);
                k_ingest_keyed_vec<IdT, ValT, T><<<grid, T, 0, s>>>(ids + head, vals + head, n4, ctx->hot_replicas, ko, ctx->pc);
                ctx->stats.kernel_launches++;
                hot_used = n4 * 4;
                ctx->keyed_kernel = "k_ingest_keyed_vec";
            }
        }
        if (tail_off < m) {
            size_t r = m - tail_off;
            int grid = grid_1d(ctx, r, T, 1, ctx->keyed_blocks_per_sm);
            k_ingest_keyed<IdT, ValT, T><<<grid, T, 0, s>>>(ids + tail_off, vals + tail_off, r, ko, ctx->pc);
            ctx->stats.kernel_launches++;
        }
        LH_CUDA(ctx, cudaGetLastError());
        ctx->buf[b].hot_pending += hot_used;     // only k_ingest_keyed_small / _vec count into the uint32 hot window
        done += m;
    }
    LH_CUDA(ctx, cudaEventRecord(ctx->ev_t1, s));
    ctx->timing_valid = true;
    ctx->stats.samples += n;
    return after_write(ctx, b, s);
}

// Histogram samples (float64) and Timer samples (int64 ns, metrics.go:242-246) of one batch in ONE launch of the
// write-combining kernel: its fixed costs (zeroing and flushing the owners' windows, the last partly filled chunk) are
// paid once.  Needs both arrays vector-aligned and the write-combining kernel eligible; otherwise two keyed ingests.
template <typename IdT>
lh_status launch_keyed_pair(lh_ctx *ctx, const IdT *ids_f, const double *vals_f, size_t n_f, const IdT *ids_ns, const long long *vals_ns,
                            size_t n_ns, cudaStream_t s) {
    auto aligned = [](const void *v, const void *i) { return (((uintptr_t)v & 31u) == 0) && (((uintptr_t)i & (4 * sizeof(IdT) - 1)) == 0); };
    // few histograms: the shared-memory privatised kernel of launch_keyed() is the better one, per array
    const uint32_t small_passes = (ctx->H + ks_ids_per_pass(ctx) - 1) / ks_ids_per_pass(ctx);
    const bool small = small_passes <= 4 && ctx->keyed_mode == 0;
    const bool fuse = n_f && n_ns && ctx->keyed_mode != 1 && !small && aligned(vals_f, ids_f) && aligned(vals_ns, ids_ns);
    if (fuse) {
        const int b = ctx->active;
        lh_status st = before_write(ctx, b, s);
        if (st != LH_OK) return st;
        next_timing_slot(ctx);
        LH_CUDA(ctx, cudaEventRecord(ctx->ev_t0, s));
        bool used = false;
        size_t took_f = 0, took_ns = 0;
        st = launch_keyed_wc<IdT, double>(ctx, b, ids_f, vals_f, n_f, s, &used, &took_f, ids_ns, vals_ns, n_ns, &took_ns);
        if (st != LH_OK) return st;
        if (used) {
            constexpr int T = 256;
            const KeyedOut ko = keyed_out(ctx, b);
            ctx->keyed_kernel = "k_ingest_keyed_wc";
            if (took_f < n_f) {          // the ragged ends go through the scalar kernel
                k_ingest_keyed<IdT, double, T><<<grid_1d(ctx, n_f - took_f, T, 1, ctx->keyed_blocks_per_sm), T, 0, s>>>(
                    ids_f + took_f, vals_f + took_f, n_f - took_f, ko, ctx->pc);
                ctx->stats.kernel_launches++;
            }
            if (took_ns < n_ns) {
                k_ingest_keyed<IdT, long long, T><<<grid_1d(ctx, n_ns - took_ns, T, 1, ctx->keyed_blocks_per_sm), T, 0, s>>>(
                    ids_ns + took_ns, vals_ns + took_ns, n_ns - took_ns, ko, ctx->pc);
                ctx->stats.kernel_launches++;
            }
            LH_CUDA(ctx, cudaGetLastError());
            LH_CUDA(ctx, cudaEventRecord(ctx->ev_t1, s));
            ctx->timing_valid = true;
            ctx->stats.samples += n_f + n_ns;
            return after_write(ctx, b, s);
        }
        // not eligible after all (few histograms, small batch): the events recorded above are simply overwritten below
        st = after_write(ctx, b, s);
        if (st != LH_OK) return st;
    }
    lh_status st = n_f ? launch_keyed<IdT, double>(ctx, ids_f, vals_f, n_f, s) : LH_OK;
    if (st != LH_OK) return st;
    return n_ns ? launch_keyed<IdT, long long>(ctx, ids_ns, vals_ns, n_ns, s) : LH_OK;
}

template <typename IdT>
lh_status launch_counter(lh_ctx *ctx, const IdT *d_ids, const uint64_t *d_amounts, size_t n, cudaStream_t s) {
    const int b = ctx->active;
    lh_status st = before_write(ctx, b, s);
    if (st != LH_OK) return st;
    next_timing_slot(ctx);
    LH_CUDA(ctx, cudaEventRecord(ctx->ev_t0, s));
    if (n) {
        constexpr int T = 512;
        const unsigned long long *amts = reinterpret_cast<const unsigned long long *>(d_amounts);
        if (ctx->C <= (uint32_t)K2_SMEM_COUNTERS) {
            // privatised per CTA (lo/hi halves in shared memory).  Vector body where the alignment allows: 4 ops per
            // thread and iteration; ragged head / tail through the scalar form of the same kernel.
            size_t head = std::min<size_t>(n, ((32u - ((uintptr_t)amts & 31u)) & 31u) / 8u);
            const bool vec_ok = (((uintptr_t)(d_ids + head)) & (4 * sizeof(IdT) - 1)) == 0 && (((uintptr_t)amts & 7u) == 0);
            size_t n4 = vec_ok ? (n - head) / 4 : 0;
            if (n4 < 4096) { head = 0; n4 = 0; }
            const size_t tail_off = head + n4 * 4;
            if (head) {
                k_counter_add_smem<IdT, T><<<1, T, (size_t)ctx->C * 8, s>>>(d_ids, amts, head, ctx->buf[b].d_counters, ctx->C, ctx->d_dropped);
                ctx->stats.kernel_launches++;
            }
            if (n4) {
                // one CTA per SM (the per-CTA flush is C global atomics), fewer for small batches
                const int grid = (int)std::max<size_t>(1, std::min<size_t>((size_t)std::max(1, ctx->sm_count - ctx->k1_reserve_sms) * 2, n4 / (T * 4)));
                k_counter_add_smem_vec<IdT, T><<<grid, T, (size_t)ctx->C * 8, s>>>(d_ids + head, amts + head, n4, ctx->buf[b].d_counters, ctx->C, ctx->d_dropped);
                ctx->stats.kernel_launches++;
            }
            if (tail_off < n) {
                int grid = grid_1d(ctx, n - tail_off, T, 8, 2);
                k_counter_add_smem<IdT, T><<<grid, T, (size_t)ctx->C * 8, s>>>(d_ids + tail_off, amts + tail_off, n - tail_off, ctx->buf[b].d_counters, ctx->C, ctx->d_dropped);
                ctx->stats.kernel_launches++;
            }
        } else {
            int grid = grid_1d(ctx, n, T, 4, 4);
            k_counter_add<IdT, T><<<grid, T, 0, s>>>(d_ids, amts, n, ctx->buf[b].d_counters, ctx->C, ctx->d_dropped);
            ctx->stats.kernel_launches++;
        }
        LH_CUDA(ctx, cudaGetLastError());
    }
    LH_CUDA(ctx, cudaEventRecord(ctx->ev_t1, s));
    ctx->timing_valid = true;
    ctx->stats.counter_ops += n;
    return after_write(ctx, b, s);
}

// ---- staging ring (locked) ----
// Called with ctx->mu held through `lk`.  The host-side wait for an in-flight slot happens with the mutex RELEASED
// (the slot is parked as SLOT_WAITED meanwhile so nobody else takes it): other ingest threads are never held up by
// it, and a thread that finds every slot either acquired or being waited for sleeps on slot_cv until one comes back.
lh_status slot_wait_free(lh_ctx *ctx, std::unique_lock<std::mutex> &lk, int *out) {
    for (;;) {
        // prefer a free slot that already has memory, then an in-flight one that has already finished, then a fresh
        // slot (allocating its pinned + device memory), and only then wait for the oldest in-flight one
        int best = -1, fresh = -1, waited = 0;
        for (size_t i = 0; i < ctx->slots.size(); i++) {
            if (ctx->slots[i].state == SLOT_WAITED || ctx->slots[i].state == SLOT_FILLING) waited++;   // will come back by itself
            if (ctx->slots[i].state != SLOT_FREE) continue;
            if (ctx->slots[i].h) { *out = (int)i; return LH_OK; }
            if (fresh < 0) fresh = (int)i;
        }
        for (size_t i = 0; i < ctx->slots.size(); i++)
            if (ctx->slots[i].state == SLOT_INFLIGHT && cudaEventQuery(ctx->slots[i].done) == cudaSuccess) {
                ctx->slots[i].state = SLOT_FREE;
                *out = (int)i;
                return LH_OK;
            }
        cudaGetLastError();   // cudaErrorNotReady from the queries above is not an error
        if (fresh >= 0) {
            Slot &sl = ctx->slots[fresh];
            cudaError_t e = cudaMallocHost(&sl.h, ctx->staging_bytes);
            if (e == cudaSuccess) e = cudaMalloc(&sl.d, ctx->staging_bytes);
            if (e != cudaSuccess) {
                if (sl.h) cudaFreeHost(sl.h);
                sl.h = nullptr; sl.d = nullptr;
                return fail(ctx, e == cudaErrorMemoryAllocation ? LH_ERR_NOMEM : LH_ERR_CUDA, "allocating a staging slot", e);
            }
            *out = fresh;
            return LH_OK;
        }
        for (size_t i = 0; i < ctx->slots.size(); i++)
            if (ctx->slots[i].state == SLOT_INFLIGHT && (best < 0 || ctx->slots[i].seq < ctx->slots[best].seq)) best = (int)i;
        if (best >= 0) {
            ctx->slots[best].state = SLOT_WAITED;
            cudaEvent_t ev = ctx->slots[best].done;
            lk.unlock();
            cudaError_t e = cudaEventSynchronize(ev);
            lk.lock();
            ctx->slots[best].state = SLOT_FREE;
            ctx->slot_cv.notify_all();
            if (e != cudaSuccess) return fail(ctx, LH_ERR_CUDA, "cudaEventSynchronize(slot)", e);
            *out = best;
            return LH_OK;
        }
        if (!waited) return fail(ctx, LH_ERR_STATE, "every staging slot is acquired and none is in flight");
        ctx->slot_cv.wait(lk);   // other threads are waiting for kernels: one of them will free a slot (or take it; then retry)
    }
}

// close the IPC mappings of the peers (lh_comm_import), if any
void comm_unmap(lh_ctx *ctx) {
    for (int r = 0; r < kMaxRanks; r++) {
        PeerMap &pm = ctx->peers[r];
        if (pm.ipc) {
            for (int b = 0; b < 2; b++) {
                if (pm.buckets[b]) cudaIpcCloseMemHandle(pm.buckets[b]);
                if (pm.flags[b]) cudaIpcCloseMemHandle(pm.flags[b]);
                if (pm.counters[b]) cudaIpcCloseMemHandle(pm.counters[b]);
            }
            if (pm.comm) cudaIpcCloseMemHandle(pm.comm);
            if (pm.red) cudaIpcCloseMemHandle(pm.red);
        }
        pm = PeerMap{};
    }
    ctx->comm_world = 0;
}

// the arrays the all-reduce writes (this rank's own kernel and, for its slices, every peer's)
lh_status comm_alloc_reduced(lh_ctx *ctx) {
    if (ctx->d_red_buckets) return LH_OK;
    const size_t bucket_bytes = (size_t)ctx->H * 65536u * 8u;
    LH_CUDA(ctx, cudaMalloc(&ctx->d_red_buckets, bucket_bytes));
    LH_CUDA(ctx, cudaMalloc(&ctx->d_red_flags, (size_t)ctx->H * 4));
    LH_CUDA(ctx, cudaMalloc(&ctx->d_red_counters, (size_t)ctx->C * 8));
    LH_CUDA(ctx, cudaMemsetAsync(ctx->d_red_buckets, 0, bucket_bytes, ctx->snap_stream));
    LH_CUDA(ctx, cudaMemsetAsync(ctx->d_red_flags, 0, (size_t)ctx->H * 4, ctx->snap_stream));
    LH_CUDA(ctx, cudaMemsetAsync(ctx->d_red_counters, 0, (size_t)ctx->C * 8, ctx->snap_stream));
    LH_CUDA(ctx, cudaStreamSynchronize(ctx->snap_stream));
    return LH_OK;
}

bool is_pinned_or_managed(const void *p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeManaged;
}

cudaError_t export_bufs_alloc(ExportBufs &x, size_t H, size_t C) {
    cudaError_t e = cudaMalloc(&x.d_nnz, H * 4);
    if (e == cudaSuccess) e = cudaMalloc(&x.d_offsets, (H + 1) * 4);
    if (e == cudaSuccess) e = cudaMallocHost(&x.h_offsets, (H + 1) * 4);
    if (e == cudaSuccess) e = cudaMallocHost(&x.h_counters, C * 8);
    return e;
}

void export_bufs_free_lists(ExportBufs &x) {
    cudaFree(x.d_keys); cudaFree(x.d_counts);
    if (x.h_keys) cudaFreeHost(x.h_keys);
    if (x.h_counts) cudaFreeHost(x.h_counts);
    x.d_keys = nullptr; x.d_counts = nullptr; x.h_keys = nullptr; x.h_counts = nullptr; x.cap = 0;
}

void export_bufs_free(ExportBufs &x) {
    export_bufs_free_lists(x);
    cudaFree(x.d_nnz); cudaFree(x.d_offsets);
    if (x.h_offsets) cudaFreeHost(x.h_offsets);
    if (x.h_counters) cudaFreeHost(x.h_counters);
    x = ExportBufs{};
}

void window_free(Window *w) {
    if (!w) return;
    cudaFree(w->d_acc); cudaFree(w->d_flags); cudaFree(w->d_levels); cudaFree(w->d_counters);
    for (auto &sl : w->ring) {
        cudaFree(sl.d_offsets); cudaFree(sl.d_flags); cudaFree(sl.d_counters); cudaFree(sl.d_keys); cudaFree(sl.d_counts);
    }
    if (w->h_total) cudaFreeHost(w->h_total);
    cudaFree(w->d_ps); cudaFree(w->d_res);
    if (w->h_res) cudaFreeHost(w->h_res);
    export_bufs_free(w->x);
    delete w;
}

}  // namespace

// =========================================================== lifecycle
extern "C" uint32_t lh_abi_version(void) { return LH_ABI_VERSION; }

extern "C" const char *lh_strerror(lh_status st) {
    switch (st) {
    case LH_OK: return "ok";
    case LH_ERR_INVALID: return "invalid argument";
    case LH_ERR_CUDA: return "CUDA runtime error";
    case LH_ERR_NOMEM: return "out of memory";
    case LH_ERR_NO_DEVICE: return "no usable CUDA device (there is no CPU fallback)";
    case LH_ERR_STATE: return "call out of order";
    case LH_ERR_RANGE: return "id or size out of range";
    default: return "unknown status";
    }
}

extern "C" const char *lh_last_error(const lh_ctx *ctx) { return ctx ? ctx->last_error.c_str() : ""; }

extern "C" lh_status lh_create(const lh_config *cfg, lh_ctx **out) {
    if (!cfg || !out || cfg->struct_size != sizeof(lh_config) || cfg->max_histograms == 0 || cfg->max_counters == 0)
        return LH_ERR_INVALID;
    if (cfg->precision > LH_MAX_PRECISION) return LH_ERR_RANGE;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); return LH_ERR_NO_DEVICE; }
    if (cfg->device < 0 || cfg->device >= ndev) return LH_ERR_NO_DEVICE;
    lh_ctx *ctx = new (std::nothrow) lh_ctx();
    if (!ctx) return LH_ERR_NOMEM;
    ctx->cfg = *cfg;
    ctx->device = cfg->device;
    ctx->H = cfg->max_histograms;
    ctx->C = cfg->max_counters;
    ctx->pc = make_prec(cfg->precision ? cfg->precision : 100);
    {
        static std::mutex id_mu;
        static uint64_t next_id = 1;
        std::lock_guard<std::mutex> lk(id_mu);
        ctx->ctx_id = next_id++;
    }
    {   // replicas of the keyed hot window: as many as keep all copies within ~48 MB (L2-resident), at most 32
        const size_t one = (size_t)ctx->H * 2u * ctx->pc.win * 4u;
        ctx->hot_replicas = (uint32_t)std::max<size_t>(1, std::min<size_t>(32, ((size_t)48 << 20) / one));
    }
    ctx->staging_bytes = cfg->staging_bytes ? (size_t)cfg->staging_bytes : ((size_t)32 << 20);
    ctx->staging_bytes = (ctx->staging_bytes + 255) & ~(size_t)255;
    const uint32_t nslots = cfg->staging_slots ? cfg->staging_slots : 3;

#define LH_CREATE_CUDA(call)                                                            \
    do {                                                                                \
        cudaError_t _e = (call);                                                        \
        if (_e != cudaSuccess) {                                                        \
            fprintf(stderr, "loghisto_b200: lh_create: %s failed: %s\n", #call, cudaGetErrorString(_e)); \
            lh_destroy(ctx);                                                            \
            return _e == cudaErrorMemoryAllocation ? LH_ERR_NOMEM : LH_ERR_CUDA;        \
        }                                                                               \
    } while (0)

    LH_CREATE_CUDA(cudaSetDevice(ctx->device));
    cudaDeviceProp prop;
    LH_CREATE_CUDA(cudaGetDeviceProperties(&prop, ctx->device));
    if (prop.major < 10) {
        fprintf(stderr, "loghisto_b200: device %d is sm_%d%d; this library is built for sm_100a only\n", ctx->device, prop.major, prop.minor);
        lh_destroy(ctx);
        return LH_ERR_NO_DEVICE;
    }
    ctx->sm_count = prop.multiProcessorCount;
    LH_CREATE_CUDA(cudaStreamCreateWithFlags(&ctx->ingest_stream, cudaStreamNonBlocking));
    LH_CREATE_CUDA(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    {   // the snapshot stream outranks ingest: its small kernels slot in as soon as any ingest CTA retires
        int least = 0, greatest = 0;
        LH_CREATE_CUDA(cudaDeviceGetStreamPriorityRange(&least, &greatest));
        LH_CREATE_CUDA(cudaStreamCreateWithPriority(&ctx->snap_stream, cudaStreamNonBlocking, greatest));
    }
    for (int i = 0; i < lh_ctx::kTimingRing; i++) {
        LH_CREATE_CUDA(cudaEventCreate(&ctx->ev_t0s[i]));
        LH_CREATE_CUDA(cudaEventCreate(&ctx->ev_t1s[i]));
    }
    for (int i = 0; i < lh_ctx::kCommRing; i++) {
        LH_CREATE_CUDA(cudaEventCreate(&ctx->comm_t0[i]));
        LH_CREATE_CUDA(cudaEventCreate(&ctx->comm_t1[i]));
    }

    const size_t bucket_bytes = (size_t)ctx->H * 65536u * 8u, counter_bytes = (size_t)ctx->C * 8u;
    const size_t hot_bytes = (size_t)ctx->hot_replicas * ctx->H * 2u * ctx->pc.win * 4u;
    for (int b = 0; b < 2; b++) {
        LH_CREATE_CUDA(cudaMalloc(&ctx->buf[b].d_buckets, bucket_bytes));
        LH_CREATE_CUDA(cudaMalloc(&ctx->buf[b].d_counters, counter_bytes));
        LH_CREATE_CUDA(cudaMalloc(&ctx->buf[b].d_flags, (size_t)ctx->H * 4u));
        LH_CREATE_CUDA(cudaMemsetAsync(ctx->buf[b].d_buckets, 0, bucket_bytes, ctx->snap_stream));
        LH_CREATE_CUDA(cudaMemsetAsync(ctx->buf[b].d_counters, 0, counter_bytes, ctx->snap_stream));
        LH_CREATE_CUDA(cudaMemsetAsync(ctx->buf[b].d_flags, 0, (size_t)ctx->H * 4u, ctx->snap_stream));
        LH_CREATE_CUDA(cudaMalloc(&ctx->buf[b].d_hot, hot_bytes));
        LH_CREATE_CUDA(cudaMemsetAsync(ctx->buf[b].d_hot, 0, hot_bytes, ctx->snap_stream));
        LH_CREATE_CUDA(cudaEventCreateWithFlags(&ctx->buf[b].cleared, cudaEventDisableTiming));
        LH_CREATE_CUDA(cudaEventRecord(ctx->buf[b].cleared, ctx->snap_stream));
    }
    LH_CREATE_CUDA(cudaMalloc(&ctx->d_decomp, 65536 * sizeof(double)));
    k_fill_decompress<<<65536 / 256, 256, 0, ctx->snap_stream>>>(ctx->d_decomp, ctx->pc.precision);
    LH_CREATE_CUDA(cudaGetLastError());
    LH_CREATE_CUDA(cudaMalloc(&ctx->d_comm, kCommWords * 8));
    LH_CREATE_CUDA(cudaMemsetAsync(ctx->d_comm, 0, kCommWords * 8, ctx->snap_stream));
    LH_CREATE_CUDA(cudaMalloc(&ctx->d_comm_aux, 16));
    LH_CREATE_CUDA(cudaMemsetAsync(ctx->d_comm_aux, 0, 16, ctx->snap_stream));
    LH_CREATE_CUDA(cudaMalloc(&ctx->d_dropped, 8));
    LH_CREATE_CUDA(cudaMemsetAsync(ctx->d_dropped, 0, 8, ctx->snap_stream));
    for (int i = 0; i < 3; i++) {
        const size_t res_bytes = (size_t)ctx->H * (24 + LH_MAX_PERCENTILES * 12);
        LH_CREATE_CUDA(cudaMalloc(&ctx->d_ps[i], LH_MAX_PERCENTILES * sizeof(double)));
        LH_CREATE_CUDA(cudaMalloc(&ctx->d_res[i], res_bytes));
        LH_CREATE_CUDA(cudaMallocHost(&ctx->h_res[i], res_bytes));
        LH_CREATE_CUDA(cudaEventCreateWithFlags(&ctx->res_done[i], cudaEventDisableTiming));
    }
    LH_CREATE_CUDA(export_bufs_alloc(ctx->x, ctx->H, ctx->C));

    ctx->slots.resize(nslots);   // pinned + device memory of a slot is allocated the first time it is handed out
    for (auto &sl : ctx->slots) {
        LH_CREATE_CUDA(cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming));
        LH_CREATE_CUDA(cudaEventCreateWithFlags(&sl.copied, cudaEventDisableTiming));
    }

    LH_CREATE_CUDA(cudaFuncSetAttribute((const void *)k_reduce, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    LH_CREATE_CUDA(cudaFuncSetAttribute((const void *)k_peer_allreduce, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
    LH_CREATE_CUDA(cudaFuncSetAttribute((const void *)k_counter_add_smem<unsigned short, 512>, cudaFuncAttributeMaxDynamicSharedMemorySize, K2_SMEM_COUNTERS * 8));
    LH_CREATE_CUDA(cudaFuncSetAttribute((const void *)k_counter_add_smem<unsigned int, 512>, cudaFuncAttributeMaxDynamicSharedMemorySize, K2_SMEM_COUNTERS * 8));
    LH_CREATE_CUDA(cudaFuncSetAttribute((const void *)k_counter_add_smem_vec<unsigned short, 512>, cudaFuncAttributeMaxDynamicSharedMemorySize, K2_SMEM_COUNTERS * 8));
    LH_CREATE_CUDA(cudaFuncSetAttribute((const void *)k_counter_add_smem_vec<unsigned int, 512>, cudaFuncAttributeMaxDynamicSharedMemorySize, K2_SMEM_COUNTERS * 8));
    for (int i = 0; i < kNumK1Variants; i++) {
        ctx->k1[i] = g_k1_variants[i];
        const bool probe = ctx->k1[i].launch == launch_probe;
        const size_t hist = ((size_t)2 * ctx->pc.win + 8) * 4;
        ctx->k1[i].smem = probe ? 0 : ctx->k1[i].smem_fixed + hist;
        if (ctx->k1[i].smem > kSmemBudget) {
            // this ring does not fit beside the sub-histogram at this precision: take the next smaller ring with the same
            // arithmetic, and the register-pipelined kernel when none fits
            static const int smaller[] = {5, 0, 2, 3};
            for (int j : smaller) {
                if (g_k1_variants[j].smem_fixed + hist <= kSmemBudget) {
                    const char *name = ctx->k1[i].name;
                    ctx->k1[i] = g_k1_variants[j];
                    ctx->k1[i].name = name;
                    ctx->k1[i].smem = g_k1_variants[j].smem_fixed + hist;
                    break;
                }
            }
        }
        LH_CREATE_CUDA(cudaFuncSetAttribute(ctx->k1[i].func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ctx->k1[i].smem));
        int nb = 0;
        LH_CREATE_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, ctx->k1[i].func, ctx->k1[i].threads, ctx->k1[i].smem));
        ctx->k1[i].blocks_per_sm = std::max(nb, 1);
    }
    LH_CREATE_CUDA(cudaStreamSynchronize(ctx->snap_stream));
#undef LH_CREATE_CUDA
    *out = ctx;
    return LH_OK;
}

extern "C" lh_status lh_destroy(lh_ctx *ctx) {
    if (!ctx) return LH_OK;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    comm_unmap(ctx);
    cudaFree(ctx->d_comm); cudaFree(ctx->d_comm_aux);
    cudaFree(ctx->d_red_buckets); cudaFree(ctx->d_red_flags); cudaFree(ctx->d_red_counters);
    for (int i = 0; i < lh_ctx::kCommRing; i++) {
        if (ctx->comm_t0[i]) cudaEventDestroy(ctx->comm_t0[i]);
        if (ctx->comm_t1[i]) cudaEventDestroy(ctx->comm_t1[i]);
    }
    for (int b = 0; b < 2; b++) {
        cudaFree(ctx->buf[b].d_buckets); cudaFree(ctx->buf[b].d_counters); cudaFree(ctx->buf[b].d_hot); cudaFree(ctx->buf[b].d_flags);
        if (ctx->buf[b].cleared) cudaEventDestroy(ctx->buf[b].cleared);
        for (auto &w : ctx->buf[b].writers) cudaEventDestroy(w.ev);
    }
    cudaFree(ctx->d_decomp); cudaFree(ctx->d_dropped);
    cudaFree(ctx->d_kp_queues); cudaFree(ctx->d_kp_cnt); cudaFree(ctx->d_kp_rare);
    for (int i = 0; i < 3; i++) {
        cudaFree(ctx->d_ps[i]); cudaFree(ctx->d_res[i]);
        if (ctx->h_res[i]) cudaFreeHost(ctx->h_res[i]);
        if (ctx->res_done[i]) cudaEventDestroy(ctx->res_done[i]);
    }
    export_bufs_free(ctx->x);
    window_free(ctx->win);
    ctx->win = nullptr;
    for (auto &sl : ctx->slots) {
        if (sl.h) cudaFreeHost(sl.h);
        cudaFree(sl.d);
        if (sl.done) cudaEventDestroy(sl.done);
        if (sl.copied) cudaEventDestroy(sl.copied);
    }
    for (int i = 0; i < lh_ctx::kTimingRing; i++) {
        if (ctx->ev_t0s[i]) cudaEventDestroy(ctx->ev_t0s[i]);
        if (ctx->ev_t1s[i]) cudaEventDestroy(ctx->ev_t1s[i]);
    }
    if (ctx->ingest_stream) cudaStreamDestroy(ctx->ingest_stream);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->snap_stream) cudaStreamDestroy(ctx->snap_stream);
    cudaGetLastError();
    delete ctx;
    return LH_OK;
}

// =========================================================== ingest (device)
#define LH_ENTER(ctx)                                   \
    if (!(ctx)) return LH_ERR_INVALID;                  \
    std::unique_lock<std::mutex> _lk((ctx)->mu);        \
    LH_CUDA((ctx), cudaSetDevice((ctx)->device))

extern "C" lh_status lh_ingest_f64(lh_ctx *ctx, uint32_t hid, const double *d_values, size_t n, void *stream) {
    LH_ENTER(ctx);
    if (n && !d_values) return fail(ctx, LH_ERR_INVALID, "d_values is NULL");
    if (n == 0) return LH_OK;
    return launch_single(ctx, hid, d_values, n, pick_stream(ctx, stream));
}
extern "C" lh_status lh_ingest_keyed_f64_u16(lh_ctx *ctx, const uint16_t *d_ids, const double *d_values, size_t n, void *stream) {
    LH_ENTER(ctx);
    if (n && (!d_ids || !d_values)) return fail(ctx, LH_ERR_INVALID, "NULL input");
    return launch_keyed<unsigned short, double>(ctx, d_ids, d_values, n, pick_stream(ctx, stream));
}
extern "C" lh_status lh_ingest_keyed_f64_u32(lh_ctx *ctx, const uint32_t *d_ids, const double *d_values, size_t n, void *stream) {
    LH_ENTER(ctx);
    if (n && (!d_ids || !d_values)) return fail(ctx, LH_ERR_INVALID, "NULL input");
    return launch_keyed<unsigned int, double>(ctx, d_ids, d_values, n, pick_stream(ctx, stream));
}
extern "C" lh_status lh_ingest_keyed_i64ns_u16(lh_ctx *ctx, const uint16_t *d_ids, const int64_t *d_nanos, size_t n, void *stream) {
    LH_ENTER(ctx);
    if (n && (!d_ids || !d_nanos)) return fail(ctx, LH_ERR_INVALID, "NULL input");
    return launch_keyed<unsigned short, long long>(ctx, d_ids, reinterpret_cast<const long long *>(d_nanos), n, pick_stream(ctx, stream));
}
extern "C" lh_status lh_ingest_keyed_pair_u16(lh_ctx *ctx, const uint16_t *d_ids_f64, const double *d_values, size_t n_f64,
                                              const uint16_t *d_ids_ns, const int64_t *d_nanos, size_t n_ns, void *stream) {
    LH_ENTER(ctx);
    if ((n_f64 && (!d_ids_f64 || !d_values)) || (n_ns && (!d_ids_ns || !d_nanos))) return fail(ctx, LH_ERR_INVALID, "NULL input");
    if (((uintptr_t)d_values & 7u) || ((uintptr_t)d_nanos & 7u) || ((uintptr_t)d_ids_f64 & 1u) || ((uintptr_t)d_ids_ns & 1u))
        return fail(ctx, LH_ERR_INVALID, "ids / values are not naturally aligned");
    return launch_keyed_pair<unsigned short>(ctx, d_ids_f64, d_values, n_f64, d_ids_ns, reinterpret_cast<const long long *>(d_nanos), n_ns,
                                             pick_stream(ctx, stream));
}
extern "C" lh_status lh_counter_add_u16(lh_ctx *ctx, const uint16_t *d_ids, const uint64_t *d_amounts, size_t n, void *stream) {
    LH_ENTER(ctx);
    if (n && (!d_ids || !d_amounts)) return fail(ctx, LH_ERR_INVALID, "NULL input");
    return launch_counter<unsigned short>(ctx, d_ids, d_amounts, n, pick_stream(ctx, stream));
}
extern "C" lh_status lh_counter_add_u32(lh_ctx *ctx, const uint32_t *d_ids, const uint64_t *d_amounts, size_t n, void *stream) {
    LH_ENTER(ctx);
    if (n && (!d_ids || !d_amounts)) return fail(ctx, LH_ERR_INVALID, "NULL input");
    return launch_counter<unsigned int>(ctx, d_ids, d_amounts, n, pick_stream(ctx, stream));
}

// =========================================================== ingest (host)
// Chunks of staging_bytes go through the slot ring: (memcpy into pinned if the
// source is pageable) -> async H2D -> kernel, all on the ingest stream.
namespace {
enum HostKind { HK_SINGLE, HK_KEYED_U16, HK_COUNTER_U16, HK_KEYED_I64_U16 };

lh_status ingest_host(lh_ctx *ctx, std::unique_lock<std::mutex> &lk, HostKind kind, uint32_t hid,
                      const void *h_a /* 8-byte items */, const uint16_t *h_ids, size_t n) {
    const bool pinned = is_pinned_or_managed(h_a) && (!h_ids || is_pinned_or_managed(h_ids));
    const size_t item = (kind == HK_SINGLE) ? 8 : 10;
    size_t per = ctx->staging_bytes / item;
    per &= ~(size_t)15;   // keeps the ids region 16-byte aligned
    if (per == 0) return fail(ctx, LH_ERR_INVALID, "staging_bytes too small");
    cudaStream_t s = ctx->ingest_stream;
    size_t done = 0;
    cudaEvent_t last_copied = nullptr;
    while (done < n) {
        size_t m = std::min(per, n - done);
        int si;
        lh_status st = slot_wait_free(ctx, lk, &si);
        if (st != LH_OK) return st;
        Slot &sl = ctx->slots[si];
        const char *src_a = (const char *)h_a + done * 8;
        char *d_a = (char *)sl.d;
        char *d_i = (char *)sl.d + per * 8;
        const void *cp_a = src_a;
        const void *cp_i = h_ids ? (const void *)(h_ids + done) : nullptr;
        if (!pinned) {
            // pageable source: stage through the slot's pinned buffer.  The memcpy (milliseconds per 32 MiB) runs with
            // the context mutex RELEASED -- the slot is parked as ACQUIRED so no other thread can take it.
            sl.state = SLOT_FILLING;
            lk.unlock();
            memcpy(sl.h, src_a, m * 8);
            if (h_ids) memcpy((char *)sl.h + per * 8, h_ids + done, m * 2);
            lk.lock();
            cp_a = sl.h;
            cp_i = (char *)sl.h + per * 8;
        }
        // copies run on their own stream so that chunk k+1's DMA overlaps chunk k's kernel; the slot's device
        // buffer is free again once the kernel that read it last is done (slot_wait_free already waited on the host
        // for a recycled slot, the event wait covers the rest)
        cudaStream_t cs = ctx->copy_stream;
        if (sl.seq) LH_CUDA(ctx, cudaStreamWaitEvent(cs, sl.done, 0));
        LH_CUDA(ctx, cudaMemcpyAsync(d_a, cp_a, m * 8, cudaMemcpyHostToDevice, cs));
        if (h_ids) LH_CUDA(ctx, cudaMemcpyAsync(d_i, cp_i, m * 2, cudaMemcpyHostToDevice, cs));
        LH_CUDA(ctx, cudaEventRecord(sl.copied, cs));
        LH_CUDA(ctx, cudaStreamWaitEvent(s, sl.copied, 0));
        last_copied = sl.copied;
        ctx->stats.h2d_bytes += m * item;
        if (kind == HK_SINGLE) st = launch_single(ctx, hid, (const double *)d_a, m, s);
        else if (kind == HK_KEYED_U16) st = launch_keyed<unsigned short, double>(ctx, (const unsigned short *)d_i, (const double *)d_a, m, s);
        else if (kind == HK_KEYED_I64_U16) st = launch_keyed<unsigned short, long long>(ctx, (const unsigned short *)d_i, (const long long *)d_a, m, s);
        else st = launch_counter<unsigned short>(ctx, (const unsigned short *)d_i, (const uint64_t *)d_a, m, s);
        if (st != LH_OK) { sl.state = SLOT_FREE; return st; }
        LH_CUDA(ctx, cudaEventRecord(sl.done, s));
        sl.state = SLOT_INFLIGHT;
        sl.seq = ++ctx->slot_seq;
        ctx->slot_cv.notify_all();
        done += m;
    }
    if (pinned && last_copied) {
        // the caller may reuse its buffers on return: the async copies must have READ them (the kernels may still run);
        // waited for with the mutex released
        lk.unlock();
        cudaError_t e = cudaEventSynchronize(last_copied);
        lk.lock();
        if (e != cudaSuccess) return fail(ctx, LH_ERR_CUDA, "cudaEventSynchronize(copied)", e);
    }
    return LH_OK;
}
}  // namespace

extern "C" lh_status lh_ingest_f64_host(lh_ctx *ctx, uint32_t hid, const double *h_values, size_t n) {
    LH_ENTER(ctx);
    if (n && !h_values) return fail(ctx, LH_ERR_INVALID, "h_values is NULL");
    if (hid >= ctx->H) return fail(ctx, LH_ERR_RANGE, "histogram_id >= max_histograms");
    return ingest_host(ctx, _lk, HK_SINGLE, hid, h_values, nullptr, n);
}
extern "C" lh_status lh_ingest_keyed_f64_u16_host(lh_ctx *ctx, const uint16_t *h_ids, const double *h_values, size_t n) {
    LH_ENTER(ctx);
    if (n && (!h_ids || !h_values)) return fail(ctx, LH_ERR_INVALID, "NULL input");
    return ingest_host(ctx, _lk, HK_KEYED_U16, 0, h_values, h_ids, n);
}
extern "C" lh_status lh_ingest_keyed_i64ns_u16_host(lh_ctx *ctx, const uint16_t *h_ids, const int64_t *h_nanos, size_t n) {
    LH_ENTER(ctx);
    if (n && (!h_ids || !h_nanos)) return fail(ctx, LH_ERR_INVALID, "NULL input");
    return ingest_host(ctx, _lk, HK_KEYED_I64_U16, 0, h_nanos, h_ids, n);
}
extern "C" lh_status lh_counter_add_u16_host(lh_ctx *ctx, const uint16_t *h_ids, const uint64_t *h_amounts, size_t n) {
    LH_ENTER(ctx);
    if (n && (!h_ids || !h_amounts)) return fail(ctx, LH_ERR_INVALID, "NULL input");
    return ingest_host(ctx, _lk, HK_COUNTER_U16, 0, h_amounts, h_ids, n);
}

// Merge sparse bucket counts held in host memory (e.g. another process's lh_snapshot_export) into the ACTIVE arrays.
extern "C" lh_status lh_merge_counts_host(lh_ctx *ctx, const uint32_t *h_ids, const int16_t *h_keys, const uint64_t *h_counts, size_t n) {
    LH_ENTER(ctx);
    if (n && (!h_ids || !h_keys || !h_counts)) return fail(ctx, LH_ERR_INVALID, "NULL input");
    if (!n) return LH_OK;
    cudaStream_t s = ctx->ingest_stream;
    const int b = ctx->active;
    lh_status st = before_write(ctx, b, s);
    if (st != LH_OK) return st;
    char *d = nullptr;
    const size_t off_keys = n * 4, off_counts = ((n * 6 + 7) / 8) * 8, total = off_counts + n * 8;
    LH_CUDA(ctx, cudaMallocAsync((void **)&d, total, s));
    cudaError_t e = cudaMemcpyAsync(d, h_ids, n * 4, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d + off_keys, h_keys, n * 2, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d + off_counts, h_counts, n * 8, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) {
        int grid = grid_1d(ctx, n, 256, 1, 8);
        k_merge_sparse<<<grid, 256, 0, s>>>((const uint32_t *)d, (const short *)(d + off_keys), (const unsigned long long *)(d + off_counts),
                                            n, ctx->H, ctx->buf[b].d_buckets, ctx->buf[b].d_flags, ctx->d_dropped, ctx->pc.win);
        e = cudaGetLastError();
    }
    cudaFreeAsync(d, s);
    if (e != cudaSuccess) return fail(ctx, LH_ERR_CUDA, "lh_merge_counts_host", e);
    ctx->stats.kernel_launches++;
    ctx->stats.h2d_bytes += n * 14;
    LH_CUDA(ctx, cudaStreamSynchronize(s));   // the host arrays may be pageable: they have been read by now
    return after_write(ctx, b, s);
}

// =========================================================== staging ring
extern "C" lh_status lh_staging_acquire(lh_ctx *ctx, lh_staging *out) {
    LH_ENTER(ctx);
    if (!out) return fail(ctx, LH_ERR_INVALID, "out is NULL");
    int si;
    lh_status st = slot_wait_free(ctx, _lk, &si);
    if (st != LH_OK) return st;
    ctx->slots[si].state = SLOT_ACQUIRED;
    out->host = ctx->slots[si].h;
    out->bytes = ctx->staging_bytes;
    out->slot = (uint32_t)si;
    out->reserved = 0;
    return LH_OK;
}

namespace {
lh_status staging_commit(lh_ctx *ctx, const lh_staging *sg, HostKind kind, uint32_t hid, size_t n, uint64_t ids_offset) {
    if (!sg || sg->slot >= ctx->slots.size()) return fail(ctx, LH_ERR_INVALID, "bad staging handle");
    Slot &sl = ctx->slots[sg->slot];
    if (sl.state != SLOT_ACQUIRED) return fail(ctx, LH_ERR_STATE, "staging slot was not acquired");
    const size_t item_bytes = n * 8;
    if (kind == HK_SINGLE) {
        if (item_bytes > ctx->staging_bytes) return fail(ctx, LH_ERR_RANGE, "n exceeds the staging slot");
    } else {
        if ((ids_offset & 15u) || ids_offset < item_bytes || ids_offset + n * 2 > ctx->staging_bytes)
            return fail(ctx, LH_ERR_RANGE, "ids_offset / n do not fit the staging slot");
    }
    cudaStream_t s = ctx->ingest_stream;
    lh_status st = LH_OK;
    if (n) {
        cudaStream_t cs = ctx->copy_stream;
        if (sl.seq) LH_CUDA(ctx, cudaStreamWaitEvent(cs, sl.done, 0));
        LH_CUDA(ctx, cudaMemcpyAsync(sl.d, sl.h, item_bytes, cudaMemcpyHostToDevice, cs));
        ctx->stats.h2d_bytes += item_bytes;
        if (kind != HK_SINGLE) {
            LH_CUDA(ctx, cudaMemcpyAsync((char *)sl.d + ids_offset, (char *)sl.h + ids_offset, n * 2, cudaMemcpyHostToDevice, cs));
            ctx->stats.h2d_bytes += n * 2;
        }
        LH_CUDA(ctx, cudaEventRecord(sl.copied, cs));
        LH_CUDA(ctx, cudaStreamWaitEvent(s, sl.copied, 0));
        if (kind == HK_SINGLE) st = launch_single(ctx, hid, (const double *)sl.d, n, s);
        else if (kind == HK_KEYED_U16) st = launch_keyed<unsigned short, double>(ctx, (const unsigned short *)((char *)sl.d + ids_offset), (const double *)sl.d, n, s);
        else st = launch_counter<unsigned short>(ctx, (const unsigned short *)((char *)sl.d + ids_offset), (const uint64_t *)sl.d, n, s);
    }
    LH_CUDA(ctx, cudaEventRecord(sl.done, s));
    sl.state = SLOT_INFLIGHT;
    sl.seq = ++ctx->slot_seq;
    ctx->slot_cv.notify_all();
    return st;
}
}  // namespace

extern "C" lh_status lh_staging_commit_f64(lh_ctx *ctx, const lh_staging *s, uint32_t hid, size_t n) {
    LH_ENTER(ctx);
    if (hid >= ctx->H) return fail(ctx, LH_ERR_RANGE, "histogram_id >= max_histograms");
    return staging_commit(ctx, s, HK_SINGLE, hid, n, 0);
}
extern "C" lh_status lh_staging_commit_keyed_f64_u16(lh_ctx *ctx, const lh_staging *s, size_t n, uint64_t ids_offset) {
    LH_ENTER(ctx);
    return staging_commit(ctx, s, HK_KEYED_U16, 0, n, ids_offset);
}
extern "C" lh_status lh_staging_commit_counter_u16(lh_ctx *ctx, const lh_staging *s, size_t n, uint64_t ids_offset) {
    LH_ENTER(ctx);
    return staging_commit(ctx, s, HK_COUNTER_U16, 0, n, ids_offset);
}
extern "C" lh_status lh_staging_abandon(lh_ctx *ctx, const lh_staging *s) {
    LH_ENTER(ctx);
    if (!s || s->slot >= ctx->slots.size()) return fail(ctx, LH_ERR_INVALID, "bad staging handle");
    if (ctx->slots[s->slot].state != SLOT_ACQUIRED) return fail(ctx, LH_ERR_STATE, "staging slot was not acquired");
    ctx->slots[s->slot].state = SLOT_FREE;
    ctx->slot_cv.notify_all();
    return LH_OK;
}

// =========================================================== snapshot
extern "C" lh_status lh_snapshot_begin(lh_ctx *ctx) {
    LH_ENTER(ctx);
    if (ctx->frozen) return fail(ctx, LH_ERR_STATE, "previous snapshot not ended");
    const int f = ctx->active;
    // order the snapshot stream after every ingest launch that wrote the buffer being frozen
    for (auto &w : ctx->buf[f].writers) LH_CUDA(ctx, cudaStreamWaitEvent(ctx->snap_stream, w.ev, 0));
    if (ctx->buf[f].hot_pending) {   // drain the keyed path's uint32 window into the uint64 buckets
        lh_status st = fold_hot(ctx, f, ctx->snap_stream);
        if (st != LH_OK) return st;
    }
    ctx->active ^= 1;
    ctx->frozen = true;
    ctx->nnz_valid = false;
    ctx->view_reduced = false;
    ctx->view_counters_reduced = false;
    ctx->stats.snapshots++;
    return LH_OK;
}

extern "C" lh_status lh_snapshot_device(lh_ctx *ctx, lh_device_view *out) {
    LH_ENTER(ctx);
    if (!out) return fail(ctx, LH_ERR_INVALID, "out is NULL");
    if (!ctx->frozen) return fail(ctx, LH_ERR_STATE, "no snapshot in progress");
    const int f = ctx->active ^ 1;
    out->d_buckets = reinterpret_cast<uint64_t *>(ctx->buf[f].d_buckets);
    out->d_counters = reinterpret_cast<uint64_t *>(ctx->buf[f].d_counters);
    out->n_bucket_words = (uint64_t)ctx->H * 65536u;
    out->n_counter_words = ctx->C;
    out->stream = ctx->snap_stream;
    out->d_flags = ctx->buf[f].d_flags;
    out->n_flag_words = ctx->H;
    return LH_OK;
}

namespace {
struct ResLayout { size_t count, sum, avg, pvals, pkeys, total; };
ResLayout res_layout(size_t H, uint32_t np) {
    ResLayout l;
    l.count = 0; l.sum = H * 8; l.avg = H * 16; l.pvals = H * 24; l.pkeys = H * 24 + H * np * 8;
    l.total = l.pkeys + H * np * 4;
    return l;
}

// the arrays the open snapshot's reduction / export read: this rank's frozen buffer, or the sums over all ranks
// once lh_snapshot_allreduce has run
struct View { const unsigned long long *buckets; const uint32_t *flags; const unsigned long long *counters; };
View snapshot_view(lh_ctx *ctx) {
    const int f = ctx->active ^ 1;
    View v;
    v.buckets = ctx->view_reduced ? ctx->d_red_buckets : ctx->buf[f].d_buckets;
    v.flags = ctx->view_reduced ? ctx->d_red_flags : ctx->buf[f].d_flags;
    v.counters = ctx->view_counters_reduced ? ctx->d_red_counters : ctx->buf[f].d_counters;
    return v;
}

// enqueue the percentiles' H2D and K3 over (buckets, flags) into the packed result array d, on the snapshot stream
lh_status launch_reduce(lh_ctx *ctx, const unsigned long long *buckets, const uint32_t *flags, const double *ps, uint32_t np,
                        double *d_ps, char *d, uint32_t *d_nnz) {
    cudaStream_t s = ctx->snap_stream;
    const ResLayout l = res_layout(ctx->H, np);
    if (np) {
        LH_CUDA(ctx, cudaMemcpyAsync(d_ps, ps, np * sizeof(double), cudaMemcpyHostToDevice, s));
    }
    // shared-memory window path when the 2*win-1 cells fit comfortably (two CTAs per SM); the dense path otherwise
    const size_t cells = (size_t)2 * ctx->pc.win - 1;
    const uint32_t smem_cells = cells * 8 <= (size_t)100 * 1024 ? (uint32_t)cells : 0u;
    k_reduce<<<ctx->H, K3_THREADS, (size_t)smem_cells * 8, s>>>(buckets, flags, ctx->pc.win, ctx->d_decomp, d_ps, (int)np,
                                           (unsigned long long *)(d + l.count), (double *)(d + l.sum), (double *)(d + l.avg),
                                           (int *)(d + l.pkeys), (double *)(d + l.pvals), d_nnz, smem_cells);
    LH_CUDA(ctx, cudaGetLastError());
    ctx->stats.kernel_launches++;
    return LH_OK;
}

// copy the packed results of h (laid out by res_layout(H, np)) into the caller's arrays (any may be NULL)
void unpack_results(const char *h, size_t H, uint32_t np, uint64_t *counts, double *sums, double *avgs, int32_t *pkeys,
                    double *pvals) {
    const ResLayout l = res_layout(H, np);
    if (counts) memcpy(counts, h + l.count, H * 8);
    if (sums) memcpy(sums, h + l.sum, H * 8);
    if (avgs) memcpy(avgs, h + l.avg, H * 8);
    if (pvals && np) memcpy(pvals, h + l.pvals, H * np * 8);
    if (pkeys && np) memcpy(pkeys, h + l.pkeys, H * np * 4);
}

// Sparse lists of (buckets, flags) into x, whose d_nnz already holds K3's non-empty counts of that view, plus a copy
// of `counters`.  Synchronises the snapshot stream (twice when there is anything to list).
lh_status export_lists(lh_ctx *ctx, ExportBufs &x, const unsigned long long *buckets, const uint32_t *flags,
                       const unsigned long long *counters, lh_sparse *out) {
    cudaStream_t s = ctx->snap_stream;
    k_scan_nnz<<<1, 1024, 0, s>>>(x.d_nnz, ctx->H, x.d_offsets);
    LH_CUDA(ctx, cudaGetLastError());
    LH_CUDA(ctx, cudaMemcpyAsync(x.h_offsets, x.d_offsets, ((size_t)ctx->H + 1) * 4, cudaMemcpyDeviceToHost, s));
    LH_CUDA(ctx, cudaMemcpyAsync(x.h_counters, counters, (size_t)ctx->C * 8, cudaMemcpyDeviceToHost, s));
    LH_CUDA(ctx, cudaStreamSynchronize(s));
    const size_t total = x.h_offsets[ctx->H];
    if (total > x.cap) {
        size_t cap = std::max<size_t>(total, 4096) * 2;
        export_bufs_free_lists(x);
        LH_CUDA(ctx, cudaMalloc(&x.d_keys, cap * 2));
        LH_CUDA(ctx, cudaMalloc(&x.d_counts, cap * 8));
        LH_CUDA(ctx, cudaMallocHost(&x.h_keys, cap * 2));
        LH_CUDA(ctx, cudaMallocHost(&x.h_counts, cap * 8));
        x.cap = cap;
    }
    if (total) {
        k_export<<<ctx->H, K3_THREADS, 0, s>>>(buckets, flags, ctx->pc.win, x.d_offsets, x.d_keys, x.d_counts);
        LH_CUDA(ctx, cudaGetLastError());
        ctx->stats.kernel_launches += 2;
        LH_CUDA(ctx, cudaMemcpyAsync(x.h_keys, x.d_keys, total * 2, cudaMemcpyDeviceToHost, s));
        LH_CUDA(ctx, cudaMemcpyAsync(x.h_counts, x.d_counts, total * 8, cudaMemcpyDeviceToHost, s));
        LH_CUDA(ctx, cudaStreamSynchronize(s));
    }
    ctx->stats.d2h_bytes += total * 10 + ((size_t)ctx->H + 1) * 4 + (size_t)ctx->C * 8;
    out->offsets = x.h_offsets;
    out->keys = x.h_keys;
    out->counts = reinterpret_cast<const uint64_t *>(x.h_counts);
    out->counter_deltas = reinterpret_cast<const uint64_t *>(x.h_counters);
    out->total_entries = total;
    return LH_OK;
}

// enqueue K3 + one packed D2H for the open snapshot into result slot `slot`
lh_status enqueue_reduce(lh_ctx *ctx, const double *ps, uint32_t np, int slot) {
    cudaStream_t s = ctx->snap_stream;
    const ResLayout l = res_layout(ctx->H, np);
    const View v = snapshot_view(ctx);
    char *d = ctx->d_res[slot];
    if (lh_status st = launch_reduce(ctx, v.buckets, v.flags, ps, np, ctx->d_ps[slot], d, ctx->x.d_nnz)) return st;
    LH_CUDA(ctx, cudaMemcpyAsync(ctx->h_res[slot], d, l.total, cudaMemcpyDeviceToHost, s));
    LH_CUDA(ctx, cudaEventRecord(ctx->res_done[slot], s));
    ctx->stats.d2h_bytes += l.total;
    ctx->nnz_valid = true;
    ctx->res_np[slot] = np;
    return LH_OK;
}
}  // namespace

extern "C" lh_status lh_snapshot_reduce_async(lh_ctx *ctx, const double *percentiles, uint32_t np, uint64_t *ticket) {
    LH_ENTER(ctx);
    if (!ticket) return fail(ctx, LH_ERR_INVALID, "ticket is NULL");
    if (!ctx->frozen) return fail(ctx, LH_ERR_STATE, "no snapshot in progress");
    if (np > LH_MAX_PERCENTILES || (np && !percentiles)) return fail(ctx, LH_ERR_INVALID, "bad percentile array");
    const uint64_t t = ctx->next_ticket++;
    const int slot = (int)(t & 1);
    // the slot's previous results (ticket t-2) are overwritten: make sure its copy is not still in flight
    // (waited for with the mutex released: ingest threads are not held up)
    if (ctx->res_ticket[slot]) {
        cudaEvent_t ev = ctx->res_done[slot];
        _lk.unlock();
        cudaError_t e = cudaEventSynchronize(ev);
        _lk.lock();
        if (e != cudaSuccess) return fail(ctx, LH_ERR_CUDA, "cudaEventSynchronize(result slot)", e);
        if (!ctx->frozen) return fail(ctx, LH_ERR_STATE, "snapshot ended while waiting");
    }
    lh_status st = enqueue_reduce(ctx, percentiles, np, slot);
    if (st != LH_OK) return st;
    ctx->res_ticket[slot] = t;
    *ticket = t;
    return LH_OK;
}

extern "C" lh_status lh_snapshot_result(lh_ctx *ctx, uint64_t ticket, uint64_t *counts, double *sums, double *avgs,
                                        int32_t *pkeys, double *pvals) {
    if (!ctx) return LH_ERR_INVALID;
    const int slot = (int)(ticket & 1);
    cudaEvent_t ev;
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        if (ticket == 0 || ctx->res_ticket[slot] != ticket) return fail(ctx, LH_ERR_STATE, "ticket expired or unknown");
        ev = ctx->res_done[slot];
    }
    // wait outside the lock so ingest threads are not held up by the reaper
    cudaError_t e = cudaEventSynchronize(ev);
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (e != cudaSuccess) return fail(ctx, LH_ERR_CUDA, "cudaEventSynchronize(result)", e);
    if (ctx->res_ticket[slot] != ticket) return fail(ctx, LH_ERR_STATE, "ticket expired while waiting");
    unpack_results(ctx->h_res[slot], ctx->H, ctx->res_np[slot], counts, sums, avgs, pkeys, pvals);
    return LH_OK;
}

extern "C" lh_status lh_snapshot_reduce(lh_ctx *ctx, const double *percentiles, uint32_t np, uint64_t *counts,
                                        double *sums, double *avgs, int32_t *pkeys, double *pvals) {
    uint64_t t = 0;
    lh_status st = lh_snapshot_reduce_async(ctx, percentiles, np, &t);
    if (st != LH_OK) return st;
    return lh_snapshot_result(ctx, t, counts, sums, avgs, pkeys, pvals);
}

extern "C" lh_status lh_snapshot_export(lh_ctx *ctx, lh_sparse *out) {
    LH_ENTER(ctx);
    if (!out) return fail(ctx, LH_ERR_INVALID, "out is NULL");
    if (!ctx->frozen) return fail(ctx, LH_ERR_STATE, "no snapshot in progress");
    const View v = snapshot_view(ctx);
    if (!ctx->nnz_valid) {
        // non-empty bucket counts come out of K3: run it with no percentiles into the scratch result slot, which never
        // carries a ticket (outstanding lh_snapshot_reduce_async tickets keep their documented lifetime)
        lh_status st = enqueue_reduce(ctx, nullptr, 0, 2);
        if (st != LH_OK) return st;
    }
    return export_lists(ctx, ctx->x, v.buckets, v.flags, v.counters, out);
}

extern "C" lh_status lh_snapshot_copy_histogram(lh_ctx *ctx, uint32_t hid, uint64_t *h_out) {
    LH_ENTER(ctx);
    if (!ctx->frozen) return fail(ctx, LH_ERR_STATE, "no snapshot in progress");
    if (hid >= ctx->H) return fail(ctx, LH_ERR_RANGE, "histogram_id >= max_histograms");
    if (!h_out) return fail(ctx, LH_ERR_INVALID, "h_out is NULL");
    const View v = snapshot_view(ctx);
    LH_CUDA(ctx, cudaMemcpyAsync(h_out, v.buckets + (size_t)hid * 65536u, 65536 * 8, cudaMemcpyDeviceToHost, ctx->snap_stream));
    LH_CUDA(ctx, cudaStreamSynchronize(ctx->snap_stream));
    ctx->stats.d2h_bytes += 65536 * 8;
    return LH_OK;
}

extern "C" lh_status lh_snapshot_end(lh_ctx *ctx) {
    LH_ENTER(ctx);
    if (!ctx->frozen) return fail(ctx, LH_ERR_STATE, "no snapshot in progress");
    const int f = ctx->active ^ 1;
    cudaStream_t s = ctx->snap_stream;
    // zero only what the interval touched (flags), not the whole uint64[H][65536] array
    k_clear_touched<<<ctx->H, 256, 0, s>>>(ctx->buf[f].d_buckets, ctx->buf[f].d_flags, ctx->pc.win);
    LH_CUDA(ctx, cudaGetLastError());
    if (ctx->view_reduced) {
        k_clear_touched<<<ctx->H, 256, 0, s>>>(ctx->d_red_buckets, ctx->d_red_flags, ctx->pc.win);
        LH_CUDA(ctx, cudaGetLastError());
        ctx->stats.kernel_launches++;
    }
    ctx->stats.kernel_launches++;
    LH_CUDA(ctx, cudaMemsetAsync(ctx->buf[f].d_counters, 0, (size_t)ctx->C * 8u, s));
    LH_CUDA(ctx, cudaEventRecord(ctx->buf[f].cleared, s));
    ctx->frozen = false;
    ctx->view_reduced = false;
    ctx->view_counters_reduced = false;
    return LH_OK;
}

// =========================================================== multi-GPU (peer memory)
extern "C" lh_status lh_comm_export(lh_ctx *ctx, lh_peer_handle *out) {
    LH_ENTER(ctx);
    if (!out) return fail(ctx, LH_ERR_INVALID, "out is NULL");
    PeerWire w{};
    w.magic = kPeerMagic; w.abi = LH_ABI_VERSION; w.H = ctx->H; w.C = ctx->C;
    w.precision = (uint32_t)ctx->pc.precision; w.device = (uint32_t)ctx->device;
    w.pid = (int64_t)getpid(); w.ctx_id = ctx->ctx_id;
    for (int b = 0; b < 2; b++) {
        w.ptr_buckets[b] = (uint64_t)(uintptr_t)ctx->buf[b].d_buckets;
        w.ptr_flags[b] = (uint64_t)(uintptr_t)ctx->buf[b].d_flags;
        w.ptr_counters[b] = (uint64_t)(uintptr_t)ctx->buf[b].d_counters;
        LH_CUDA(ctx, cudaIpcGetMemHandle(&w.ipc_buckets[b], ctx->buf[b].d_buckets));
        LH_CUDA(ctx, cudaIpcGetMemHandle(&w.ipc_flags[b], ctx->buf[b].d_flags));
        LH_CUDA(ctx, cudaIpcGetMemHandle(&w.ipc_counters[b], ctx->buf[b].d_counters));
    }
    w.ptr_comm = (uint64_t)(uintptr_t)ctx->d_comm;
    LH_CUDA(ctx, cudaIpcGetMemHandle(&w.ipc_comm, ctx->d_comm));
    if (lh_status st = comm_alloc_reduced(ctx)) return st;
    w.ptr_red = (uint64_t)(uintptr_t)ctx->d_red_buckets;
    LH_CUDA(ctx, cudaIpcGetMemHandle(&w.ipc_red, ctx->d_red_buckets));
    memset(out, 0, sizeof *out);
    memcpy(out->bytes, &w, sizeof w);
    return LH_OK;
}

extern "C" lh_status lh_comm_import(lh_ctx *ctx, uint32_t rank, uint32_t world, const lh_peer_handle *all) {
    LH_ENTER(ctx);
    if (!all || world < 1 || world > (uint32_t)kMaxRanks || rank >= world) return fail(ctx, LH_ERR_INVALID, "bad rank / world / handles");
    if (ctx->frozen) return fail(ctx, LH_ERR_STATE, "lh_comm_import during a snapshot");
    comm_unmap(ctx);
    const int64_t my_pid = (int64_t)getpid();
    for (uint32_t r = 0; r < world; r++) {
        PeerWire w;
        memcpy(&w, all[r].bytes, sizeof w);
        if (w.magic != kPeerMagic || w.abi != LH_ABI_VERSION) return fail(ctx, LH_ERR_INVALID, "peer handle is not from this library version");
        if (w.H != ctx->H || w.C != ctx->C || w.precision != (uint32_t)ctx->pc.precision)
            return fail(ctx, LH_ERR_INVALID, "peer context has a different shape (max_histograms / max_counters / precision)");
        PeerMap &pm = ctx->peers[r];
        if (r == rank) {
            if (w.ctx_id != ctx->ctx_id || w.pid != my_pid) return fail(ctx, LH_ERR_INVALID, "handles[rank] is not this context's own handle");
            for (int b = 0; b < 2; b++) { pm.buckets[b] = ctx->buf[b].d_buckets; pm.flags[b] = ctx->buf[b].d_flags; pm.counters[b] = ctx->buf[b].d_counters; }
            pm.comm = ctx->d_comm;
            if (lh_status st = comm_alloc_reduced(ctx)) return st;
            pm.red = ctx->d_red_buckets;
            continue;
        }
        if (w.pid == my_pid) {
            // same process (one thread per GPU): plain peer access on the raw pointers
            if ((int)w.device != ctx->device) {
                int can = 0;
                LH_CUDA(ctx, cudaDeviceCanAccessPeer(&can, ctx->device, (int)w.device));
                if (!can) return fail(ctx, LH_ERR_NO_DEVICE, "no peer access between the two devices");
                cudaError_t e = cudaDeviceEnablePeerAccess((int)w.device, 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return fail(ctx, LH_ERR_CUDA, "cudaDeviceEnablePeerAccess", e);
                cudaGetLastError();
            }
            for (int b = 0; b < 2; b++) {
                pm.buckets[b] = (unsigned long long *)(uintptr_t)w.ptr_buckets[b];
                pm.flags[b] = (uint32_t *)(uintptr_t)w.ptr_flags[b];
                pm.counters[b] = (unsigned long long *)(uintptr_t)w.ptr_counters[b];
            }
            pm.comm = (unsigned long long *)(uintptr_t)w.ptr_comm;
            pm.red = (unsigned long long *)(uintptr_t)w.ptr_red;
        } else {
            // another process on this node: CUDA IPC mappings (NVLink peer-to-peer underneath)
            pm.ipc = true;
            for (int b = 0; b < 2; b++) {
                LH_CUDA(ctx, cudaIpcOpenMemHandle((void **)&pm.buckets[b], w.ipc_buckets[b], cudaIpcMemLazyEnablePeerAccess));
                LH_CUDA(ctx, cudaIpcOpenMemHandle((void **)&pm.flags[b], w.ipc_flags[b], cudaIpcMemLazyEnablePeerAccess));
                LH_CUDA(ctx, cudaIpcOpenMemHandle((void **)&pm.counters[b], w.ipc_counters[b], cudaIpcMemLazyEnablePeerAccess));
            }
            LH_CUDA(ctx, cudaIpcOpenMemHandle((void **)&pm.comm, w.ipc_comm, cudaIpcMemLazyEnablePeerAccess));
            LH_CUDA(ctx, cudaIpcOpenMemHandle((void **)&pm.red, w.ipc_red, cudaIpcMemLazyEnablePeerAccess));
        }
    }
    ctx->comm_rank = rank;
    ctx->comm_world = world;
    return LH_OK;
}

extern "C" lh_status lh_snapshot_allreduce(lh_ctx *ctx, uint32_t include_counters, uint64_t *seq_out) {
    LH_ENTER(ctx);
    if (!ctx->frozen) return fail(ctx, LH_ERR_STATE, "no snapshot in progress");
    if (ctx->comm_world < 2) return fail(ctx, LH_ERR_STATE, "lh_comm_import has not been called with world >= 2");
    if (ctx->view_reduced) return fail(ctx, LH_ERR_STATE, "this snapshot has already been all-reduced");
    const int f = ctx->active ^ 1;
    cudaStream_t s = ctx->snap_stream;
    PeerParams p{};
    p.rank = ctx->comm_rank; p.world = ctx->comm_world; p.H = ctx->H; p.C = ctx->C; p.win = ctx->pc.win;
    p.do_counters = include_counters ? 1u : 0u; p.frozen = (uint32_t)f;
    p.seq = ++ctx->comm_seq;
    p.timeout_ns = 10ull * 1000ull * 1000ull * 1000ull;
    for (uint32_t r = 0; r < ctx->comm_world; r++) {
        p.buckets[r] = ctx->peers[r].buckets[f];
        p.flags[r] = ctx->peers[r].flags[f];
        p.counters[r] = ctx->peers[r].counters[f];
        p.comm[r] = ctx->peers[r].comm;
    }
    p.out_buckets = ctx->d_red_buckets; p.out_flags = ctx->d_red_flags; p.out_counters = ctx->d_red_counters;
    p.block_counter = ctx->d_comm_aux; p.status = ctx->d_comm_aux + 1;
    p.cells = reinterpret_cast<unsigned long long *>(ctx->d_comm_aux + 2);
    for (uint32_t r = 0; r < ctx->comm_world; r++) p.out_peer[r] = ctx->peers[r].red;
    // payload = the window cells of every histogram that can be live; above 1 MiB the reduce-scatter + push form wins
    const size_t payload = (size_t)ctx->H * (2u * ctx->pc.win - 1u) * 8u;
    p.two_shot = payload >= (1u << 20) ? 1u : 0u;
    ctx->comm_two_shot = p.two_shot != 0;
    const int ring = (int)(p.seq % lh_ctx::kCommRing);
    // a few CTAs: the kernel shares the GPU with the next interval's ingest (which leaves k1_reserve_sms SMs free);
    // CTAs that are not resident yet simply start later (no CTA waits for another CTA of its own grid before the end)
    const size_t items = (size_t)ctx->H * (65536u / K5_CHUNK);
    int grid = (int)std::min<size_t>(items, ctx->H == 1 ? 5 : 16);
    LH_CUDA(ctx, cudaEventRecord(ctx->comm_t0[ring], s));
    if (p.two_shot) {
        // An SM sustains only ~4 GB/s of NVLink loads (measured, tools/peer_probe.py: 36 MB take 9.1 / 2.3 / 0.64 / 0.21 ms
        // on 1 / 4 / 16 / 64 SMs), so the large payload cannot hide on the few SMs the ingest kernels leave free.  It goes
        // wide and short instead: one small CTA announces this rank and waits for the peers (it may spin for as long as
        // the ranks are skewed, on one SM), then up to 128 CTAs do the sums in ~0.2 ms; the next ingest kernel's CTAs
        // start as those finish.
        PeerParams pa = p;
        pa.arrive_only = 1;
        k_peer_allreduce<<<1, K5_THREADS, ctx->H, s>>>(pa);
        LH_CUDA(ctx, cudaGetLastError());
        ctx->stats.kernel_launches++;
        grid = (int)std::min<size_t>((ctx->H + ctx->comm_world - 1) / ctx->comm_world, (size_t)std::max(1, std::min(128, ctx->sm_count - 20)));
    }
    k_peer_allreduce<<<grid, K5_THREADS, ctx->H, s>>>(p);
    LH_CUDA(ctx, cudaGetLastError());
    LH_CUDA(ctx, cudaEventRecord(ctx->comm_t1[ring], s));
    ctx->stats.kernel_launches++;
    ctx->view_reduced = true;
    ctx->view_counters_reduced = include_counters != 0;
    ctx->nnz_valid = false;
    if (seq_out) *seq_out = p.seq;
    return LH_OK;
}

extern "C" lh_status lh_comm_allreduce_ms(lh_ctx *ctx, uint64_t seq, float *ms) {
    if (!ctx || !ms) return LH_ERR_INVALID;
    cudaEvent_t e0, e1;
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        if (seq == 0 || seq > ctx->comm_seq || ctx->comm_seq - seq >= (uint64_t)lh_ctx::kCommRing)
            return fail(ctx, LH_ERR_STATE, "that all-reduce is unknown or its events were recycled");
        const int ring = (int)(seq % lh_ctx::kCommRing);
        e0 = ctx->comm_t0[ring]; e1 = ctx->comm_t1[ring];
    }
    cudaError_t e = cudaEventSynchronize(e1);
    if (e == cudaSuccess) e = cudaEventElapsedTime(ms, e0, e1);
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (e != cudaSuccess) return fail(ctx, LH_ERR_CUDA, "lh_comm_allreduce_ms", e);
    return LH_OK;
}

extern "C" lh_status lh_comm_info(lh_ctx *ctx, lh_comm_stats *out) {
    LH_ENTER(ctx);
    if (!out) return fail(ctx, LH_ERR_INVALID, "out is NULL");
    memset(out, 0, sizeof *out);
    out->rank = ctx->comm_rank; out->world = ctx->comm_world; out->allreduces = ctx->comm_seq;
    if (ctx->comm_world >= 2) {
        unsigned int aux[2] = {0, 0};
        LH_CUDA(ctx, cudaMemcpy(aux, ctx->d_comm_aux, 8, cudaMemcpyDeviceToHost));
        out->status = aux[1];
        // bytes this rank read from its peers in the last all-reduce: window (or dense) cells of every touched histogram
        unsigned long long cells = 0;
        LH_CUDA(ctx, cudaMemcpy(&cells, ctx->d_comm_aux + 2, 8, cudaMemcpyDeviceToHost));
        // one-shot: every cell from every peer; two-shot: this rank's 1/world of the cells from every peer (and as much pushed back)
        out->last_bytes_from_peers = ctx->comm_two_shot ? cells * 8u * (ctx->comm_world - 1) / ctx->comm_world : cells * 8u * (ctx->comm_world - 1);
    }
    return LH_OK;
}

// =========================================================== windows
namespace {
// offsets / flags / counters of a ring slot, on its first use
lh_status win_slot_alloc(lh_ctx *ctx, WinSlot &sl) {
    if (sl.d_offsets) return LH_OK;
    LH_CUDA(ctx, cudaMalloc(&sl.d_offsets, ((size_t)ctx->H + 1) * 4));
    LH_CUDA(ctx, cudaMalloc(&sl.d_flags, (size_t)ctx->H * 4));
    LH_CUDA(ctx, cudaMalloc(&sl.d_counters, (size_t)ctx->C * 8));
    return LH_OK;
}

WinSlotView win_slot_view(const WinSlot *sl) {
    if (!sl) return WinSlotView{nullptr, nullptr, nullptr, nullptr, nullptr};
    return WinSlotView{sl->d_offsets, sl->d_keys, sl->d_counts, sl->d_flags, sl->d_counters};
}

#define LH_WINDOW(ctx)                                                                          \
    if (!(ctx)->win) return fail((ctx), LH_ERR_STATE, "no window configured (lh_window_configure)")
}  // namespace

extern "C" lh_status lh_window_configure(lh_ctx *ctx, uint32_t intervals) {
    LH_ENTER(ctx);
    if (intervals > LH_MAX_WINDOW_INTERVALS) return fail(ctx, LH_ERR_INVALID, "intervals > LH_MAX_WINDOW_INTERVALS");
    if (ctx->frozen) return fail(ctx, LH_ERR_STATE, "lh_window_configure while a snapshot is open");
    LH_CUDA(ctx, cudaStreamSynchronize(ctx->snap_stream));   // nothing in flight may still use the old window
    window_free(ctx->win);
    ctx->win = nullptr;
    Window *w = new (std::nothrow) Window();
    if (!w) return fail(ctx, LH_ERR_NOMEM, "window");
    ctx->win = w;
    w->intervals = intervals;
    w->ring.resize(intervals ? (size_t)intervals + 1 : 1);
    const size_t H = ctx->H, C = ctx->C, acc_bytes = H * 65536u * 8u;
    cudaError_t e = cudaMalloc(&w->d_acc, acc_bytes);
    if (e == cudaSuccess) e = cudaMalloc(&w->d_flags, H * 4);
    if (e == cudaSuccess) e = cudaMalloc(&w->d_levels, H * 8);
    if (e == cudaSuccess) e = cudaMalloc(&w->d_counters, C * 8);
    if (e == cudaSuccess) e = cudaMallocHost(&w->h_total, 4);
    if (e == cudaSuccess) e = cudaMalloc(&w->d_ps, LH_MAX_PERCENTILES * sizeof(double));
    if (e == cudaSuccess) e = cudaMalloc(&w->d_res, H * (24 + LH_MAX_PERCENTILES * 12));
    if (e == cudaSuccess) e = cudaMallocHost(&w->h_res, H * (24 + LH_MAX_PERCENTILES * 12));
    if (e == cudaSuccess) e = export_bufs_alloc(w->x, H, C);
    if (e == cudaSuccess) e = cudaMemsetAsync(w->d_acc, 0, acc_bytes, ctx->snap_stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(w->d_flags, 0, H * 4, ctx->snap_stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(w->d_levels, 0, H * 8, ctx->snap_stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(w->d_counters, 0, C * 8, ctx->snap_stream);
    if (e != cudaSuccess) {
        window_free(w);
        ctx->win = nullptr;
        return fail(ctx, e == cudaErrorMemoryAllocation ? LH_ERR_NOMEM : LH_ERR_CUDA, "allocating the window", e);
    }
    return LH_OK;
}

extern "C" lh_status lh_window_release(lh_ctx *ctx) {
    LH_ENTER(ctx);
    LH_WINDOW(ctx);
    LH_CUDA(ctx, cudaStreamSynchronize(ctx->snap_stream));
    window_free(ctx->win);
    ctx->win = nullptr;
    return LH_OK;
}

// Capture the open snapshot's view as sparse lists into the next ring slot (K3's non-empty counts, the one host
// synchronisation that sizes the slot, k_export), then fold it in and the slot of K folds ago out (k_window_apply).
extern "C" lh_status lh_window_fold(lh_ctx *ctx) {
    LH_ENTER(ctx);
    LH_WINDOW(ctx);
    Window *w = ctx->win;
    if (!ctx->frozen) return fail(ctx, LH_ERR_STATE, "lh_window_fold without an open snapshot");
    if (w->folded_snapshot == ctx->stats.snapshots) return fail(ctx, LH_ERR_STATE, "this snapshot has already been folded");
    cudaStream_t s = ctx->snap_stream;
    const View v = snapshot_view(ctx);
    const uint32_t K = w->intervals;
    const size_t nslots = w->ring.size();
    WinSlot &add = w->ring[w->folds % nslots];
    const WinSlot *sub = (K && w->folds >= K) ? &w->ring[(w->folds - K) % nslots] : nullptr;
    if (lh_status st = win_slot_alloc(ctx, add)) return st;
    if (!ctx->nnz_valid) {   // the snapshot's non-empty counts, exactly as lh_snapshot_export obtains them
        if (lh_status st = enqueue_reduce(ctx, nullptr, 0, 2)) return st;
    }
    k_scan_nnz<<<1, 1024, 0, s>>>(ctx->x.d_nnz, ctx->H, add.d_offsets);
    LH_CUDA(ctx, cudaGetLastError());
    LH_CUDA(ctx, cudaMemcpyAsync(w->h_total, add.d_offsets + ctx->H, 4, cudaMemcpyDeviceToHost, s));
    LH_CUDA(ctx, cudaMemcpyAsync(add.d_flags, v.flags, (size_t)ctx->H * 4, cudaMemcpyDeviceToDevice, s));
    LH_CUDA(ctx, cudaMemcpyAsync(add.d_counters, v.counters, (size_t)ctx->C * 8, cudaMemcpyDeviceToDevice, s));
    LH_CUDA(ctx, cudaStreamSynchronize(s));
    const size_t total = *w->h_total;
    if (total > add.cap) {   // geometric growth, as the export buffers
        const size_t cap = std::max<size_t>(total, 4096) * 2;
        cudaFree(add.d_keys); cudaFree(add.d_counts);
        add.d_keys = nullptr; add.d_counts = nullptr; add.cap = 0;
        LH_CUDA(ctx, cudaMalloc(&add.d_keys, cap * 2));
        LH_CUDA(ctx, cudaMalloc(&add.d_counts, cap * 8));
        add.cap = cap;
    }
    if (total) {
        k_export<<<ctx->H, K3_THREADS, 0, s>>>(v.buckets, v.flags, ctx->pc.win, add.d_offsets, add.d_keys, add.d_counts);
        LH_CUDA(ctx, cudaGetLastError());
        ctx->stats.kernel_launches++;
    }
    k_window_apply<<<ctx->H, KW_THREADS, 0, s>>>(w->d_acc, w->d_flags, w->d_levels, w->d_counters, ctx->H, ctx->C,
                                                 win_slot_view(&add), win_slot_view(sub));
    LH_CUDA(ctx, cudaGetLastError());
    ctx->stats.kernel_launches += 2;
    add.entries = total;
    w->folds++;
    w->folded_snapshot = ctx->stats.snapshots;
    w->nnz_valid = false;
    return LH_OK;
}

extern "C" lh_status lh_window_reduce(lh_ctx *ctx, const double *percentiles, uint32_t np, uint64_t *counts, double *sums,
                                      double *avgs, int32_t *pkeys, double *pvals) {
    LH_ENTER(ctx);
    LH_WINDOW(ctx);
    if (np > LH_MAX_PERCENTILES || (np && !percentiles)) return fail(ctx, LH_ERR_INVALID, "bad percentile array");
    Window *w = ctx->win;
    const ResLayout l = res_layout(ctx->H, np);
    if (lh_status st = launch_reduce(ctx, w->d_acc, w->d_flags, percentiles, np, w->d_ps, w->d_res, w->x.d_nnz)) return st;
    LH_CUDA(ctx, cudaMemcpyAsync(w->h_res, w->d_res, l.total, cudaMemcpyDeviceToHost, ctx->snap_stream));
    LH_CUDA(ctx, cudaStreamSynchronize(ctx->snap_stream));
    ctx->stats.d2h_bytes += l.total;
    w->nnz_valid = true;
    unpack_results(w->h_res, ctx->H, np, counts, sums, avgs, pkeys, pvals);
    return LH_OK;
}

extern "C" lh_status lh_window_export(lh_ctx *ctx, lh_sparse *out) {
    LH_ENTER(ctx);
    LH_WINDOW(ctx);
    if (!out) return fail(ctx, LH_ERR_INVALID, "out is NULL");
    Window *w = ctx->win;
    if (!w->nnz_valid) {
        if (lh_status st = launch_reduce(ctx, w->d_acc, w->d_flags, nullptr, 0, w->d_ps, w->d_res, w->x.d_nnz)) return st;
        w->nnz_valid = true;
    }
    return export_lists(ctx, w->x, w->d_acc, w->d_flags, w->d_counters, out);
}

extern "C" lh_status lh_window_info(lh_ctx *ctx, lh_window_stats *out) {
    LH_ENTER(ctx);
    LH_WINDOW(ctx);
    if (!out) return fail(ctx, LH_ERR_INVALID, "out is NULL");
    const Window *w = ctx->win;
    const size_t H = ctx->H, C = ctx->C;
    memset(out, 0, sizeof *out);
    out->intervals = w->intervals;
    out->folds = w->folds;
    const uint64_t held = w->intervals ? std::min<uint64_t>(w->folds, w->intervals) : w->folds;
    out->held = (uint32_t)std::min<uint64_t>(held, UINT32_MAX);
    if (w->intervals)
        for (uint64_t i = 0; i < held; i++) out->entries_held += w->ring[(w->folds - 1 - i) % w->ring.size()].entries;
    uint64_t bytes = H * 65536u * 8u + H * 4 + H * 8 + C * 8 + LH_MAX_PERCENTILES * 8 + H * (24 + LH_MAX_PERCENTILES * 12)
                   + H * 4 + (H + 1) * 4 + w->x.cap * 10;
    for (const auto &sl : w->ring)
        if (sl.d_offsets) bytes += (H + 1) * 4 + H * 4 + C * 8 + sl.cap * 10;
    out->device_bytes = bytes;
    return LH_OK;
}

extern "C" const char *lh_keyed_kernel_name(lh_ctx *ctx) { return ctx ? ctx->keyed_kernel : ""; }

// =========================================================== probes
extern "C" lh_status lh_compress_f64(lh_ctx *ctx, const double *d_values, size_t n, int16_t *d_out, int mode, void *stream) {
    LH_ENTER(ctx);
    if (n && (!d_values || !d_out)) return fail(ctx, LH_ERR_INVALID, "NULL input");
    if (!n) return LH_OK;
    cudaStream_t s = pick_stream(ctx, stream);
    k_compress_probe<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(d_values, n, d_out, mode, ctx->pc);
    LH_CUDA(ctx, cudaGetLastError());
    return LH_OK;
}

extern "C" lh_status lh_decompress_table(lh_ctx *ctx, double *h_out) {
    LH_ENTER(ctx);
    if (!h_out) return fail(ctx, LH_ERR_INVALID, "h_out is NULL");
    LH_CUDA(ctx, cudaMemcpy(h_out, ctx->d_decomp, 65536 * sizeof(double), cudaMemcpyDeviceToHost));
    return LH_OK;
}

extern "C" lh_status lh_fastpath_margin(lh_ctx *ctx, const double *d_values, size_t n, double *h_max_err, uint64_t *h_n_slow, void *stream) {
    LH_ENTER(ctx);
    if (n && !d_values) return fail(ctx, LH_ERR_INVALID, "NULL input");
    cudaStream_t s = pick_stream(ctx, stream);
    unsigned long long *d = nullptr;
    LH_CUDA(ctx, cudaMalloc(&d, 24));
    LH_CUDA(ctx, cudaMemsetAsync(d, 0, 24, s));
    if (n) k_fastpath_margin<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(d_values, n, d, ctx->pc);
    unsigned long long h[3];
    cudaError_t e = cudaMemcpyAsync(h, d, 24, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    cudaFree(d);
    if (e != cudaSuccess) return fail(ctx, LH_ERR_CUDA, "lh_fastpath_margin", e);
    // the larger of the two estimators' errors (positive doubles order like their bit patterns)
    const unsigned long long worst = std::max(h[0], h[2]);
    if (h_max_err) memcpy(h_max_err, &worst, 8);
    if (h_n_slow) *h_n_slow = h[1];
    ctx->last_margin[0] = h[0]; ctx->last_margin[1] = h[2];
    return LH_OK;
}

// the two estimators' errors of the last lh_fastpath_margin call, separately (bucket units)
extern "C" lh_status lh_fastpath_margin_detail(lh_ctx *ctx, double *h_err_estimator1, double *h_err_estimator2) {
    LH_ENTER(ctx);
    if (h_err_estimator1) memcpy(h_err_estimator1, &ctx->last_margin[0], 8);
    if (h_err_estimator2) memcpy(h_err_estimator2, &ctx->last_margin[1], 8);
    return LH_OK;
}

// =========================================================== streams
extern "C" lh_status lh_gen_stream_f64(lh_ctx *ctx, int kind, uint64_t seed, uint64_t start, size_t n, double *d_out, void *stream) {
    LH_ENTER(ctx);
    if (n && !d_out) return fail(ctx, LH_ERR_INVALID, "d_out is NULL");
    if (!n) return LH_OK;
    k_gen_stream<<<ctx->sm_count * 8, 256, 0, pick_stream(ctx, stream)>>>(kind, seed, start, n, d_out);
    LH_CUDA(ctx, cudaGetLastError());
    return LH_OK;
}
extern "C" lh_status lh_gen_ids_u16(lh_ctx *ctx, int kind, uint64_t seed, uint64_t start, size_t n, uint32_t n_ids, uint16_t *d_out, void *stream) {
    LH_ENTER(ctx);
    if (n && !d_out) return fail(ctx, LH_ERR_INVALID, "d_out is NULL");
    if (n_ids == 0 || n_ids > 65536) return fail(ctx, LH_ERR_RANGE, "n_ids must be in 1..65536");
    if (!n) return LH_OK;
    k_gen_ids_u16<<<ctx->sm_count * 8, 256, 0, pick_stream(ctx, stream)>>>(kind, seed, start, n, n_ids, d_out);
    LH_CUDA(ctx, cudaGetLastError());
    return LH_OK;
}

// =========================================================== misc
extern "C" lh_status lh_get_stats(lh_ctx *ctx, lh_stats *out) {
    LH_ENTER(ctx);
    if (!out) return fail(ctx, LH_ERR_INVALID, "out is NULL");
    unsigned long long dropped = 0;
    LH_CUDA(ctx, cudaMemcpy(&dropped, ctx->d_dropped, 8, cudaMemcpyDeviceToHost));
    ctx->stats.dropped = dropped;
    *out = ctx->stats;
    return LH_OK;
}
extern "C" lh_status lh_sync(lh_ctx *ctx) {
    LH_ENTER(ctx);
    // this context's work only (its three streams and every caller stream that carried an ingest), not the whole
    // device: another context on the same GPU may be inside a collective that waits for THIS caller's next step
    std::vector<cudaStream_t> streams = {ctx->ingest_stream, ctx->copy_stream, ctx->snap_stream};
    for (int b = 0; b < 2; b++)
        for (auto &w : ctx->buf[b].writers)
            if (std::find(streams.begin(), streams.end(), w.stream) == streams.end()) streams.push_back(w.stream);
    _lk.unlock();
    cudaError_t e = cudaSuccess;
    for (cudaStream_t st : streams) { cudaError_t x = cudaStreamSynchronize(st); if (e == cudaSuccess) e = x; }
    _lk.lock();
    if (e != cudaSuccess) return fail(ctx, LH_ERR_CUDA, "lh_sync", e);
    for (auto &sl : ctx->slots)
        if (sl.state == SLOT_INFLIGHT && cudaEventQuery(sl.done) == cudaSuccess) sl.state = SLOT_FREE;
    cudaGetLastError();
    return LH_OK;
}
extern "C" void *lh_ingest_stream(lh_ctx *ctx) { return ctx ? (void *)ctx->ingest_stream : nullptr; }

extern "C" lh_status lh_device_alloc(lh_ctx *ctx, size_t bytes, void **d_out) {
    LH_ENTER(ctx);
    if (!d_out) return fail(ctx, LH_ERR_INVALID, "d_out is NULL");
    cudaError_t e = cudaMalloc(d_out, bytes ? bytes : 1);
    if (e != cudaSuccess) return fail(ctx, e == cudaErrorMemoryAllocation ? LH_ERR_NOMEM : LH_ERR_CUDA, "cudaMalloc", e);
    return LH_OK;
}
extern "C" lh_status lh_device_free(lh_ctx *ctx, void *d_ptr) {
    LH_ENTER(ctx);
    LH_CUDA(ctx, cudaFree(d_ptr));
    return LH_OK;
}
extern "C" lh_status lh_host_alloc_pinned(lh_ctx *ctx, size_t bytes, void **h_out) {
    LH_ENTER(ctx);
    if (!h_out) return fail(ctx, LH_ERR_INVALID, "h_out is NULL");
    cudaError_t e = cudaMallocHost(h_out, bytes ? bytes : 1);
    if (e != cudaSuccess) return fail(ctx, e == cudaErrorMemoryAllocation ? LH_ERR_NOMEM : LH_ERR_CUDA, "cudaMallocHost", e);
    return LH_OK;
}
extern "C" lh_status lh_host_free_pinned(lh_ctx *ctx, void *h_ptr) {
    LH_ENTER(ctx);
    LH_CUDA(ctx, cudaFreeHost(h_ptr));
    return LH_OK;
}
extern "C" lh_status lh_memcpy_h2d(lh_ctx *ctx, void *d_dst, const void *h_src, size_t bytes) {
    LH_ENTER(ctx);
    LH_CUDA(ctx, cudaMemcpy(d_dst, h_src, bytes, cudaMemcpyHostToDevice));
    return LH_OK;
}
extern "C" lh_status lh_memcpy_d2h(lh_ctx *ctx, void *h_dst, const void *d_src, size_t bytes) {
    LH_ENTER(ctx);
    LH_CUDA(ctx, cudaMemcpy(h_dst, d_src, bytes, cudaMemcpyDeviceToHost));
    return LH_OK;
}

extern "C" lh_status lh_tune(lh_ctx *ctx, const char *key, int64_t value) {
    LH_ENTER(ctx);
    if (!key) return fail(ctx, LH_ERR_INVALID, "key is NULL");
    if (!strcmp(key, "k1")) {
        if (value < 0 || value >= kNumK1Variants) return fail(ctx, LH_ERR_RANGE, "unknown k1 variant");
        ctx->k1_variant = (int)value;
        return LH_OK;
    }
    if (!strcmp(key, "k1_grid_mult")) {
        if (value < 1 || value > 64) return fail(ctx, LH_ERR_RANGE, "k1_grid_mult out of range");
        ctx->k1_grid_mult = (int)value;
        return LH_OK;
    }
    if (!strcmp(key, "k1_reserve_sms")) {
        if (value < 0 || value >= ctx->sm_count) return fail(ctx, LH_ERR_RANGE, "k1_reserve_sms out of range");
        ctx->k1_reserve_sms = (int)value;
        return LH_OK;
    }
    if (!strcmp(key, "keyed_mode")) {
        if (value < 0 || value > 2) return fail(ctx, LH_ERR_RANGE, "keyed_mode is 0 (auto), 1 (L2 atomics) or 2 (owner-partitioned, write-combining)");
        ctx->keyed_mode = (int)value;
        return LH_OK;
    }
    if (!strcmp(key, "wc_pf")) {
        if (value < 0 || value > 8) return fail(ctx, LH_ERR_RANGE, "wc_pf is 0 ... 8 tiles");
        ctx->wc_pf_tiles = (uint32_t)value;
        return LH_OK;
    }
    if (!strcmp(key, "wc_flush")) {
        if (value < 4096 || value > 65536) return fail(ctx, LH_ERR_RANGE, "wc_flush is 4096 ... 65536 samples");
        ctx->wc_flush_samples = (uint32_t)value;
        return LH_OK;
    }
    if (!strcmp(key, "wc_spt")) {
        if (value != 4 && value != 6 && value != 3 && value != 8)
            return fail(ctx, LH_ERR_RANGE, "wc_spt is a shape code: 6 (896 threads x 4 samples), 4 (1024 x 4), 3 (768 x 4) or 8 (512 x 8)");
        ctx->wc_spt = (int)value;
        return LH_OK;
    }
    if (!strcmp(key, "kp_chunk")) {
        if (value < (1 << 16) || value > ((int64_t)1 << 28)) return fail(ctx, LH_ERR_RANGE, "kp_chunk out of range");
        ctx->kp_chunk = value;
        return LH_OK;
    }
    if (!strcmp(key, "keyed_blocks_per_sm")) {
        if (value < 1 || value > 32) return fail(ctx, LH_ERR_RANGE, "keyed_blocks_per_sm out of range");
        ctx->keyed_blocks_per_sm = (int)value;
        return LH_OK;
    }
    return fail(ctx, LH_ERR_INVALID, "unknown tuning key");
}

extern "C" int32_t lh_k1_variant_count(void) { return kNumK1Variants; }
extern "C" int32_t lh_k1_variant_current(lh_ctx *ctx) { return ctx ? ctx->k1_variant : -1; }
extern "C" const char *lh_k1_variant_name(lh_ctx *ctx, int32_t i) {
    if (!ctx || i < 0 || i >= kNumK1Variants) return "";
    return ctx->k1[i].name;
}

extern "C" uint64_t lh_ingest_seq(lh_ctx *ctx) {
    if (!ctx) return 0;
    std::lock_guard<std::mutex> lk(ctx->mu);
    return ctx->ingest_seq;
}

extern "C" lh_status lh_kernel_ms(lh_ctx *ctx, uint64_t seq, float *ms) {
    LH_ENTER(ctx);
    if (!ms) return fail(ctx, LH_ERR_INVALID, "ms is NULL");
    if (seq == 0 || seq > ctx->ingest_seq || ctx->ingest_seq - seq >= (uint64_t)lh_ctx::kTimingRing)
        return fail(ctx, LH_ERR_STATE, "that ingest launch is unknown or its events were recycled");
    const int i = (int)((seq - 1) % lh_ctx::kTimingRing);
    LH_CUDA(ctx, cudaEventSynchronize(ctx->ev_t1s[i]));
    LH_CUDA(ctx, cudaEventElapsedTime(ms, ctx->ev_t0s[i], ctx->ev_t1s[i]));
    return LH_OK;
}

extern "C" lh_status lh_last_kernel_ms(lh_ctx *ctx, float *ms) {
    LH_ENTER(ctx);
    if (!ms) return fail(ctx, LH_ERR_INVALID, "ms is NULL");
    if (!ctx->timing_valid) return fail(ctx, LH_ERR_STATE, "no ingest kernel has been launched");
    LH_CUDA(ctx, cudaEventSynchronize(ctx->ev_t1));
    LH_CUDA(ctx, cudaEventElapsedTime(ms, ctx->ev_t0, ctx->ev_t1));
    return LH_OK;
}
