// lh_kernels.cuh -- sm_100a kernels of the loghisto hot path.
//
//   K1   k_ingest_single_*  one histogram, float64 stream -> bucket counts
//                           (compress + Histogram increment, metrics.go:273-295, 316-322)
//          _bulk  : cp.async.bulk (TMA 1-D, UBLKCP) into a shared-memory ring guarded by mbarriers, one producer
//                   warp + N consumer warps, packed-FP32 bucket arithmetic: the shipped default
//          _ldg   : 256-bit ld.global.nc loads, software-pipelined in registers, scalar fast_candidate() (first version;
//                   kept as the second, independently written evaluator the parity tests run against the oracle)
//        both privatise the histogram in shared memory (uint32 sub-histograms, ATOMS.POPC.INC) and flush once per
//        CTA with one global 64-bit atomic per non-empty bucket.
//   K1k  k_ingest_keyed_small   (id,value) pairs, as many ids per pass as fit privatised in shared memory (HBM-bound)
//        k_ingest_keyed_vec     any number of ids: one L2 RED per sample into a compact, replicated uint32 window
//        k_ingest_keyed_wc      owner-partitioned, write-combining cooperative kernel (many histograms)
//        k_ingest_keyed         scalar fallback for ragged / misaligned pieces;  k_fold_hot drains the window
//   K2   k_counter_add{_smem}   (id,amount) pairs -> counters[id]        (metrics.go:251-269)
//   K3   k_reduce               per histogram: count, sum, avg, percentiles (processHistograms + percentile,
//                               metrics.go:336-418)
//   K4   k_scan_nnz, k_export   sparse (key,count) lists (RawMetricSet.Histograms);  k_merge_sparse is the inverse
//   K5   k_peer_allreduce       multi-GPU: sums the live window of every peer's frozen arrays over NVLink peer
//                               mappings (SURVEY.md section 8e) -- no library collective
//   misc k_clear_touched, k_fill_decompress, k_compress_probe, k_fastpath_margin, k_stream_probe, k_gen_stream,
//        k_gen_ids_u16
//
// Per-histogram flags (uint32[H], one array per bucket buffer): 0 = untouched since the buffer was cleared,
// 1 = counts inside the fast window only, 3 = some count outside it.  Every kernel that adds into the uint64
// arrays raises them; the snapshot kernels (reduce, export, clear, all-reduce) scan only what they cover.
#pragma once
#include "../../include/loghisto_b200.h"
#include <type_traits>
#include "lh_device.cuh"

namespace lh {

// ---------------------------------------------------------------- helpers
// Streaming loads: read-once data, keep it out of L1 and first in line for L2 eviction.
// sm_100 has 256-bit global loads (ld.global.v4.b64 -> LDG.E.256); the L2
// eviction-priority qualifier is only accepted on those.
struct f64x4 { double a, b, c, d; };
__device__ __forceinline__ f64x4 ldg_stream_f64x4(const void *p) {
    unsigned long long a, b, c, d;
    asm volatile("ld.global.nc.L1::no_allocate.L2::evict_first.v4.b64 {%0, %1, %2, %3}, [%4];"
                 : "=l"(a), "=l"(b), "=l"(c), "=l"(d) : "l"(p));
    f64x4 r;
    r.a = __longlong_as_double((long long)a); r.b = __longlong_as_double((long long)b);
    r.c = __longlong_as_double((long long)c); r.d = __longlong_as_double((long long)d);
    return r;
}
__device__ __forceinline__ f64x4 ldg_stream_f64x2x2(const void *p) {   // two 128-bit loads (comparison variant)
    f64x4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.f64 {%0, %1}, [%2];" : "=d"(r.a), "=d"(r.b) : "l"(p));
    asm volatile("ld.global.nc.L1::no_allocate.v2.f64 {%0, %1}, [%2];" : "=d"(r.c), "=d"(r.d) : "l"((const char *)p + 16));
    return r;
}
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "LH_WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra LH_DONE_%=;\n\t"
        "bra LH_WAIT_%=;\n\t"
        "LH_DONE_%=:\n\t}"
        ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// 1-D bulk copy global -> shared, completion signalled on an mbarrier (SASS: UBLKCP).
__device__ __forceinline__ void bulk_g2s(void *smem_dst, const void *gsrc, uint32_t bytes, uint64_t *bar,
                                         uint64_t policy) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
        ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar)), "l"(policy) : "memory");
}
__device__ __forceinline__ uint64_t policy_evict_first() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}

__device__ __forceinline__ uint64_t policy_evict_last() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ void red_add_u32_keep(unsigned int *addr, unsigned int v, uint64_t policy) {
    asm volatile("red.relaxed.gpu.global.add.L2::cache_hint.u32 [%0], %1, %2;" ::"l"(addr), "r"(v), "l"(policy) : "memory");
}

// ---------------------------------------------------------------- flags
// level 1 = the histogram has counts inside the fast window, 3 = also outside it.  Plain read first: the flag is
// almost always already set, and same-address atomics from every thread would serialise in L2.
__device__ __forceinline__ void mark(uint32_t *flag, uint32_t level) {
    if ((*reinterpret_cast<volatile uint32_t *>(flag) & level) != level) atomicOr(flag, level);
}
// One count (or c of them) straight into the uint64 row of a histogram, raising its flag.
__device__ __forceinline__ void add_bucket_global(unsigned long long *__restrict__ row, uint32_t *flag, uint32_t key16,
                                                  unsigned long long c, uint32_t win) {
    atomicAdd(&row[key16], c);
    mark(flag, key16_in_window(key16, win) ? 1u : 3u);
}

// Shared sub-histogram of one histogram: [0, 2*win) slots + one trash slot that is never flushed (samples
// outside the window are counted straight into the global array and redirected there so that the shared atomic
// stays unconditional).
__device__ __forceinline__ uint32_t subhist_words(uint32_t win) { return 2u * win + 8u; }

// Flush: one 64-bit global atomic per non-empty slot, then one flag update per CTA.
__device__ __forceinline__ void flush_subhist(const uint32_t *hist, int tid, int nthreads,
                                              unsigned long long *__restrict__ counts, uint32_t *flag, uint32_t win) {
    int any = 0;
    for (uint32_t slot = tid; slot < 2u * win; slot += nthreads) {
        const uint32_t c = hist[slot];
        if (c) { atomicAdd(&counts[slot_to_key16(slot, win)], (unsigned long long)c); any = 1; }
    }
    any = __syncthreads_or(any);
    if (any && tid == 0) mark(flag, 1u);
}

// Exact slot of one sample for the fix-up paths; out-of-window keys are counted globally and sent to the trash slot.
__device__ __forceinline__ uint32_t fixup_slot(double v, const Prec &pc, unsigned long long *__restrict__ counts,
                                               uint32_t *flag) {
    const uint32_t key = key16_of(v, pc);
    uint32_t slot = key16_to_slot(key, pc.win);
    if (slot == 0xFFFFFFFFu) { add_bucket_global(counts, flag, key, 1ull, pc.win); slot = 2u * pc.win; }
    return slot;
}

// Up to three scalar stragglers on either side of the vector body (misaligned head, ragged tail).
__device__ __forceinline__ void bucket_stragglers(const double *p, int n, const Prec &pc,
                                                  unsigned long long *__restrict__ counts, uint32_t *flag) {
    for (int i = 0; i < n; i++) add_bucket_global(counts, flag, key16_of(p[i], pc), 1ull, pc.win);
}

// ------------------------------------------------------------------- K1/ldg
// First version, kept as a second evaluator: scalar fast_candidate() per sample, 256-bit loads double-buffered in
// registers.  vals32: 32-byte aligned, nvec 32-byte vectors (4 samples each).
template <int NS>
__device__ __forceinline__ void bucket_samples(const double (&v)[NS], uint32_t *hist, const Prec &pc,
                                               unsigned long long *__restrict__ counts, uint32_t *flag) {
    uint32_t idx[NS];
    bool slow[NS];
    bool any = false;
#pragma unroll
    for (int i = 0; i < NS; i++) { fast_candidate(v[i], pc, idx[i], slow[i]); any |= slow[i]; }
    if (__any_sync(0xFFFFFFFFu, any)) {
#pragma unroll
        for (int i = 0; i < NS; i++) {
            if (slow[i]) {
                const uint32_t key = exact_key16(v[i], pc.precision);
                uint32_t slot = key16_to_slot(key, pc.win);
                if (slot == 0xFFFFFFFFu) { add_bucket_global(counts, flag, key, 1ull, pc.win); slot = 2u * pc.win; }
                idx[i] = slot;
            }
        }
    }
#pragma unroll
    for (int i = 0; i < NS; i++) atomicAdd(&hist[idx[i]], 1u);
}

template <int THREADS, int UNROLL, int MINB>
__global__ void __launch_bounds__(THREADS, MINB)
k_ingest_single_ldg(const double *__restrict__ vals32, size_t nvec, const double *head, int nhead,
                    const double *tail, int ntail, unsigned long long *__restrict__ counts, uint32_t *flag, Prec pc) {
    extern __shared__ __align__(16) uint32_t s_hist[];
    for (uint32_t i = threadIdx.x; i < subhist_words(pc.win); i += THREADS) s_hist[i] = 0;
    __syncthreads();
    const char *base = reinterpret_cast<const char *>(vals32);

    constexpr size_t TILE = (size_t)THREADS * UNROLL;   // 32-byte vectors per tile
    const size_t ntiles = nvec / TILE;
    f64x4 cur[UNROLL], nxt[UNROLL];
    size_t tile = blockIdx.x;
    if (tile < ntiles) {
#pragma unroll
        for (int u = 0; u < UNROLL; u++) cur[u] = ldg_stream_f64x4(base + (tile * TILE + (size_t)u * THREADS + threadIdx.x) * 32);
    }
    while (tile < ntiles) {
        const size_t nt = tile + gridDim.x;
        if (nt < ntiles) {
#pragma unroll
            for (int u = 0; u < UNROLL; u++) nxt[u] = ldg_stream_f64x4(base + (nt * TILE + (size_t)u * THREADS + threadIdx.x) * 32);
        }
        double v[4 * UNROLL];
#pragma unroll
        for (int u = 0; u < UNROLL; u++) { v[4 * u] = cur[u].a; v[4 * u + 1] = cur[u].b; v[4 * u + 2] = cur[u].c; v[4 * u + 3] = cur[u].d; }
        bucket_samples<4 * UNROLL>(v, s_hist, pc, counts, flag);
#pragma unroll
        for (int u = 0; u < UNROLL; u++) cur[u] = nxt[u];
        tile = nt;
    }
    // partial last tile + stragglers: one CTA, bounds-checked (rare, < TILE vectors)
    if (blockIdx.x == ntiles % gridDim.x) {
        for (size_t j = ntiles * TILE * 4 + threadIdx.x; j < nvec * 4; j += THREADS)
            atomicAdd(&s_hist[fixup_slot(vals32[j], pc, counts, flag)], 1u);
        if (threadIdx.x == 0) { bucket_stragglers(head, nhead, pc, counts, flag); bucket_stragglers(tail, ntail, pc, counts, flag); }
    }
    __syncthreads();
    flush_subhist(s_hist, threadIdx.x, THREADS, counts, flag, pc.win);
}

// ------------------------------------------------------- packed-FP32 bucket arithmetic
// Same algorithm as fast_candidate() with the per-sample instruction count cut from ~30 to ~20 so that the
// kernel stays HBM-bound under sustained load (profiles/r01/sustained_probe.txt):
//   * samples are processed in pairs with Blackwell's packed FP32 ops (fma.rn.f32x2 / add.f32x2);
//   * (float)e comes from one I2FP and the -1023 bias rides in the FMA addend (Prec::kb);
//   * ONE flag per sample: estimate too close to a bucket boundary, OR x = 1+|v| outside the window
//     (x's high word >= 0x43E00000: |v| >= 2^63, Inf, NaN);
//   * the sign of v is folded into the slot (negative values land in [win, 2*win)) instead of being flagged, so a
//     stream with many negative durations (readme.md:43) stays on the fast path;
//   * the shared-memory byte offset is built as eb*a4 + (rounded bits << 2) + const: one IMAD and one LEA.
// Extra estimate error vs fast_candidate(): the float constant -1023*c2 (|err| <= 1.6e-5 bucket units at
// precision 100), still well inside eps.
// FOLD_SIGN = false: positive-only layout (rows of `win` slots); negative samples are flagged instead.
// SHIFT = 2: byte offsets into a uint32 sub-histogram; SHIFT = 0: slot indices.
template <int NS, bool FOLD_SIGN, int SHIFT = 2>
__device__ __forceinline__ void bucket_offsets_v2(const double (&v)[NS], const Prec &pc, uint32_t one_bits,
                                                  uint32_t (&off)[NS], bool (&flag)[NS]) {
    static_assert(NS % 2 == 0, "pairs");
    constexpr float MAGIC = 12582912.0f;
    const uint32_t negoff = pc.win << SHIFT;
    const uint32_t am = SHIFT ? pc.a4 : pc.a_int, cm = SHIFT ? pc.coff : pc.coff0;
#pragma unroll
    for (int i = 0; i < NS; i += 2) {
        const double x0 = __dadd_rn(1.0, fabs(v[i])), x1 = __dadd_rn(1.0, fabs(v[i + 1]));
        const uint32_t h0 = (uint32_t)__double2hiint(x0), h1 = (uint32_t)__double2hiint(x1);
        const uint32_t t0 = __funnelshift_l((uint32_t)__double2loint(x0), h0, 3);
        const uint32_t t1 = __funnelshift_l((uint32_t)__double2loint(x1), h1, 3);
        uint32_t m0, m1;
        asm("lop3.b32 %0, %1, 0x007FFFFF, %2, 0xEA;" : "=r"(m0) : "r"(t0), "r"(one_bits));   // (t & mask) | 1.0f
        asm("lop3.b32 %0, %1, 0x007FFFFF, %2, 0xEA;" : "=r"(m1) : "r"(t1), "r"(one_bits));
        float2 lg;
        asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg.x) : "f"(__uint_as_float(m0)));
        asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg.y) : "f"(__uint_as_float(m1)));
        const uint32_t e0 = h0 >> 20, e1 = h1 >> 20;                    // 1023 + e
        const float2 ef = make_float2(__uint2float_rn(e0), __uint2float_rn(e1));
        const float2 a = __ffma2_rn(ef, make_float2(pc.c2, pc.c2), make_float2(pc.kb, pc.kb));
        const float2 w = __ffma2_rn(lg, make_float2(pc.c1, pc.c1), a);
        const float2 r = __fadd2_rn(w, make_float2(MAGIC, MAGIC));
        const float2 s = __fadd2_rn(r, make_float2(-MAGIC, -MAGIC));
        const float2 d = __ffma2_rn(s, make_float2(-1.0f, -1.0f), w);   // w - s, one rounding
        if (FOLD_SIGN) {
            flag[i] = (fabsf(d.x) > pc.thresh) | (h0 >= 0x43E00000u);
            flag[i + 1] = (fabsf(d.y) > pc.thresh) | (h1 >= 0x43E00000u);
            const uint32_t n0 = (uint32_t)__double2hiint(v[i]) >> 31, n1 = (uint32_t)__double2hiint(v[i + 1]) >> 31;
            off[i] = e0 * am + (__float_as_uint(r.x) << SHIFT) + (n0 * negoff + cm);
            off[i + 1] = e1 * am + (__float_as_uint(r.y) << SHIFT) + (n1 * negoff + cm);
        } else {
            // v's high word >= 0x43E00000 unsigned: |v| >= 2^63, Inf, NaN and every negative value
            flag[i] = (fabsf(d.x) > pc.thresh) | ((uint32_t)__double2hiint(v[i]) >= 0x43E00000u);
            flag[i + 1] = (fabsf(d.y) > pc.thresh) | ((uint32_t)__double2hiint(v[i + 1]) >= 0x43E00000u);
            off[i] = e0 * am + (__float_as_uint(r.x) << SHIFT) + cm;
            off[i + 1] = e1 * am + (__float_as_uint(r.y) << SHIFT) + cm;
        }
    }
}

template <int NS, bool FOLD_SIGN>
__device__ __forceinline__ void bucket_samples_v2(const double (&v)[NS], uint32_t *hist, const Prec &pc, uint32_t one_bits,
                                                  unsigned long long *__restrict__ counts, uint32_t *gflag) {
    uint32_t off[NS];
    bool flag[NS];
    bucket_offsets_v2<NS, FOLD_SIGN>(v, pc, one_bits, off, flag);
    bool any = false;
#pragma unroll
    for (int i = 0; i < NS; i++) any |= flag[i];
    if (__any_sync(0xFFFFFFFFu, any)) {
        // only the sample positions some lane flagged are re-derived (a warp-uniform branch per position)
#pragma unroll
        for (int i = 0; i < NS; i++)
            if (__any_sync(0xFFFFFFFFu, flag[i])) {
                if (flag[i]) off[i] = fixup_slot(v[i], pc, counts, gflag) * 4u;
            }
    }
#pragma unroll
    for (int i = 0; i < NS; i++) atomicAdd(reinterpret_cast<uint32_t *>(reinterpret_cast<char *>(hist) + off[i]), 1u);
}

// --------------------------------------------------------------- read probe
// Diagnostic only (a K1 "variant" that produces NO counts): the same 256-bit streaming loads as K1/ldg with the
// bucket arithmetic replaced by an XOR fold, to separate memory-side from SM-side limits.
template <int THREADS, int UNROLL>
__global__ void __launch_bounds__(THREADS, 2)
k_stream_probe(const double *__restrict__ vals32, size_t nvec, const double *, int, const double *, int,
               unsigned long long *__restrict__ counts, uint32_t *, Prec) {
    const char *base = reinterpret_cast<const char *>(vals32);
    constexpr size_t TILE = (size_t)THREADS * UNROLL;
    const size_t ntiles = nvec / TILE;
    unsigned long long acc = 0;
    for (size_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        f64x4 v[UNROLL];
#pragma unroll
        for (int u = 0; u < UNROLL; u++) v[u] = ldg_stream_f64x4(base + (tile * TILE + (size_t)u * THREADS + threadIdx.x) * 32);
#pragma unroll
        for (int u = 0; u < UNROLL; u++)
            acc ^= f64_as_u64(v[u].a) ^ f64_as_u64(v[u].b) ^ f64_as_u64(v[u].c) ^ f64_as_u64(v[u].d);
    }
    if (acc == 0x123456789ABCDEFull) counts[65535] = acc;   // never true in practice; keeps the loads alive
}

// ------------------------------------------------------------------ K1/bulk
// Producer warp streams STAGE_BYTES tiles into a STAGES-deep shared ring with
// cp.async.bulk; CW consumer warps bucket them.  Tiles are dealt round-robin.
// FOLD_SIGN: negative samples stay on the fast path (their slot is offset by `win`) at the price of two more integer
// instructions per sample; without it they are flagged and re-derived in the fix-up.
template <int CW, int STAGES, int STAGE_BYTES, int MINB, bool FOLD_SIGN>
__global__ void __launch_bounds__((CW + 1) * 32, MINB)
k_ingest_single_bulk(const double *__restrict__ vals32, size_t nvec32, const double *head, int nhead,
                     const double *tail, int ntail, unsigned long long *__restrict__ counts, uint32_t *flag, Prec pc) {
    const double2 *vals16 = reinterpret_cast<const double2 *>(vals32);
    const size_t nvec = nvec32 * 2;   // 16-byte vectors
    constexpr int CT = CW * 32;                       // consumer threads
    constexpr int STAGE_VEC = STAGE_BYTES / 16;
    constexpr int PER_THREAD = STAGE_VEC / CT;        // double2 per consumer thread per stage
    static_assert(STAGE_VEC % CT == 0, "stage must divide evenly over consumer threads");
    extern __shared__ __align__(128) unsigned char s_raw[];
    double2 *s_data = reinterpret_cast<double2 *>(s_raw);
    uint64_t *full = reinterpret_cast<uint64_t *>(s_raw + (size_t)STAGES * STAGE_BYTES);
    uint64_t *empty = full + STAGES;
    uint32_t *s_hist = reinterpret_cast<uint32_t *>(empty + STAGES);

    const int tid = threadIdx.x;
    const int warp = tid >> 5;
    for (uint32_t i = tid; i < subhist_words(pc.win); i += (CW + 1) * 32) s_hist[i] = 0;
    if (tid == 0) {
        for (int s = 0; s < STAGES; s++) { mbar_init(&full[s], 1); mbar_init(&empty[s], CW); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    const size_t ntiles = (nvec + STAGE_VEC - 1) / STAGE_VEC;
    if (warp == CW) {
        // ===== producer =====
        if ((tid & 31) == 0) {
            const uint64_t pol = policy_evict_first();
            uint32_t it = 0;
            for (size_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x, it++) {
                const int s = it % STAGES;
                mbar_wait(&empty[s], ((it / STAGES) & 1) ^ 1);
                size_t first = tile * (size_t)STAGE_VEC;
                size_t rem = nvec - first;
                uint32_t bytes = (uint32_t)((rem < (size_t)STAGE_VEC ? rem : (size_t)STAGE_VEC) * 16);
                mbar_expect_tx(&full[s], bytes);
                bulk_g2s(s_data + (size_t)s * STAGE_VEC, vals16 + first, bytes, &full[s], pol);
            }
        }
    } else {
        // ===== consumers =====
        uint32_t one_bits;
        asm volatile("mov.b32 %0, 0x3F800000;" : "=r"(one_bits));   // opaque to constant folding: keeps LOP3 at one instruction
        uint32_t it = 0;
        for (size_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x, it++) {
            const int s = it % STAGES;
            mbar_wait(&full[s], (it / STAGES) & 1);
            const double2 *st = s_data + (size_t)s * STAGE_VEC;
            size_t first = tile * (size_t)STAGE_VEC;
            size_t rem = nvec - first;
            if (rem >= (size_t)STAGE_VEC) {
                double v[2 * PER_THREAD];
#pragma unroll
                for (int u = 0; u < PER_THREAD; u++) {
                    double2 d = st[u * CT + tid];
                    v[2 * u] = d.x; v[2 * u + 1] = d.y;
                }
                __syncwarp();
                if ((tid & 31) == 0) mbar_arrive(&empty[s]);   // registers hold the data: release early
#pragma unroll
                for (int q = 0; q < 2 * PER_THREAD; q += 4) {
                    const double v4[4] = {v[q], v[q + 1], v[q + 2], v[q + 3]};
                    bucket_samples_v2<4, FOLD_SIGN>(v4, s_hist, pc, one_bits, counts, flag);
                }
            } else {
                for (int j = tid; j < (int)rem; j += CT) {
                    double2 d = st[j];
                    atomicAdd(&s_hist[fixup_slot(d.x, pc, counts, flag)], 1u);
                    atomicAdd(&s_hist[fixup_slot(d.y, pc, counts, flag)], 1u);
                }
                __syncwarp();
                if ((tid & 31) == 0) mbar_arrive(&empty[s]);
            }
        }
        if (blockIdx.x == 0 && tid == 0) { bucket_stragglers(head, nhead, pc, counts, flag); bucket_stragglers(tail, ntail, pc, counts, flag); }
    }
    __syncthreads();
    flush_subhist(s_hist, tid, (CW + 1) * 32, counts, flag, pc.win);
}

// --------------------------------------------------------------------- K1k
// (id,value) pairs.  1024 histograms x ~4.4K live buckets cannot be privatised
// in one CTA's shared memory.  The general fallback keeps the cells in L2: a compact uint32 "hot window"
// [H][2*win] (36 MB at H = 1024, vs 512 MB for the dense uint64 arrays)
// updated with no-return atomics that carry an L2 evict_last policy, while the
// sample stream is read once with 256-bit evict_first loads so it does not push
// the cells out of the 126 MB L2.  Keys outside the window go straight to the
// uint64 array.  k_fold_hot drains the window into the uint64 buckets at every
// snapshot (and before any cell could reach 2^32).
template <typename T> __device__ __forceinline__ double sample_to_f64(T v);
template <> __device__ __forceinline__ double sample_to_f64<double>(double v) { return v; }
// float64(duration.Nanoseconds()): CVTSQ2SD, round-to-nearest-even
template <> __device__ __forceinline__ double sample_to_f64<long long>(long long v) { return __ll2double_rn(v); }

struct KeyedOut {
    unsigned int *hot;                 // [replicas][H][2*win] uint32
    unsigned long long *buckets;       // [H][65536]
    uint32_t *flags;                   // [H]
    unsigned long long *dropped;
    uint32_t H;
};

template <typename ValT>
__device__ __forceinline__ void keyed_one(uint32_t id, ValT raw, const Prec &pc, const KeyedOut &o, unsigned int *hot, uint64_t pol) {
    if (id >= o.H) { atomicAdd(o.dropped, 1ull); return; }
    double v = sample_to_f64<ValT>(raw);
    uint32_t idx; bool slow;
    fast_candidate(v, pc, idx, slow);
    if (slow) {
        uint32_t key = exact_key16(v, pc.precision);
        idx = key16_to_slot(key, pc.win);
        if (idx == 0xFFFFFFFFu) { add_bucket_global(o.buckets + (size_t)id * 65536u, o.flags + id, key, 1ull, pc.win); return; }
    }
    red_add_u32_keep(&hot[(size_t)id * (2u * pc.win) + idx], 1u, pol);
}
// The same sample straight into the uint64 arrays (one 64-bit atomic + the histogram's flag): for the few samples
// that reach the scalar kernel (ragged heads / tails) and the rare paths of the write-combining kernel, so that those
// launches leave nothing in the uint32 hot window for the snapshot to fold.
template <typename ValT>
__device__ __forceinline__ void keyed_one_direct(uint32_t id, ValT raw, const Prec &pc, const KeyedOut &o) {
    if (id >= o.H) { atomicAdd(o.dropped, 1ull); return; }
    add_bucket_global(o.buckets + (size_t)id * 65536u, o.flags + id, key16_of(sample_to_f64<ValT>(raw), pc), 1ull, pc.win);
}

// Out-of-line form for kernels whose common path must stay small (the write-combining kernel calls it for the
// ~0.05 % of samples its fast path does not cover).
template <typename ValT>
__device__ __noinline__ void keyed_one_slow(uint32_t id, unsigned long long raw, Prec pc, KeyedOut o) {
    ValT r;
    memcpy(&r, &raw, 8);
    keyed_one_direct<ValT>(id, r, pc, o);
}

template <typename IdT>
__device__ __forceinline__ void load_ids4(const IdT *ids, size_t g, uint32_t (&id4)[4]) {
    if (sizeof(IdT) == 2) {
        unsigned int lo, hi;
        asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0, %1}, [%2];" : "=r"(lo), "=r"(hi)
                     : "l"(reinterpret_cast<const char *>(ids) + g * 8));
        id4[0] = lo & 0xFFFFu; id4[1] = lo >> 16; id4[2] = hi & 0xFFFFu; id4[3] = hi >> 16;
    } else {
        asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(id4[0]), "=r"(id4[1]), "=r"(id4[2]), "=r"(id4[3])
                     : "l"(reinterpret_cast<const char *>(ids) + g * 16));
    }
}
__device__ __forceinline__ void load_vals4(const void *vals, size_t g, unsigned long long (&raw)[4]) {
    asm volatile("ld.global.nc.L1::no_allocate.L2::evict_first.v4.b64 {%0, %1, %2, %3}, [%4];"
                 : "=l"(raw[0]), "=l"(raw[1]), "=l"(raw[2]), "=l"(raw[3]) : "l"(reinterpret_cast<const char *>(vals) + g * 32));
}

// ids of one 4-sample group, kept PACKED while they wait in registers (unpacking right after the load would make the
// prefetch wait for its own data)
template <typename IdT> struct IdPack;
template <> struct IdPack<unsigned short> {
    unsigned int lo, hi;
    __device__ __forceinline__ void load(const unsigned short *ids, size_t g) {
        asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0, %1}, [%2];" : "=r"(lo), "=r"(hi) : "l"(reinterpret_cast<const char *>(ids) + g * 8));
    }
    __device__ __forceinline__ uint32_t get(int j) const { const unsigned int w = j < 2 ? lo : hi; return (j & 1) ? (w >> 16) : (w & 0xFFFFu); }
};
template <> struct IdPack<unsigned int> {
    unsigned int w[4];
    __device__ __forceinline__ void load(const unsigned int *ids, size_t g) {
        asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3])
                     : "l"(reinterpret_cast<const char *>(ids) + g * 16));
    }
    __device__ __forceinline__ uint32_t get(int j) const { return w[j]; }
};

// Vector body: every thread takes 4 consecutive pairs (one 256-bit value load, one 64/128-bit id load).
// vals must be 32-byte aligned and ids 4*sizeof(IdT)-aligned; n4 = number of 4-sample groups.
// `hot` holds `replicas` copies of the window ([replicas][H][2*win]); CTA b updates copy b % replicas, which
// divides the same-address pressure on hot cells (clustered, latency-like data) by the replica count while every
// copy stays L2-resident.  k_fold_hot sums the copies.
template <typename IdT, typename ValT, int THREADS>
__global__ void __launch_bounds__(THREADS)
k_ingest_keyed_vec(const IdT *__restrict__ ids, const ValT *__restrict__ vals, size_t n4, uint32_t replicas, KeyedOut o, Prec pc) {
    unsigned int *hot = o.hot + (size_t)(blockIdx.x % replicas) * o.H * (2u * pc.win);
    const uint64_t pol = policy_evict_last();
    const size_t stride = (size_t)gridDim.x * THREADS;
    for (size_t g = (size_t)blockIdx.x * THREADS + threadIdx.x; g < n4; g += stride) {
        unsigned long long raw[4];
        uint32_t id4[4];
        load_vals4(vals, g, raw);
        load_ids4<IdT>(ids, g, id4);
#pragma unroll
        for (int j = 0; j < 4; j++) {
            ValT r;
            memcpy(&r, &raw[j], 8);
            keyed_one<ValT>(id4[j], r, pc, o, hot, pol);
        }
    }
}

// Scalar version for ragged heads/tails and misaligned inputs.
template <typename IdT, typename ValT, int THREADS>
__global__ void __launch_bounds__(THREADS)
k_ingest_keyed(const IdT *__restrict__ ids, const ValT *__restrict__ vals, size_t n, KeyedOut o, Prec pc) {
    const size_t stride = (size_t)gridDim.x * THREADS;
    for (size_t i = (size_t)blockIdx.x * THREADS + threadIdx.x; i < n; i += stride)
        keyed_one_direct<ValT>((uint32_t)ids[i], vals[i], pc, o);
}

// ------------------------------------------------------------------ K1k/small
// Keyed ingest when only a few histograms are configured: all their windows (uint32[ids][2*win]) are privatised
// per CTA in shared memory, exactly like K1, so the kernel is HBM-bound (10 B/sample) instead of L2-atomic-bound.
// Same packed-FP32 bucket arithmetic as K1 but with positive-only rows (uint32[ids][win]) so that twice as many
// histograms fit; the ONE flag per sample also covers id >= H, and flagged samples (boundary-close estimates,
// negatives, |v| >= 2^63, NaN/Inf, bad ids) take the L2 route of keyed_one().  Windows are added into the uint32
// hot window at the end.
constexpr int KS_THREADS = 1024;
constexpr int KS_SMEM_BYTES = 196608;        // shared memory the windows of one pass may take (11 ids at precision 100)

template <typename IdT, typename ValT>
__global__ void __launch_bounds__(KS_THREADS, 1)
k_ingest_keyed_small(const IdT *__restrict__ ids, const ValT *__restrict__ vals, size_t n4,
                     uint32_t id_lo, uint32_t id_cnt, KeyedOut o, Prec pc) {
    // This launch owns ids [id_lo, id_lo + id_cnt); with more histograms than fit, the host
    // runs one pass per id sub-range over the same batch.  Samples of other valid ids are skipped; ids >= H are
    // dropped (and counted) by the pass that starts at id 0.
    extern __shared__ __align__(16) uint32_t ks_hist[];          // [id_cnt][win] + trash word
    const uint32_t row = pc.win;
    const uint32_t words = id_cnt * row;
    for (uint32_t i = threadIdx.x; i <= words; i += KS_THREADS) ks_hist[i] = 0;
    __syncthreads();
    const uint64_t pol = policy_evict_last();
    uint32_t one_bits;
    asm volatile("mov.b32 %0, 0x3F800000;" : "=r"(one_bits));
    const uint32_t trash_off = words * 4u;

    // The loop bound is warp-uniform (base index of the CTA's row of groups); lanes past the end are predicated
    // off, because the fix-up below votes with the full warp mask.
    const size_t stride = (size_t)gridDim.x * KS_THREADS;
    size_t base = (size_t)blockIdx.x * KS_THREADS;
    unsigned long long cur[4] = {0, 0, 0, 0}, nxt[4] = {0, 0, 0, 0};
    uint32_t cur_id[4] = {0, 0, 0, 0}, nxt_id[4] = {0, 0, 0, 0};
    if (base + threadIdx.x < n4) { load_vals4(vals, base + threadIdx.x, cur); load_ids4<IdT>(ids, base + threadIdx.x, cur_id); }
    for (; base < n4; base += stride) {
        const bool valid = base + threadIdx.x < n4;
        const size_t gn = base + stride + threadIdx.x;
        if (gn < n4) { load_vals4(vals, gn, nxt); load_ids4<IdT>(ids, gn, nxt_id); }
        double v[4];
#pragma unroll
        for (int i = 0; i < 4; i++) { ValT r; memcpy(&r, &cur[i], 8); v[i] = sample_to_f64<ValT>(r); }
        uint32_t off[4];
        bool flag[4];
        bucket_offsets_v2<4, false>(v, pc, one_bits, off, flag);
        bool any = false;
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const uint32_t l = cur_id[i] - id_lo;                                  // local id (wraps when below id_lo)
            const bool mine = valid & (l < id_cnt);
            const bool bad = valid & (cur_id[i] >= o.H) & (id_lo == 0);
            flag[i] = (mine & flag[i]) | bad;
            off[i] = mine ? off[i] + l * (row * 4u) : trash_off;
            any |= flag[i];
        }
        if (__any_sync(0xFFFFFFFFu, any)) {
#pragma unroll
            for (int i = 0; i < 4; i++) {
                if (!flag[i]) continue;
                ValT rv;
                memcpy(&rv, &cur[i], 8);
                // uncertain samples of a valid id could stay in shared memory; the L2 route is exact too
                // and keeps this path trivial (it handles ~0.05 % of the samples)
                keyed_one<ValT>(cur_id[i], rv, pc, o, o.hot, pol);
                off[i] = trash_off;
            }
        }
#pragma unroll
        for (int i = 0; i < 4; i++) atomicAdd(reinterpret_cast<uint32_t *>(reinterpret_cast<char *>(ks_hist) + off[i]), 1u);
#pragma unroll
        for (int i = 0; i < 4; i++) { cur[i] = nxt[i]; cur_id[i] = nxt_id[i]; }
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < words; i += KS_THREADS) {
        const uint32_t c = ks_hist[i];
        if (!c) continue;
        const uint32_t lid = i / row, slot = i - lid * row;
        atomicAdd(&o.hot[(size_t)(id_lo + lid) * (2u * pc.win) + slot], c);
    }
}

// ------------------------------------------------------------------- K1k/wc
// Many histograms (H x window does not fit one CTA's shared memory): gets the keyed path past the L2 atomic
// rate (one RED sector per sample, ~0.25 x HBM roofline) by routing every sample to the SM that OWNS its histogram.
// One persistent cooperative CTA per SM; CTA p owns the ids {p, p+P, p+2P, ...} and keeps their positive windows
// (uint32[ids_per][win]) in shared memory for the whole launch.  The stream is processed in chunks; per chunk
//   phase A  every CTA ("writer") bins its slice: bucket index via the packed-FP32 fast path, one 16-bit record
//            (lid*win + slot) per sample appended to a per-owner WRITE-COMBINING buffer in shared memory -- the
//            position comes from one returning shared atomic on the owner's fill counter (measured 3.6 cycles per
//            warp on ~148 spread addresses, profiles/r02/ubench_smem_primitives.txt; MATCH.ANY or ballot ranking
//            cost 8-16x that).  After each tile of WC_TILE samples the full 128-byte lines are copied to the
//            (owner, writer) sub-queue in global memory (L2-resident) with 128-bit stores and the remainder (< 64
//            records) moves to the front of the buffer.  Every (owner, writer) pair has its own region, so the
//            append offsets live in shared memory and no global atomic is needed;
//   barrier  grid-wide (one per chunk; sub-queues are double-buffered by chunk parity);
//   phase B  every owner drains its P sub-queues (L2 hits) into its shared-memory windows (ATOMS.POPC.INC).
// Samples the window does not cover (negative, |v| >= 2^63, NaN/Inf, estimates within eps of a bucket boundary),
// ids >= H, and records that do not fit their buffer or sub-queue (heavily skewed ids) take the exact L2-atomic
// route of keyed_one().  At the end each CTA adds its windows into the uint32 hot window.
constexpr int WC_MAX_PARTS = 160;             // owners = CTAs (one per SM)
constexpr int WC_LINE = 64;                   // records per line (128 B)

template <int SPT> struct WcShape {           // shape code -> threads x samples per thread and tile (registers per thread):
                                              // 6: 896 x 4 (72, default), 4: 1024 x 4 (64), 3: 768 x 4 (80), 8: 512 x 8 (128);
                                              // 640 x 4 and 512 x 4 were 3 - 10 % slower, and a register pipeline three tiles
                                              // deep (640 x 4, 96 registers) gained nothing over the L2 prefetch below
    static constexpr int THREADS = SPT == 4 ? 1024 : SPT == 6 ? 896 : SPT == 3 ? 768 : 512;
    static constexpr int PER = SPT == 8 ? 8 : 4;               // samples per thread per tile
    static constexpr int TILE = THREADS * PER;
};
// An owner's shared-memory buffer holds row_cap records (WcParams; 256 when it fits, else 192 or 128): < WC_LINE carried
// over from the last flush + its share of the samples binned between two flushes + ~3.5 sigma of the binomial; a record
// that does not fit takes the exact route.  Storage per owner = row_cap + one spill line (the remainder copy reads a
// whole line) + 8 records of padding so that the 128-bit accesses of the flush are bank-conflict free.
constexpr int WC_ROW_EXTRA = WC_LINE + 8;

struct WcParams {
    const void *ids;                 // IdT[n], 4*sizeof(IdT)-aligned
    const void *vals;                // ValT[n], 32-byte aligned
    size_t n;                        // multiple of the tile size (the host sends the ragged tail to k_ingest_keyed)
    const void *ids2;                // optional second segment of the same launch (ValT = double only): int64 nanosecond
    const void *vals2;               //   values (TimerToken.Stop(), metrics.go:242-246), converted with (double) like Go's
    size_t n2;                       //   float64(duration.Nanoseconds()); multiple of the tile size, 0 = none
    uint32_t ids_per;                // ceil(H / P)
    uint32_t cap;                    // records per (owner, writer) sub-queue per parity, multiple of WC_LINE
    uint32_t slice_tiles;            // tiles per CTA per chunk
    uint32_t inv_p;                  // floor(2^32 / P) + 1: id / P == __umulhi(id, inv_p) for id < 65536
    uint32_t flush_tiles;            // tiles binned between two flushes of the owner buffers
    uint32_t pf_tiles;               // the tile this many tiles past the one being loaded is asked of L2 (0 = off)
    uint32_t row_cap;                // records an owner's shared-memory buffer holds (multiple of 64; the host takes what fits)
    uint32_t row_stride;             // row_cap + one spill line + 8 records of padding (bank-conflict-free 128-bit flush)
    unsigned short *queues;          // [2][P owners][P writers][cap]
    unsigned int *q_cnt;             // [2][P owners][P writers]
    unsigned int *barrier;           // grid barrier counter, zeroed by the host before the launch
    uint4 *rare;                     // [P][WC_RARE_CAP] samples set aside for the exact path: {raw lo, raw hi, id, -}
    KeyedOut o;
};
constexpr uint32_t WC_RARE_CAP = 8192;       // per CTA and chunk; beyond that a rare sample is resolved on the spot

__device__ __forceinline__ void grid_barrier(unsigned int *bar, unsigned int target) {
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        atomicAdd(bar, 1u);
        unsigned int v;
        do {
            asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(bar) : "memory");
        } while (v < target);
    }
    __syncthreads();
}

// a record that could not be queued: add it to its bucket directly (exact, one L2 atomic; positive rows: slot == key)
__device__ __forceinline__ void wc_spill(uint32_t rec, uint32_t owner, uint32_t P, const Prec &pc, const KeyedOut &o) {
    const uint32_t lid = rec / pc.win, slot = rec - lid * pc.win, id = lid * P + owner;
    add_bucket_global(o.buckets + (size_t)id * 65536u, o.flags + id, slot, 1ull, pc.win);
}

template <typename IdT, typename ValT, int SPT, bool PAIR = false>      // PAIR: a second, int64 segment follows the float64 one
__global__ void __launch_bounds__(WcShape<SPT>::THREADS, 1)
k_ingest_keyed_wc(WcParams prm, Prec pc) {
    static_assert(!PAIR || std::is_same<ValT, double>::value, "the int64 segment rides on the float64 instantiation");
    using S = WcShape<SPT>;
    constexpr int WC_THREADS = S::THREADS;
    constexpr int GROUPS = S::PER / 4;
    extern __shared__ __align__(16) unsigned char wc_smem[];
    const uint32_t P = gridDim.x, p = blockIdx.x, tid = threadIdx.x;
    unsigned int *s_hist = reinterpret_cast<unsigned int *>(wc_smem);                       // [ids_per][win]
    const uint32_t hist_words = prm.ids_per * pc.win;
    unsigned int *s_fill = s_hist + ((hist_words + 3u) & ~3u);                              // records in each owner's buffer
    unsigned int *s_off = s_fill + WC_MAX_PARTS;                                            // records appended to my sub-queues this chunk; phase B: record counts
    unsigned short *s_buf = reinterpret_cast<unsigned short *>(s_off + WC_MAX_PARTS);       // [P + 1][STRIDE], row P = trash
    uint32_t fill_addr = smem_u32(s_fill);
    const uint32_t hist_addr = smem_u32(s_hist);
    asm volatile("mov.b32 %0, %0;" : "+r"(fill_addr));          // keep it in a register: recomputing it costs 7 instructions per tile
    const uint32_t buf_addr = fill_addr + 2u * WC_MAX_PARTS * 4u;
    unsigned int *s_rare = s_fill + (WC_MAX_PARTS - 1);                                     // samples set aside this chunk (slot P..158 of s_fill are free)
    uint4 *rareq = prm.rare + (size_t)p * WC_RARE_CAP;
    uint32_t negP = 0u - P;
    asm volatile("mov.b32 %0, %0;" : "+r"(negP));

    for (uint32_t i = tid; i < hist_words; i += WC_THREADS) s_hist[i] = 0;
    if (tid < WC_MAX_PARTS) { s_fill[tid] = 0; s_off[tid] = 0; }
    uint32_t one_bits;
    asm volatile("mov.b32 %0, 0x3F800000;" : "=r"(one_bits));
    __syncthreads();

    const size_t tiles_seg0 = prm.n / S::TILE;                   // the host passes whole tiles only
    const size_t tiles_total = tiles_seg0 + (PAIR ? prm.n2 / S::TILE : 0);    // tiles [tiles_seg0, tiles_total) are the int64 segment
    const size_t chunk_tiles = (size_t)prm.slice_tiles * P;
    const size_t nchunks = (tiles_total + chunk_tiles - 1) / chunk_tiles;
    const IdT *ids = reinterpret_cast<const IdT *>(prm.ids);
    const unsigned int cap = prm.cap;
    const uint32_t row_cap = prm.row_cap, row_stride = prm.row_stride;


    unsigned long long cur[GROUPS][4], nxt[GROUPS][4];
    IdPack<IdT> cur_id[GROUPS], nxt_id[GROUPS];
    uint32_t since_flush = 0;
    // tile `tile` = TILE consecutive samples; thread tid takes the 4-sample groups tid, tid + THREADS, ... of it.  The
    // pointers below walk the CTA's slice one tile at a time (no 64-bit multiplies inside the loop).
    const char *vptr = nullptr;                  // this thread's first 32-byte value group of the current tile
    const IdT *iptr = nullptr;                   // ... and its 4 ids
    // The register pipeline is one tile deep and the first use of a tile (DADD) is the kernel's hottest stall site: the
    // loads come back late.  A steady L2 prefetch of the tile AFTER the one being loaded turns that load into an L2 hit.
    const size_t pf_v = (size_t)prm.pf_tiles * S::TILE * 8, pf_i = (size_t)prm.pf_tiles * S::TILE;
    auto load_tile = [&](const char *vp, const IdT *ip, unsigned long long (&raw)[GROUPS][4], IdPack<IdT> (&idp)[GROUPS]) {
#pragma unroll
        for (int g = 0; g < GROUPS; g++) {
            load_vals4(vp, (size_t)g * WC_THREADS, raw[g]);
            idp[g].load(ip, (size_t)g * WC_THREADS);
        }
    };

    for (size_t c = 0; c < nchunks; c++) {
        const size_t par = c & 1;
        unsigned short *qset = prm.queues + par * (size_t)P * P * cap;      // [owner][writer][cap]
        unsigned int *cset = prm.q_cnt + par * (size_t)P * P;              // [owner][writer]
        const bool last_chunk = c + 1 == nchunks;
        // ---------------- phase A: bin my slice of chunk c (I am writer p)
        const size_t tile0 = c * chunk_tiles + (size_t)p * prm.slice_tiles;
        const uint32_t ntile_all = tile0 >= tiles_total ? 0u : (uint32_t)min((size_t)prm.slice_tiles, tiles_total - tile0);   // uniform per CTA
        // one tile: bin the 4-sample groups held in (raw, idp), then flush when due.  Two register sets alternate (A is
        // being binned while B's loads are in flight and vice versa), so no register copies between tiles.
        auto bin_tile = [&](unsigned long long (&raw)[GROUPS][4], IdPack<IdT> (&idp)[GROUPS], const bool as_i64) {
            if constexpr (PAIR) {
                if (as_i64) {                    // tile of the int64 segment (warp-uniform): from here on the bits are a float64
#pragma unroll
                    for (int g = 0; g < GROUPS; g++)
#pragma unroll
                        for (int j = 0; j < 4; j++) raw[g][j] = (unsigned long long)__double_as_longlong(__ll2double_rn((long long)raw[g][j]));
                }
            }
#pragma unroll
            for (int g = 0; g < GROUPS; g++) {
                double v[4];
#pragma unroll
                for (int j = 0; j < 4; j++) { ValT r; memcpy(&r, &raw[g][j], 8); v[j] = sample_to_f64<ValT>(r); }
                uint32_t idx[4];
                bool flag[4];
                bucket_offsets_v2<4, false, 0>(v, pc, one_bits, idx, flag);      // slot indices (positive-only rows)
                bool any = false;
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    const uint32_t id = idp[g].get(j);
                    const uint32_t lid = __umulhi(id, prm.inv_p), owner = lid * negP + id;   // id / P, id % P
                    const uint32_t rec = lid * pc.win + idx[j];
                    const bool rare = flag[j] | (id >= prm.o.H);
                    // branch-free append: rare samples draw from a trash counter (a predicated atomic makes ptxas branch and spill)
                    const uint32_t oe = rare ? P : owner;
                    uint32_t pos;
                    asm volatile("atom.shared.add.u32 %0, [%1], 1;" : "=r"(pos) : "r"(fill_addr + oe * 4u) : "memory");
                    flag[j] = rare | (pos >= row_cap);                            // buffer full (skewed ids): exact route as well
                    if (!flag[j])                                                          // one predicated store, no branch
                        asm volatile("st.shared.u16 [%0], %1;" ::"r"(buf_addr + (oe * row_stride + pos) * 2u), "h"((unsigned short)rec) : "memory");
                    any |= flag[j];
                }
                if (__any_sync(0xFFFFFFFFu, any)) {
                    // set the sample aside: the exact path (FP64 log, ~1K cycles) is run for all of them together at the end of
                    // the chunk, every lane busy, instead of stalling this warp lane by lane in the middle of the stream
#pragma unroll
                    for (int j = 0; j < 4; j++)
                        if (flag[j]) {
                            const unsigned int at = atomicAdd(s_rare, 1u);
                            if (at < WC_RARE_CAP) rareq[at] = make_uint4((unsigned int)raw[g][j], (unsigned int)(raw[g][j] >> 32), idp[g].get(j), 0u);
                            else keyed_one_slow<ValT>(idp[g].get(j), raw[g][j], pc, prm.o);
                        }
                }
            }
            // ---- flush every prm.flush_tiles tiles.  Four lanes (4 x 32 B = one 128-byte line) serve one owner, so the
            //      8 x 32 = 256 lane groups of the CTA cover all owners in ONE pass: an owner's full lines go to my sub-queue
            //      of that owner as coalesced 128-byte stores, the remainder (< 64 records) moves to the front.  No barrier
            //      is needed between tiles that do not flush: appends are atomic.
            if (++since_flush == prm.flush_tiles) {
                since_flush = 0;
                __syncthreads();
                constexpr uint32_t GROUPS_PER_WARP = 8;
                const uint32_t sub = (tid & 31) >> 2, k4 = (tid & 3) * 2;
                for (uint32_t base = (tid >> 5) * GROUPS_PER_WARP; base < P; base += (WC_THREADS / 32) * GROUPS_PER_WARP) {   // warp-uniform trip count
                    const uint32_t o = base + sub;
                    const bool act = o < P;
                    unsigned int n = 0, nfull = 0, off0 = 0;
                    uint4 keep0 = make_uint4(0, 0, 0, 0), keep1 = keep0;
                    uint4 *src = reinterpret_cast<uint4 *>(s_buf + (act ? o : 0) * row_stride);
                    if (act) {
                        n = min(s_fill[o], row_cap);
                        nfull = n / WC_LINE;
                        off0 = s_off[o];
                        unsigned short *qbase = qset + ((size_t)o * P + p) * cap;
                        keep0 = src[nfull * 8 + k4];                                       // the line that holds the remainder
                        keep1 = src[nfull * 8 + k4 + 1];
                        for (unsigned int l = 0; l < nfull; l++) {
                            if (off0 + WC_LINE <= cap) {
                                uint4 *dst = reinterpret_cast<uint4 *>(qbase + off0);
                                const uint4 a0 = src[l * 8 + k4], a1 = src[l * 8 + k4 + 1];
                                dst[k4] = a0;
                                dst[k4 + 1] = a1;
                                off0 += WC_LINE;
                            } else if (k4 == 0) {                                          // sub-queue full: these records go the L2 route
                                const unsigned short *r = s_buf + o * row_stride + l * WC_LINE;
                                for (unsigned int k = 0; k < (unsigned int)WC_LINE; k++) wc_spill(r[k], o, P, pc, prm.o);
                            }
                        }
                    }
                    __syncwarp();
                    if (act) {
                        if (nfull) { src[k4] = keep0; src[k4 + 1] = keep1; }
                        if (k4 == 0) { s_off[o] = off0; s_fill[o] = n - nfull * WC_LINE; }
                    }
                }
                __syncthreads();
            }
        };
        // the slice may straddle the two segments: part 0 = its float64 tiles, part 1 = its int64 tiles
        for (int part = 0; part < (PAIR ? 2 : 1); part++) {
            const size_t lo = part == 0 ? tile0 : max(tile0, tiles_seg0);
            const size_t hi = part == 0 ? min(tile0 + ntile_all, tiles_seg0) : tile0 + ntile_all;
            if (hi <= lo) continue;
            const uint32_t ntile = (uint32_t)(hi - lo);
            const bool as_i64 = part == 1;
            const size_t first = (part == 0 ? lo : lo - tiles_seg0) * S::TILE + (size_t)tid * 4;     // sample index inside the segment
            vptr = reinterpret_cast<const char *>(part == 0 ? prm.vals : prm.vals2) + first * 8;
            iptr = (part == 0 ? ids : reinterpret_cast<const IdT *>(prm.ids2)) + first;
            load_tile(vptr, iptr, cur, cur_id);
            auto prefetch_ahead = [&](uint32_t tile_loaded) {       // tile_loaded: index (in this part) of the tile vptr points to
                if (prm.pf_tiles && tile_loaded + prm.pf_tiles < ntile) {
#pragma unroll
                    for (int g = 0; g < GROUPS; g++) {
                        asm volatile("prefetch.global.L2 [%0];" ::"l"(vptr + pf_v + (size_t)g * WC_THREADS * 32));
                        if ((tid & 3) == 0) asm volatile("prefetch.global.L2 [%0];" ::"l"(iptr + pf_i + (size_t)g * WC_THREADS * 4));
                    }
                }
            };
            for (uint32_t t = 0; t < ntile; t += 2) {
                vptr += (size_t)S::TILE * 8;                 // -> tile t + 1
                iptr += S::TILE;
                if (t + 1 < ntile) load_tile(vptr, iptr, nxt, nxt_id);
                prefetch_ahead(t + 1);
                bin_tile(cur, cur_id, as_i64);
                if (t + 1 >= ntile) break;
                vptr += (size_t)S::TILE * 8;                 // -> tile t + 2
                iptr += S::TILE;
                if (t + 2 < ntile) load_tile(vptr, iptr, cur, cur_id);
                prefetch_ahead(t + 2);
                bin_tile(nxt, nxt_id, as_i64);
            }
        }
        __syncthreads();    // every append of this chunk's tiles is in the buffers
        {   // the samples set aside: exact path, all threads at once
            const unsigned int nr = min(*s_rare, WC_RARE_CAP);
            for (unsigned int i = tid; i < nr; i += WC_THREADS) {
                const uint4 e = rareq[i];
                ValT r;
                const unsigned long long raw = ((unsigned long long)e.y << 32) | e.x;
                memcpy(&r, &raw, 8);
                keyed_one_direct<ValT>(e.z, r, pc, prm.o);
            }
            __syncthreads();
            if (tid == 0) *s_rare = 0;
        }
        if (last_chunk) {   // everything still waiting in the buffers goes out, the last line of each owner partially filled
            if (tid < P) {
                const uint32_t o = tid;
                const unsigned int n = min(s_fill[o], row_cap);
                unsigned int off0 = s_off[o];
                const uint4 *src = reinterpret_cast<const uint4 *>(s_buf + o * row_stride);
                for (unsigned int l = 0; l * WC_LINE < n; l++) {
                    const unsigned int nrec = min((unsigned int)WC_LINE, n - l * WC_LINE);
                    if (off0 + WC_LINE <= cap) {
                        uint4 *dst = reinterpret_cast<uint4 *>(qset + ((size_t)o * P + p) * cap + off0);
#pragma unroll
                        for (int k = 0; k < 8; k++) dst[k] = src[l * 8 + k];
                        off0 += nrec;
                    } else {
                        const unsigned short *r = s_buf + o * row_stride + l * WC_LINE;
                        for (unsigned int k = 0; k < nrec; k++) wc_spill(r[k], o, P, pc, prm.o);
                    }
                }
                s_off[o] = off0;
                s_fill[o] = 0;
            }
            __syncthreads();
        }
        // publish my P record counts (zero for owners I sent nothing to), then the grid-wide barrier
        if (tid < P) { cset[(size_t)tid * P + p] = s_off[tid]; }
        grid_barrier(prm.barrier, (unsigned int)((c + 1) * (size_t)P));
        // ---------------- phase B: drain the P sub-queues I own.  The record counts go to shared memory first; then the
        // P * vq 16-byte vectors of my region are dealt to the threads as ONE flat index space (vector v belongs to
        // writer v / vq), so every thread has several independent L2 loads in flight instead of a count -> data chain.
        if (tid < P) s_off[tid] = __ldcg(&cset[(size_t)p * P + tid]);
        __syncthreads();
        {
            // warp w drains the sub-queues of writers w, w + NW, ...: the record counts are already in shared memory, so the
            // 16-byte vector loads of a sub-queue are independent (a lane has several in flight) and no index is wasted
            const unsigned short *qmine = qset + (size_t)p * P * cap;
            const uint32_t lane = tid & 31;
#define LH_WC_INC2(word)                                                                                              \
            asm volatile("red.shared.add.u32 [%0], 1;" ::"r"(hist_addr + (((word) << 2) & 0x3FFFCu)) : "memory");     \
            asm volatile("red.shared.add.u32 [%0], 1;" ::"r"(hist_addr + (((word) >> 14) & 0x3FFFCu)) : "memory");
            for (uint32_t w = tid >> 5; w < P; w += WC_THREADS / 32) {
                const unsigned int cnt = s_off[w];
                const unsigned short *q = qmine + (size_t)w * cap;
                const uint4 *qv = reinterpret_cast<const uint4 *>(q);
                const unsigned int nv = cnt >> 3;
#pragma unroll 2
                for (unsigned int i = lane; i < nv; i += 32) {
                    const uint4 v4 = __ldcg(qv + i);
                    LH_WC_INC2(v4.x) LH_WC_INC2(v4.y) LH_WC_INC2(v4.z) LH_WC_INC2(v4.w)
                }
                const unsigned int r0 = nv * 8u + lane;                                    // the < 8 records after the last full vector
                if (r0 < cnt) asm volatile("red.shared.add.u32 [%0], 1;" ::"r"(hist_addr + (unsigned int)__ldcg(q + r0) * 4u) : "memory");
            }
#undef LH_WC_INC2
        }
        __syncthreads();
        if (tid < P) s_off[tid] = 0;
        // no grid barrier here: the next chunk writes the other parity; this parity is rewritten only after the
        // next grid barrier, which every CTA reaches after finishing this drain
    }
    __syncthreads();
    // ---------------- flush my windows straight into the uint64 bucket arrays (positive rows: slot == key) and raise the
    // flags of the histograms that received counts; nothing of the common path goes through the uint32 hot window
    for (uint32_t lid = 0; lid < prm.ids_per; lid++) {
        const uint32_t id = lid * P + p;
        if (id >= prm.o.H) break;
        int any = 0;
        for (uint32_t slot = tid; slot < pc.win; slot += WC_THREADS) {
            const unsigned int cnt = s_hist[lid * pc.win + slot];
            if (cnt) { atomicAdd(&prm.o.buckets[(size_t)id * 65536u + slot], (unsigned long long)cnt); any = 1; }
        }
        any = __syncthreads_or(any);
        if (any && tid == 0) mark(&prm.o.flags[id], 1u);
    }
}

// Drain the hot window into the uint64 buckets.  atomicExch/atomicAdd so that ingest on other
// streams may keep running against the same buffer.
__global__ void k_fold_hot(unsigned int *__restrict__ hot, unsigned long long *__restrict__ buckets, uint32_t *__restrict__ flags,
                           size_t cells, uint32_t replicas, uint32_t win) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const uint32_t row = 2u * win;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < cells; i += stride) {
        unsigned long long sum = 0;
        for (uint32_t r = 0; r < replicas; r++) {
            unsigned int *cell = hot + (size_t)r * cells + i;
            if (*cell) sum += atomicExch(cell, 0u);
        }
        if (sum) {
            size_t h = i / row;
            uint32_t slot = (uint32_t)(i - h * row);
            atomicAdd(&buckets[h * 65536u + slot_to_key16(slot, win)], sum);
            mark(&flags[h], 1u);
        }
    }
}

// ---------------------------------------------------------------------- K2
// Counter(name, amount): counters[id] += amount (wrapping uint64).  Up to
// K2_SMEM_COUNTERS ids are privatised per CTA as lo/hi uint32 halves in shared
// memory: one returning shared atomic on the low half, a second one on the
// high half only when the amount has high bits or the low half carried.
constexpr int K2_SMEM_COUNTERS = 8192;

template <typename IdT, int THREADS>
__global__ void __launch_bounds__(THREADS)
k_counter_add_smem(const IdT *__restrict__ ids, const unsigned long long *__restrict__ amounts, size_t n,
                   unsigned long long *__restrict__ counters, uint32_t C,
                   unsigned long long *__restrict__ dropped) {
    extern __shared__ unsigned int s_cnt[];          // [C] low halves, [C] high halves
    unsigned int *lo = s_cnt, *hi = s_cnt + C;
    for (uint32_t i = threadIdx.x; i < 2 * C; i += THREADS) s_cnt[i] = 0;
    __syncthreads();
    const size_t stride = (size_t)gridDim.x * THREADS;
    for (size_t i = (size_t)blockIdx.x * THREADS + threadIdx.x; i < n; i += stride) {
        uint32_t id = (uint32_t)ids[i];
        unsigned long long amt = amounts[i];
        if (id >= C) { atomicAdd(dropped, 1ull); continue; }
        unsigned int a_lo = (unsigned int)amt, a_hi = (unsigned int)(amt >> 32);
        unsigned int old = atomicAdd(&lo[id], a_lo);
        a_hi += (old + a_lo < old) ? 1u : 0u;        // carry out of the low half
        if (a_hi) atomicAdd(&hi[id], a_hi);
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < C; i += THREADS) {
        unsigned long long v = ((unsigned long long)hi[i] << 32) | lo[i];
        if (v) atomicAdd(&counters[i], v);
    }
}

// Vector body: 4 consecutive (id, amount) pairs per thread and iteration (one 256-bit amount load, one 64/128-bit id
// load), the next group prefetched while the current one is added.  amounts 32-byte aligned, ids 4*sizeof(IdT)-aligned.
template <typename IdT, int THREADS>
__global__ void __launch_bounds__(THREADS)
k_counter_add_smem_vec(const IdT *__restrict__ ids, const unsigned long long *__restrict__ amounts, size_t n4,
                       unsigned long long *__restrict__ counters, uint32_t C, unsigned long long *__restrict__ dropped) {
    extern __shared__ unsigned int s_cnt[];          // [C] low halves, [C] high halves
    unsigned int *lo = s_cnt, *hi = s_cnt + C;
    for (uint32_t i = threadIdx.x; i < 2 * C; i += THREADS) s_cnt[i] = 0;
    __syncthreads();
    const size_t stride = (size_t)gridDim.x * THREADS;
    size_t g = (size_t)blockIdx.x * THREADS + threadIdx.x;
    unsigned long long cur[4], nxt[4];
    IdPack<IdT> cid, nid;
    if (g < n4) { load_vals4(amounts, g, cur); cid.load(ids, g); }
    for (; g < n4; g += stride) {
        const size_t gn = g + stride;
        if (gn < n4) { load_vals4(amounts, gn, nxt); nid.load(ids, gn); }
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const uint32_t id = cid.get(j);
            const unsigned long long amt = cur[j];
            if (id >= C) { atomicAdd(dropped, 1ull); continue; }
            const unsigned int a_lo = (unsigned int)amt;
            unsigned int a_hi = (unsigned int)(amt >> 32);
            const unsigned int old = atomicAdd(&lo[id], a_lo);
            a_hi += (old + a_lo < old) ? 1u : 0u;        // carry out of the low half
            if (a_hi) atomicAdd(&hi[id], a_hi);
        }
#pragma unroll
        for (int j = 0; j < 4; j++) cur[j] = nxt[j];
        cid = nid;
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < C; i += THREADS) {
        unsigned long long v = ((unsigned long long)hi[i] << 32) | lo[i];
        if (v) atomicAdd(&counters[i], v);
    }
}

template <typename IdT, int THREADS>
__global__ void __launch_bounds__(THREADS)
k_counter_add(const IdT *__restrict__ ids, const unsigned long long *__restrict__ amounts, size_t n,
              unsigned long long *__restrict__ counters, uint32_t C,
              unsigned long long *__restrict__ dropped) {
    const size_t stride = (size_t)gridDim.x * THREADS;
    for (size_t i = (size_t)blockIdx.x * THREADS + threadIdx.x; i < n; i += stride) {
        uint32_t id = (uint32_t)ids[i];
        if (id < C) atomicAdd(&counters[id], amounts[i]);
        else atomicAdd(dropped, 1ull);
    }
}

// ------------------------------------------------------------------- merge
// Adds sparse (histogram id, int16 key, uint64 count) triples -- the wire format lh_snapshot_export produces --
// into the bucket arrays: merging snapshots from other hosts / GPUs is the same commutative uint64 sum.
__global__ void k_merge_sparse(const uint32_t *__restrict__ ids, const short *__restrict__ keys,
                               const unsigned long long *__restrict__ counts, size_t n, uint32_t H,
                               unsigned long long *__restrict__ buckets, uint32_t *__restrict__ flags,
                               unsigned long long *__restrict__ dropped, uint32_t win) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const uint32_t id = ids[i];
        if (id >= H) { atomicAdd(dropped, 1ull); continue; }
        add_bucket_global(buckets + (size_t)id * 65536u, flags + id, (uint32_t)(int)keys[i] & 0xFFFFu, counts[i], win);
    }
}

// ---------------------------------------------------------------------- K3
// One CTA per histogram, 32 warps.  Warp w owns the 2048 consecutive keys
// [-32768 + 2048 w, +2047] (ascending key == ascending value, the order
// percentile() sorts into, metrics.go:409) and reads them as 64 coalesced
// 256-byte rows.  Pass 1: per-warp count / sum / non-empty totals, then a scan
// over the 32 warp totals.  Pass 2: the warp whose range contains a
// percentile's crossing walks its rows again (L2 hits) with a warp prefix sum
// and applies the reference's rule float64(sofar)/float64(total) >= p
// (metrics.go:413) to non-empty buckets only.
// The histogram's flag prunes the scan: untouched histograms are answered without reading a bucket, and when
// every count lies in the fast window only the (at most 6) warps that overlap it read anything.
constexpr int K3_THREADS = 1024;
constexpr int K3_WARP_KEYS = 2048;

__device__ __forceinline__ bool warp_scans(int key0, uint32_t level, uint32_t win) {
    if (level & 2u) return true;
    return key0 <= (int)win - 1 && key0 + K3_WARP_KEYS - 1 >= -((int)win - 1);
}

__device__ __forceinline__ void reduce_dense(uint32_t level, const unsigned long long *__restrict__ buckets, const uint32_t *__restrict__ flags, uint32_t win,
         const double *__restrict__ decomp,
         const double *__restrict__ ps, int np, unsigned long long *__restrict__ out_count,
         double *__restrict__ out_sum, double *__restrict__ out_avg, int *__restrict__ out_pkeys,
         double *__restrict__ out_pvals, uint32_t *__restrict__ out_nnz) {
    __shared__ unsigned long long s_cnt[32];    // per-warp totals, then exclusive prefix
    __shared__ unsigned long long s_tot[32];    // per-warp totals (kept)
    __shared__ double s_sum[32];
    __shared__ unsigned int s_nnz[32];
    __shared__ int s_owner[LH_MAX_PCT];
    __shared__ unsigned long long s_total;
    const int h = blockIdx.x, t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const unsigned long long *hb = buckets + (size_t)h * 65536u;
    const int key0 = -32768 + warp * K3_WARP_KEYS;
    const bool scans = warp_scans(key0, level, win);

    unsigned long long mine = 0;
    double msum = 0.0;
    unsigned int nnz = 0;
    if (scans) {
#pragma unroll 16
        for (int r = 0; r < K3_WARP_KEYS / 32; r++) {      // 16 independent 256-byte rows in flight per warp
            unsigned int slot = (unsigned int)(key0 + r * 32 + lane) & 0xFFFFu;
            unsigned long long c = hb[slot];
            if (c) { mine += c; msum += decomp[slot] * (double)c; nnz++; }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        mine += __shfl_xor_sync(0xFFFFFFFFu, mine, o);
        msum += __shfl_xor_sync(0xFFFFFFFFu, msum, o);
        nnz += __shfl_xor_sync(0xFFFFFFFFu, nnz, o);
    }
    if (lane == 0) { s_cnt[warp] = mine; s_tot[warp] = mine; s_sum[warp] = msum; s_nnz[warp] = nnz; }
    if (t < LH_MAX_PCT) s_owner[t] = 0x7FFFFFFF;
    __syncthreads();
    if (warp == 0) {
        unsigned long long w = s_cnt[lane], wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            unsigned long long y = __shfl_up_sync(0xFFFFFFFFu, wi, o);
            if (lane >= o) wi += y;
        }
        s_cnt[lane] = wi - w;
        if (lane == 31) s_total = wi;
        double ts = s_sum[lane];
        unsigned int tn = s_nnz[lane];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            ts += __shfl_xor_sync(0xFFFFFFFFu, ts, o);
            tn += __shfl_xor_sync(0xFFFFFFFFu, tn, o);
        }
        if (lane == 0) { s_sum[0] = ts; s_nnz[0] = tn; }
    }
    __syncthreads();
    const unsigned long long total = s_total;
    const double ftotal = (double)total;
    // owner of percentile j = first non-empty warp whose inclusive prefix satisfies the rule
    if (lane == 0 && s_tot[warp]) {
        const unsigned long long end_incl = s_cnt[warp] + s_tot[warp];
        for (int j = 0; j < np; j++)
            if (__ddiv_rn((double)end_incl, ftotal) >= ps[j]) atomicMin(&s_owner[j], warp);
    }
    __syncthreads();
    unsigned int pending = 0;
    for (int j = 0; j < np; j++) if (s_owner[j] == warp) pending |= 1u << j;
    if (pending) {
        unsigned long long sofar = s_cnt[warp];
        for (int r = 0; r < K3_WARP_KEYS / 32 && pending; r++) {
            int key = key0 + r * 32 + lane;
            unsigned long long c = hb[(unsigned int)key & 0xFFFFu];
            unsigned long long incl = c;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                unsigned long long y = __shfl_up_sync(0xFFFFFFFFu, incl, o);
                if (lane >= o) incl += y;
            }
            const double frac = __ddiv_rn((double)(sofar + incl), ftotal);
            for (int j = 0; j < np; j++) {
                if (!(pending >> j & 1u)) continue;
                unsigned int hit = __ballot_sync(0xFFFFFFFFu, c != 0 && frac >= ps[j]);
                if (hit) {
                    if (lane == __ffs(hit) - 1) {
                        out_pkeys[(size_t)h * np + j] = key;
                        out_pvals[(size_t)h * np + j] = decomp[(unsigned int)key & 0xFFFFu];
                    }
                    pending &= ~(1u << j);
                }
            }
            sofar += __shfl_sync(0xFFFFFFFFu, incl, 31);
        }
    }
    if (t == 0) {
        for (int j = 0; j < np; j++)
            if (s_owner[j] == 0x7FFFFFFF) {   // percentile() error (p > 1, NaN, empty): key omitted by the caller
                out_pkeys[(size_t)h * np + j] = (int)0x80000000;
                out_pvals[(size_t)h * np + j] = __longlong_as_double(0x7FF8000000000000ll);
            }
        out_count[h] = total;
        out_sum[h] = s_sum[0];
        out_avg[h] = __ddiv_rn(s_sum[0], ftotal);    // metrics.go:356 (NaN when empty)
        out_nnz[h] = s_nnz[0];
    }
}

// Smallest s in [0, total] with float64(s)/float64(total) >= p -- the reference's rule (metrics.go:413) turned into an
// integer threshold on the running count: the quotient is monotone in s, so "first non-empty bucket whose running count
// satisfies the rule" == "first non-empty bucket whose running count reaches T".  Returns false when no s satisfies
// the rule (p > 1 or NaN: percentile() returns its error).
__device__ __forceinline__ bool percentile_threshold(double p, unsigned long long total, unsigned long long *T) {
    const double ft = (double)total;
    if (!(__ddiv_rn(ft, ft) >= p)) return false;                 // even s = total fails (p > 1, NaN)
    auto ok = [&](unsigned long long s) { return __ddiv_rn((double)s, ft) >= p; };
    unsigned long long s = 0;
    if (p > 0.0) {
        const double est = ceil(p * ft);
        s = est >= ft ? total : (unsigned long long)est;
    }
    int steps = 0;
    while (s > 0 && ok(s - 1) && steps < 8) { s--; steps++; }
    while (!ok(s) && steps < 16) { s++; steps++; }
    if (steps >= 8 && (!ok(s) || (s > 0 && ok(s - 1)))) {        // long plateaus of float64(s) (totals beyond 2^53): bisection
        unsigned long long lo = 0, hi = total;                  // ok(hi) holds
        while (lo < hi) { const unsigned long long mid = lo + (hi - lo) / 2; if (ok(mid)) hi = mid; else lo = mid + 1; }
        s = lo;
    }
    *T = s;
    return true;
}

// One CTA per histogram.  Untouched histograms are answered without reading a bucket.  A histogram whose counts all
// lie in the fast window (flag 1; the normal case) is reduced from shared memory: its 2*win-1 cells are loaded once
// (ascending key order == ascending value order, metrics.go:409), count / sum / non-empty totals come from a block
// reduction, an in-place block scan turns the cells into running counts, and every percentile is one binary search
// for its integer threshold -- no per-bucket FP64 division, no serial walk.  Histograms with out-of-window keys
// (wrapped int16 keys, NaN / Inf -> 0 ...) take the dense path over all 65 536 keys.
__global__ void __launch_bounds__(K3_THREADS)
k_reduce(const unsigned long long *__restrict__ buckets, const uint32_t *__restrict__ flags, uint32_t win,
         const double *__restrict__ decomp,
         const double *__restrict__ ps, int np, unsigned long long *__restrict__ out_count,
         double *__restrict__ out_sum, double *__restrict__ out_avg, int *__restrict__ out_pkeys,
         double *__restrict__ out_pvals, uint32_t *__restrict__ out_nnz, uint32_t smem_cells) {
    extern __shared__ __align__(16) unsigned long long k3_cells[];      // [2*win-1] when the window path is enabled
    const int h = blockIdx.x, t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const uint32_t level = flags[h];
    if (level == 0) {   // untouched this interval: the caller reports the histogram as absent
        if (t == 0) {
            out_count[h] = 0; out_sum[h] = 0.0; out_avg[h] = __longlong_as_double(0x7FF8000000000000ll); out_nnz[h] = 0;
            for (int j = 0; j < np; j++) {
                out_pkeys[(size_t)h * np + j] = (int)0x80000000;
                out_pvals[(size_t)h * np + j] = __longlong_as_double(0x7FF8000000000000ll);
            }
        }
        return;
    }
    const uint32_t n = 2u * win - 1u;
    if ((level & 2u) || smem_cells < n) {
        reduce_dense(level, buckets, flags, win, decomp, ps, np, out_count, out_sum, out_avg, out_pkeys, out_pvals, out_nnz);
        return;
    }
    __shared__ unsigned long long s_c[32];
    __shared__ double s_s[32];
    __shared__ unsigned int s_n[32];
    __shared__ unsigned long long s_total;
    const unsigned long long *hb = buckets + (size_t)h * 65536u;
    // cell i of the window holds key i - (win-1)
    constexpr int PER = 32;                                       // contiguous cells per thread in the scan (PER * 1024 >= n up to win = 16384)
    unsigned long long mine = 0;
    double msum = 0.0;
    unsigned int nnz = 0;
    for (uint32_t i = t; i < n; i += K3_THREADS) {
        const unsigned int slot = (unsigned int)((int)i - (int)(win - 1u)) & 0xFFFFu;
        const unsigned long long c = hb[slot];
        k3_cells[i] = c;
        if (c) { mine += c; msum += decomp[slot] * (double)c; nnz++; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        mine += __shfl_xor_sync(0xFFFFFFFFu, mine, o);
        msum += __shfl_xor_sync(0xFFFFFFFFu, msum, o);
        nnz += __shfl_xor_sync(0xFFFFFFFFu, nnz, o);
    }
    if (lane == 0) { s_c[warp] = mine; s_s[warp] = msum; s_n[warp] = nnz; }
    __syncthreads();
    if (warp == 0) {
        unsigned long long c = s_c[lane];
        double sm = s_s[lane];
        unsigned int nz = s_n[lane];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            c += __shfl_xor_sync(0xFFFFFFFFu, c, o);
            sm += __shfl_xor_sync(0xFFFFFFFFu, sm, o);
            nz += __shfl_xor_sync(0xFFFFFFFFu, nz, o);
        }
        if (lane == 0) {
            s_total = c;
            out_count[h] = c;
            out_sum[h] = sm;
            out_avg[h] = __ddiv_rn(sm, (double)c);                // metrics.go:356
            out_nnz[h] = nz;
        }
    }
    // in-place inclusive scan of the cells: thread t owns cells [t*per, (t+1)*per)
    const uint32_t per = (n + K3_THREADS - 1) / K3_THREADS;
    const uint32_t first = t * per, last = min(first + per, n);
    unsigned long long local = 0;
    for (uint32_t i = first; i < last; i++) local += k3_cells[i];
    unsigned long long incl = local;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long y = __shfl_up_sync(0xFFFFFFFFu, incl, o);
        if (lane >= o) incl += y;
    }
    __syncthreads();                                              // s_c was read by warp 0 above
    if (lane == 31) s_c[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        unsigned long long w = s_c[lane], wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long y = __shfl_up_sync(0xFFFFFFFFu, wi, o);
            if (lane >= o) wi += y;
        }
        s_c[lane] = wi - w;                                       // exclusive prefix of the warp totals
    }
    __syncthreads();
    unsigned long long run = s_c[warp] + incl - local;
    for (uint32_t i = first; i < last; i++) { run += k3_cells[i]; k3_cells[i] = run; }
    __syncthreads();
    (void)PER;
    // one thread per percentile: integer threshold, then the first cell whose running count reaches it
    if (t < np) {
        const unsigned long long total = s_total;
        unsigned long long T;
        int key = (int)0x80000000;
        double val = __longlong_as_double(0x7FF8000000000000ll);
        if (total && percentile_threshold(ps[t], total, &T)) {
            if (T == 0) T = 1;                                    // p <= 0: the smallest non-empty bucket
            uint32_t lo = 0, hi = n - 1;                          // k3_cells[n-1] == total >= T
            while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (k3_cells[mid] >= T) hi = mid; else lo = mid + 1; }
            key = (int)lo - (int)(win - 1u);
            val = decomp[(unsigned int)key & 0xFFFFu];
        }
        out_pkeys[(size_t)h * np + t] = key;
        out_pvals[(size_t)h * np + t] = val;
    }
}

// ---------------------------------------------------------------------- K4
// offsets[h] = exclusive prefix of nnz (computed by k_scan_nnz); entries are
// written in ascending key order.
__global__ void k_scan_nnz(const uint32_t *__restrict__ nnz, uint32_t H, uint32_t *__restrict__ offsets) {
    // single CTA, H is small (<= a few thousand): serial per-chunk scan is fine
    __shared__ uint32_t s_part[1024];
    const int t = threadIdx.x;
    const uint32_t per = (H + 1023u) / 1024u;
    uint32_t a = 0;
    for (uint32_t i = 0; i < per; i++) { uint32_t idx = t * per + i; if (idx < H) a += nnz[idx]; }
    s_part[t] = a;
    __syncthreads();
    if (t == 0) { uint32_t run = 0; for (int i = 0; i < 1024; i++) { uint32_t x = s_part[i]; s_part[i] = run; run += x; } offsets[H] = run; }
    __syncthreads();
    uint32_t run = s_part[t];
    for (uint32_t i = 0; i < per; i++) { uint32_t idx = t * per + i; if (idx < H) { offsets[idx] = run; run += nnz[idx]; } }
}

__global__ void __launch_bounds__(K3_THREADS)
k_export(const unsigned long long *__restrict__ buckets, const uint32_t *__restrict__ flags, uint32_t win,
         const uint32_t *__restrict__ offsets, short *__restrict__ out_keys, unsigned long long *__restrict__ out_counts) {
    __shared__ unsigned int s_warp[32];
    const int h = blockIdx.x, t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const uint32_t level = flags[h];
    if (level == 0) return;
    const unsigned long long *hb = buckets + (size_t)h * 65536u;
    const int key0 = -32768 + warp * K3_WARP_KEYS;
    const bool scans = warp_scans(key0, level, win);
    unsigned int nnz = 0;
    if (scans) {
#pragma unroll 4
        for (int r = 0; r < K3_WARP_KEYS / 32; r++)
            nnz += __popc(__ballot_sync(0xFFFFFFFFu, hb[(unsigned int)(key0 + r * 32 + lane) & 0xFFFFu] != 0));
    }
    if (lane == 0) s_warp[warp] = nnz;     // every lane holds the warp total
    __syncthreads();
    if (warp == 0) {
        unsigned int w = s_warp[lane], wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { unsigned int y = __shfl_up_sync(0xFFFFFFFFu, wi, o); if (lane >= o) wi += y; }
        s_warp[lane] = wi - w;
    }
    __syncthreads();
    if (!nnz) return;
    unsigned int pos = offsets[h] + s_warp[warp];
    for (int r = 0; r < K3_WARP_KEYS / 32; r++) {
        int key = key0 + r * 32 + lane;
        unsigned long long c = hb[(unsigned int)key & 0xFFFFu];
        unsigned int m = __ballot_sync(0xFFFFFFFFu, c != 0);
        if (c) {
            unsigned int p = pos + __popc(m & ((1u << lane) - 1u));
            out_keys[p] = (short)key;
            out_counts[p] = c;
        }
        pos += __popc(m);
    }
}

// Zero what an interval wrote: per touched histogram its window cells (all 65536 when it holds out-of-window
// counts), then its flag.  Replaces a memset of the whole uint64[H][65536] array (512 MiB at H = 1024).
// Window cell i of 2*win-1: i < win -> key i; otherwise key -(i - win + 1), i.e. index 65536 - (i - win + 1).
__device__ __forceinline__ uint32_t window_cell(uint32_t i, uint32_t win) { return i < win ? i : 65536u - (i - win + 1u); }

__global__ void __launch_bounds__(256)
k_clear_touched(unsigned long long *__restrict__ buckets, uint32_t *__restrict__ flags, uint32_t win) {
    const uint32_t h = blockIdx.x;
    const uint32_t level = flags[h];
    if (level == 0) return;
    unsigned long long *hb = buckets + (size_t)h * 65536u;
    if (level & 2u) {
        for (uint32_t i = threadIdx.x; i < 65536u; i += 256) hb[i] = 0ull;
    } else {
        for (uint32_t i = threadIdx.x; i < 2u * win - 1u; i += 256) hb[window_cell(i, win)] = 0ull;
    }
    __syncthreads();
    if (threadIdx.x == 0) flags[h] = 0;
}

// ------------------------------------------------------------------- window
// One folded snapshot as the window keeps it: the k_export lists of its view plus its flags and counter deltas.
struct WinSlotView {
    const uint32_t *offsets;            // [H+1]
    const short *keys;
    const unsigned long long *counts;
    const uint32_t *flags;              // [H]
    const unsigned long long *counters; // [C]
};

// acc += the new slot, acc -= the evicted one (sub.offsets == nullptr: nothing leaves the window).  One CTA per
// histogram; a (histogram, key) pair occurs at most once in a slot, so each pass writes distinct cells and needs no
// atomics, and the barrier between the passes orders the add and the subtract of a key present in both.  levels[h] /
// levels[H+h] count the held intervals that touched h at flag level >= 1 / == 3, so the window's flag is exact when
// an interval drops out.  Counter sums ride along on a grid-stride loop.
constexpr int KW_THREADS = 512;
__global__ void __launch_bounds__(KW_THREADS)
k_window_apply(unsigned long long *__restrict__ acc, uint32_t *__restrict__ acc_flags, uint32_t *__restrict__ levels,
               unsigned long long *__restrict__ acc_counters, uint32_t H, uint32_t C, WinSlotView add, WinSlotView sub) {
    const uint32_t h = blockIdx.x, t = threadIdx.x;
    for (uint32_t i = h * KW_THREADS + t; i < C; i += gridDim.x * KW_THREADS)
        acc_counters[i] += add.counters[i] - (sub.offsets ? sub.counters[i] : 0ull);
    const uint32_t fa = add.flags[h], fs = sub.offsets ? sub.flags[h] : 0u;
    if (!fa && !fs) return;
    unsigned long long *hb = acc + (size_t)h * 65536u;
    for (uint32_t i = add.offsets[h] + t; i < add.offsets[h + 1]; i += KW_THREADS)
        hb[(unsigned short)add.keys[i]] += add.counts[i];
    __syncthreads();
    if (fs)
        for (uint32_t i = sub.offsets[h] + t; i < sub.offsets[h + 1]; i += KW_THREADS)
            hb[(unsigned short)sub.keys[i]] -= sub.counts[i];
    if (t == 0) {
        const uint32_t n1 = levels[h] + (fa != 0u) - (fs != 0u);
        const uint32_t n3 = levels[H + h] + ((fa & 2u) != 0u) - ((fs & 2u) != 0u);
        levels[h] = n1;
        levels[H + h] = n3;
        acc_flags[h] = n3 ? 3u : (n1 ? 1u : 0u);
    }
}

// ---------------------------------------------------------------------- K5
// Multi-GPU snapshot: one small kernel per rank sums, for every histogram some rank touched, the window cells of
// ALL ranks' frozen arrays (peer-mapped device memory: direct NVLink loads, no staging copy, no library
// collective) into this rank's `out` arrays, so every rank ends with the global histogram (the "tiny all-reduce of
// the ~4K-entry bucket arrays").  uint64 sums are associative: bit-identical to a single-GPU run.
// Protocol (comm block = uint64[32] per rank, slot r written only by rank r):
//   arrive[r]  rank r's frozen arrays for snapshot `seq` are complete      (pushed into every peer's block)
//   depart[r]  rank r has finished reading this rank's arrays for `seq`    (pushed when its last CTA is done)
// The kernel ends only after every peer departed, so the caller may clear its frozen arrays right after it.
// token = seq*2 + frozen buffer index: ranks must take their snapshots in lock-step (same count, same order).
static_assert(LH_MAX_RANKS == 16, "comm block layout assumes 16 ranks");
constexpr int K5_THREADS = 1024;
constexpr int K5_CHUNK = 2 * K5_THREADS;     // cells per work item (one-shot form)
constexpr int K5_DEEP = 9;                   // cells per thread and pass of the two-shot form: 9 x 1024 covers the 8 735-cell window of precision 100

struct PeerParams {
    uint32_t rank, world, H, C, win, do_counters, frozen, pad;
    unsigned long long seq;
    unsigned long long timeout_ns;
    const unsigned long long *buckets[LH_MAX_RANKS];     // every rank's FROZEN uint64[H][65536] (own rank: local pointer)
    const uint32_t *flags[LH_MAX_RANKS];
    const unsigned long long *counters[LH_MAX_RANKS];
    unsigned long long *comm[LH_MAX_RANKS];               // every rank's comm block
    unsigned long long *out_buckets;                      // this rank's reduced arrays (zero outside what is written)
    unsigned long long *out_peer[LH_MAX_RANKS];           // every rank's reduced bucket array (own rank: out_buckets)
    uint32_t two_shot;                                    // 1: each rank sums 1/world of the cells and pushes the sums to every rank
    uint32_t arrive_only;                                 // 1: announce + wait for every peer, nothing else (one small CTA ahead of a wide launch)
    uint32_t *out_flags;
    unsigned long long *out_counters;
    unsigned int *block_counter;                          // local, zero between launches
    unsigned int *status;                                 // local: 1 = a peer never arrived, 2 = buffer parity mismatch
    unsigned long long *cells;                            // local: cells summed by this launch (zeroed by the host)
};

__device__ __forceinline__ unsigned long long ld_sys_u64(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
// Bulk reads of a peer's frozen arrays: ordinary L2-only loads (ld.global.cg), which a warp coalesces into 128-byte
// requests - strong system-scope loads went out as one small NVLink request per lane (35 MB took 0.7 - 3 ms).  They are
// ordered after the acquire of the peer's arrival token, and L1 (which could hold the same addresses from two
// snapshots ago) is bypassed; peer memory is not cached in the local L2.
__device__ __forceinline__ unsigned long long ld_peer_u64(const unsigned long long *p) { return __ldcg(p); }
__device__ __forceinline__ uint32_t ld_sys_u32(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long ld_acquire_sys_u64(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys_u64(unsigned long long *p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long global_timer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
// spin until slot >= token (tokens grow with the snapshot sequence); false on timeout
__device__ __forceinline__ bool wait_token(const unsigned long long *slot, unsigned long long token, unsigned long long timeout_ns,
                                           unsigned long long *seen) {
    const unsigned long long t0 = global_timer_ns();
    unsigned int spins = 0;
    for (;;) {
        const unsigned long long v = ld_acquire_sys_u64(slot);
        if ((v >> 1) >= (token >> 1)) { *seen = v; return true; }
        if ((++spins & 1023u) == 0 && global_timer_ns() - t0 > timeout_ns) return false;
    }
}

__global__ void __launch_bounds__(K5_THREADS, 1)
k_peer_allreduce(PeerParams p) {
    extern __shared__ unsigned char s_level[];               // [H]: OR over ranks of the histogram's flag
    __shared__ unsigned long long s_cells;
    const uint32_t t = threadIdx.x;
    const unsigned long long token = p.seq * 2ull + p.frozen;
    unsigned long long *mine = p.comm[p.rank];
    // 1. announce: my frozen arrays were completed by earlier kernels on this stream
    if (blockIdx.x == 0 && t < p.world && t != p.rank) {
        __threadfence_system();
        st_release_sys_u64(p.comm[t] + p.rank, token);
    }
    // 2. wait until every peer announced the same snapshot
    if (t < p.world && t != p.rank) {
        unsigned long long seen = 0;
        if (!wait_token(mine + t, token, p.timeout_ns, &seen)) atomicMax(p.status, 1u);
        else if ((seen >> 1) == p.seq && (seen & 1ull) != p.frozen) atomicMax(p.status, 2u);
    }
    if (p.arrive_only) return;
    if (t == 0) s_cells = 0;
    __syncthreads();
    const bool ok = ld_sys_u32(p.status) == 0;
    // 3. sum.  Work item = (histogram, chunk of K5_CHUNK cells); the set of cells follows the OR of all ranks' flags.
    //    one-shot (small payload): every rank sums every item into its own array - one NVLink round trip.
    //    two-shot (large payload): the rank that owns an item sums it and pushes the sum into every rank's array, so a
    //    rank moves 2 * (world - 1) / world of the payload over NVLink instead of (world - 1) times the payload.
    if (ok) {
        const uint32_t wcells = 2u * p.win - 1u;
        constexpr uint32_t PER_H = 65536u / K5_CHUNK;         // items are indexed as if every histogram were dense
        const uint32_t chunks_w = (wcells + K5_CHUNK - 1) / K5_CHUNK;
        unsigned long long cells = 0;
        for (uint32_t h = t; h < p.H; h += K5_THREADS) {
            uint32_t lv = 0;
            for (uint32_t r = 0; r < p.world; r++) lv |= ld_sys_u32(p.flags[r] + h);
            s_level[h] = (unsigned char)lv;
            if (blockIdx.x == 0 && lv) { p.out_flags[h] = lv; cells += (lv & 2u) ? 65536u : wcells; }
        }
        if (blockIdx.x == 0 && cells) atomicAdd(&s_cells, cells);
        __syncthreads();
        if (blockIdx.x == 0 && t == 0) *p.cells = s_cells;
        if (!p.two_shot) {
            const size_t nitems = (size_t)p.H * PER_H;
            for (size_t item = blockIdx.x; item < nitems; item += gridDim.x) {
                const uint32_t h = (uint32_t)(item / PER_H), chunk = (uint32_t)(item % PER_H);
                const uint32_t level = s_level[h];
                if (level == 0) continue;
                const bool dense = (level & 2u) != 0;
                if (!dense && chunk >= chunks_w) continue;
                const uint32_t ncell = dense ? 65536u : wcells;
                constexpr int K = K5_CHUNK / K5_THREADS;
#pragma unroll
                for (int k = 0; k < K; k++) {
                    const uint32_t i = chunk * K5_CHUNK + k * K5_THREADS + t;
                    if (i >= ncell) continue;
                    const size_t cell = (size_t)h * 65536u + (dense ? i : window_cell(i, p.win));
                    unsigned long long sum = 0;
                    for (uint32_t r = 0; r < p.world; r++) sum += ld_peer_u64(p.buckets[r] + cell);
                    if (sum) p.out_buckets[cell] = sum;
                }
            }
        } else {
            // two-shot: a rank owns the histograms h = rank (mod world); a CTA takes one owned histogram at a time and every
            // thread keeps K5_DEEP cells x world loads in flight (a few CTAs on the SMs the ingest kernel leaves free must
            // cover the NVLink latency-bandwidth product on their own)
            for (uint32_t h = p.rank + blockIdx.x * p.world; h < p.H; h += gridDim.x * p.world) {
                const uint32_t level = s_level[h];
                if (level == 0) continue;
                const bool dense = (level & 2u) != 0;
                const uint32_t ncell = dense ? 65536u : wcells;
                for (uint32_t base = 0; base < ncell; base += K5_DEEP * K5_THREADS) {
                    // all loads of a pass before its first store: K5_DEEP cells x world ranks, independent, as many in flight
                    // per thread as the 64 registers allow (one CTA per SM)
                    uint32_t cell[K5_DEEP];                  // cell index inside the [H][65536] array (H <= 65535: fits 32 bits)
                    unsigned long long sum[K5_DEEP];
#pragma unroll
                    for (int k = 0; k < K5_DEEP; k++) {
                        const uint32_t i = base + k * K5_THREADS + t;
                        cell[k] = i < ncell ? h * 65536u + (dense ? i : window_cell(i, p.win)) : 0xFFFFFFFFu;
                        sum[k] = 0;
                    }
#pragma unroll 4
                    for (uint32_t r = 0; r < p.world; r++) {
                        const unsigned long long *src = p.buckets[r];
#pragma unroll
                        for (int k = 0; k < K5_DEEP; k++)
                            if (cell[k] != 0xFFFFFFFFu) sum[k] += ld_peer_u64(src + cell[k]);
                    }
#pragma unroll
                    for (int k = 0; k < K5_DEEP; k++) {
                        if (cell[k] == 0xFFFFFFFFu || sum[k] == 0) continue;
                        for (uint32_t r = 0; r < p.world; r++) p.out_peer[r][cell[k]] = sum[k];
                    }
                }
            }
        }
        if (p.do_counters && blockIdx.x == 0) {
            for (uint32_t i = t; i < p.C; i += K5_THREADS) {
                unsigned long long sum = 0;
                for (uint32_t r = 0; r < p.world; r++) sum += ld_sys_u64(p.counters[r] + i);
                p.out_counters[i] = sum;
            }
        }
        if (p.two_shot) __threadfence_system();              // my pushes are performed before this CTA checks out
    }
    // 4. depart: the last CTA of this rank tells every peer it has finished reading them and that the sums it pushed
    //    are visible (every CTA fences at system scope before it checks out), then waits for the same from every peer
    __syncthreads();
    __shared__ bool s_last;
    if (t == 0) {
        __threadfence_system();
        s_last = atomicAdd(p.block_counter, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!s_last) return;
    if (t == 0) *p.block_counter = 0;
    if (t < p.world && t != p.rank) {
        __threadfence_system();
        st_release_sys_u64(p.comm[t] + LH_MAX_RANKS + p.rank, token);
        unsigned long long seen = 0;
        if (!wait_token(mine + LH_MAX_RANKS + t, token, p.timeout_ns, &seen)) atomicMax(p.status, 1u);
    }
}

// ----------------------------------------------------------- probes / tables
__global__ void k_fill_decompress(double *__restrict__ table, double precision) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < 65536) table[i] = go_decompress((int)(short)i, precision);
}

__global__ void k_compress_probe(const double *__restrict__ v, size_t n, short *__restrict__ out, int mode, Prec pc) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (short)(mode == 1 ? exact_key16(v[i], pc.precision) : key16_of(v[i], pc));
}

// max | estimate - precision*ln(x) | over samples inside the fast window, for both estimators that ship:
//   [0] fast_candidate()      (k_ingest_keyed*, probes, ragged tails)
//   [2] bucket_offsets_v2()   (packed-FP32 form with the -1023*c2 constant folded into the FMA; K1, keyed_small, keyed_wc)
// plus [1] the tally of samples fast_candidate() sends to the exact path.
__global__ void k_fastpath_margin(const double *__restrict__ v, size_t n, unsigned long long *__restrict__ out, Prec pc) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double x = __dadd_rn(1.0, fabs(v[i]));
    uint32_t hi = (uint32_t)__double2hiint(x), lo = (uint32_t)__double2loint(x);
    uint32_t idx; bool slow;
    fast_candidate(v[i], pc, idx, slow);
    if (slow) atomicAdd(&out[1], 1ull);
    if (hi >= 0x43E00000u) return;
    uint32_t t = __funnelshift_l(lo, hi, 3);
    float m = __uint_as_float((t & 0x007FFFFFu) | 0x3F800000u);
    float lg;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg) : "f"(m));
    uint32_t eb = hi >> 20;
    const double truth = pc.precision * log(x);
    const double base = (double)(int)(eb - 1023u) * (double)pc.a_int;
    {   // estimator 1
        float ef = __fadd_rn(__uint_as_float(0x4B000000u | eb), -(8388608.0f + 1023.0f));
        float w = __fmaf_rn(lg, pc.c1, __fmul_rn(ef, pc.c2));
        atomicMax(&out[0], (unsigned long long)__double_as_longlong(fabs(base + (double)w - truth)));
    }
    {   // estimator 2 (same constants as bucket_offsets_v2)
        float a = __fmaf_rn(__uint2float_rn(eb), pc.c2, pc.kb);
        float w = __fmaf_rn(lg, pc.c1, a);
        atomicMax(&out[2], (unsigned long long)__double_as_longlong(fabs(base + (double)w - truth)));
    }
}

// ---------------------------------------------------------- synthetic streams
__device__ __constant__ unsigned char c_streamL_exp[16] = {17, 18, 18, 19, 19, 19, 20, 20, 20, 20, 21, 21, 21, 22, 22, 23};

__device__ __forceinline__ uint64_t stream_bits(int kind, uint64_t seed, uint64_t i) {
    uint64_t u = splitmix64(seed + i);
    uint64_t mant = u & 0x000FFFFFFFFFFFFFull;
    switch (kind) {
    case 0: return ((uint64_t)(1023 + (u >> 52) % 63) << 52) | mant;
    case 1: return ((uint64_t)(1023 + c_streamL_exp[(u >> 52) & 15]) << 52) | mant;
    case 2: {
        uint32_t sel = (uint32_t)(u >> 52) & 0xFFFu;
        if (sel < 41) return 0x8000000000000000ull | ((uint64_t)(1023 + (u >> 40) % 63) << 52) | mant;
        if (sel < 60) return splitmix64(u);
        if (sel < 80) return ((u >> 11) & 0x8000000000000000ull) | ((uint64_t)(1023 - 10 + (u >> 40) % 12) << 52) | mant;
        if (sel < 90) return ((u >> 13) & 0x8000000000000000ull) | ((uint64_t)(1023 + 63 + (u >> 40) % 961) << 52) | mant;
        return ((uint64_t)(1023 + (u >> 40) % 63) << 52) | mant;
    }
    case 3: return 0x40F86A0000000000ull;
    case 4:
        if (u >> 63) return 0x40F86A0000000000ull;
        return ((uint64_t)(1023 + c_streamL_exp[(u >> 52) & 15]) << 52) | mant;
    case 6: {   // timer durations as int64 nanoseconds: the L stream truncated toward zero
        double d = u64_as_f64(((uint64_t)(1023 + c_streamL_exp[(u >> 52) & 15]) << 52) | mant);
        return (uint64_t)__double2ll_rz(d);
    }
    case 7: return 1 + (u >> 60);   // counter amounts 1..16
    case 8: return ((u >> 11) & 0x8000000000000000ull) | ((uint64_t)(1023 + (u >> 52) % 63) << 52) | mant;   // N: stream U, random sign
    default: return u;
    }
}

__global__ void k_gen_stream(int kind, uint64_t seed, uint64_t start, size_t n, double *__restrict__ out) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
        out[i] = u64_as_f64(stream_bits(kind, seed, start + i));
}

__global__ void k_gen_ids_u16(int kind, uint64_t seed, uint64_t start, size_t n, uint32_t H,
                              unsigned short *__restrict__ out) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        uint64_t u = splitmix64((seed ^ 0xA5A5A5A5DEADBEEFull) + start + i);
        uint32_t a = (uint32_t)((u & 0xFFFFFFFFu) % H), b = (uint32_t)((u >> 32) % H);
        out[i] = (unsigned short)(kind == 0 ? a : (a < b ? a : b));
    }
}

}  // namespace lh
