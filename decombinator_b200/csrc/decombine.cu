// decombine.cu -- the sm_100a kernels of the decombine hot path and the context that drives them.
//
// Two kernels per batch, both one thread per read, 32 reads per warp:
//
//   exact-tag kernel   every read.  128-bit loads of the packed read slot, sampled-seed search for the full V and J
//                      tags, bit-parallel deletion walk, the four dcr() filters, one 16-byte record out.  Reads it
//                      cannot finish (no exact tag, a non-ACGT symbol where the reference looks, a deletion walk that
//                      leaves the interior, `-or both` retries) are appended UNCOUNTED to a queue with one
//                      warp-aggregated atomic (ballot + popc + shuffle).  Three forms, picked per batch:
//                        dcb_exact_kernel_flat   chains with one seed geometry, reads up to 320 nt: 13-mer seeds at
//                                                stride 8, byte filter, hash-and-displace offsets, 8-byte tag slots
//                        dcb_exact_kernel_spec   V (9-mers, stride 12) + J (8-mers, stride 5) bit filters in private
//                                                copies, class-key cuckoo + prefix table (12-nt J tags, long reads)
//                        dcb_exact_kernel        the generic form of the latter (any slot size / geometry)
//   dcb_general_kernel the queued reads only (compacted, so warps stay dense): the complete vanalysis/janalysis
//                      contract incl. the half-tag fallback with Hamming <= 1 and the literal Python-slice deletion
//                      walks; candidate keyword positions marked by a union suffix filter, one hit list per read,
//                      reads regrouped by class between preparation and analysis.
//
// Tag tables are staged into shared memory once per (persistent) block with TMA bulk copies
// (cp.async.bulk + mbarrier); reads live in shared memory as [word][thread] so data-dependent word
// indices are bank-conflict free.
#include "dcb_internal.h"
#include "dcr_core.cuh"

#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstring>
#include <chrono>
#include <mutex>
#include <thread>
#include <vector>

// ------------------------------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------------------------------
struct BatchDev {
    const uint32_t* words;
    const uint16_t* lens;
    const uint32_t* flags;
    const uint32_t* exc_read;
    const uint16_t* exc_pos;
    const uint8_t* exc_kind;
    const uint32_t* exc_index;   // exc_index[k] = first exception entry whose read is >= 32 k (n_exc > 0 only)
    uint32_t n_reads, slot_words, uniform_len, n_exc;
    uint32_t first;   // the launch covers reads [first, first + n_reads); every array is indexed by the global read index
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// Stage `bytes` (multiple of 16, both sides 16-byte aligned) from global into shared memory with the
// TMA bulk-copy engine; completion is signalled on an mbarrier that all threads then wait on.
__device__ __forceinline__ void tma_stage_begin(uint64_t* bar, uint32_t total_bytes) {
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(bar)));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(total_bytes)
                     : "memory");
    }
}
__device__ __forceinline__ void tma_stage_copy(uint64_t* bar, void* dst, const void* src, uint32_t bytes) {
    if (threadIdx.x == 0) {
        const char* s = (const char*)src;
        char* d = (char*)dst;
        while (bytes) {
            uint32_t chunk = bytes > 32768u ? 32768u : bytes;
            asm volatile(
                "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                    smem_u32(d)),
                "l"(s), "r"(chunk), "r"(smem_u32(bar))
                : "memory");
            s += chunk; d += chunk; bytes -= chunk;
        }
    }
}
__device__ __forceinline__ void tma_stage_wait(uint64_t* bar) {
    uint32_t done = 0;
    const uint32_t addr = smem_u32(bar);
    while (!done) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(addr)
            : "memory");
    }
}

__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {
    uint32_t v;
    asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}

// i * (4 * DCB_BLOOM_COPIES) + base as ONE multiply-add (the compiler otherwise rewrites the shift pair into
// shift + mask + add): the byte address of word i of this lane's filter copy
__device__ __forceinline__ uint32_t mad_copy(uint32_t i, uint32_t base) {
    uint32_t v;
    asm("mad.lo.u32 %0, %1, %3, %2;" : "=r"(v) : "r"(i), "r"(base), "n"(4 * DCB_BLOOM_COPIES));
    return v;
}

__device__ __forceinline__ uint4 ldg_stream(const uint4* p) {
    uint4 r;
#ifndef DCB_VAR_LDG
#define DCB_VAR_LDG 1   // measured: L1-allocating loads 4 % faster than no_allocate (the four loads of a slot share two sectors)
#endif
#if DCB_VAR_LDG == 0
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
#elif DCB_VAR_LDG == 1
    asm volatile("ld.global.nc.v4.u32 {%0, %1, %2, %3}, [%4];"
#else
    asm volatile("ld.global.nc.L1::evict_first.v4.u32 {%0, %1, %2, %3}, [%4];"
#endif
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}

__device__ __forceinline__ void store_result(dcb_result* dst, const dcb_result& r) {
    *reinterpret_cast<uint4*>(dst) = *reinterpret_cast<const uint4*>(&r);
}

// first index e in [0, n) with a[e] >= key
__device__ __forceinline__ uint32_t lower_bound_u32(const uint32_t* a, uint32_t n, uint32_t key) {
    uint32_t lo = 0, hi = n;
    while (lo < hi) {
        uint32_t mid = (lo + hi) >> 1;
        if (__ldg(a + mid) < key) lo = mid + 1; else hi = mid;
    }
    return lo;
}

static constexpr int kExactThreads = 512;   // upper bounds; long reads launch narrower blocks (shared memory)
#ifndef DCB_GENERAL_THREADS
#define DCB_GENERAL_THREADS 768
#define DCB_GENERAL_BLOCKS 1
#endif
static constexpr int kGeneralThreads = DCB_GENERAL_THREADS;   // one wide block per SM: the 72 KB of tables are staged once, 24 warps hide the latency
static constexpr int kMaxChunks = 256;             // queue counters per context
// One counter set: two queue counters per chunk, then the reference counters.  A context has two sets (see dcb_run_resident).
static constexpr size_t kCounterSetWords = 2 * kMaxChunks + 2 * DCB_NCOUNTERS;
static constexpr size_t kZeroBlockBytes = 2 * kCounterSetWords * sizeof(uint32_t);
static constexpr uint32_t kChunkReads = 1u << 20;  // reads per chunk of the pipelined host-to-host path

// Shared-memory carve-up common to the kernels: [table 0..3][per-thread columns][counters][mbarrier]
struct Tables4 {
    const uint32_t* g[4];   // global pointers (null = absent)
    int words[4];
};
struct SmemLayout {
    uint32_t* t[4];
    uint32_t* cols;
    dcb_cnt_t* cnt;
    uint64_t* bar;
};
__device__ __forceinline__ SmemLayout carve(uint32_t* smem, const Tables4& tb, size_t col_words) {
    SmemLayout L;
    uint32_t* p = smem;
    for (int i = 0; i < 4; i++) { L.t[i] = tb.words[i] ? p : nullptr; p += tb.words[i]; }
    L.cols = p;
    L.cnt = L.cols + col_words;
    L.bar = reinterpret_cast<uint64_t*>(L.cnt + ((DCB_NCOUNTERS + 3) & ~3));
    return L;
}
// TMA-stage the tables, zero the block counters, wait.
__device__ __forceinline__ void stage_tables(const SmemLayout& L, const Tables4& tb) {
    tma_stage_begin(L.bar, (uint32_t)(tb.words[0] + tb.words[1] + tb.words[2] + tb.words[3]) * 4u);
    for (int i = 0; i < 4; i++)
        if (tb.words[i]) tma_stage_copy(L.bar, L.t[i], tb.g[i], (uint32_t)tb.words[i] * 4u);
    if (threadIdx.x < DCB_NCOUNTERS) L.cnt[threadIdx.x] = 0;
    tma_stage_wait(L.bar);
    __syncthreads();
}

__device__ __forceinline__ void flush_counters(const dcb_cnt_t* s_cnt, unsigned long long* counters) {
    __syncthreads();
    if (threadIdx.x < DCB_NCOUNTERS && s_cnt[threadIdx.x])
        atomicAdd(counters + threadIdx.x, (unsigned long long)s_cnt[threadIdx.x]);
}

// The first entry of read ri (which has some) in the sorted exception list: inside its 32-read group's run.
__device__ __forceinline__ uint32_t exc_first_entry(const BatchDev& b, uint32_t ri) {
    uint32_t e = __ldg(b.exc_index + (ri >> 5));
    while (__ldg(b.exc_read + e) < ri) e++;
    return e;
}

// Programmatic dependent launch (griddepcontrol, sm_90+).  A resident step launches its kernels with the programmatic
// stream serialization attribute, so each one is scheduled while its predecessor finishes: before pdl_wait() a kernel
// touches nothing an earlier kernel writes (shared-memory layout, its own column rows, the constant tag tables); after it,
// everything the earlier kernels wrote is complete and visible.  EVERY block waits before it exits -- an early exit
// included -- so a kernel never completes ahead of its predecessor, and a wait on the step's last kernel covers all of
// them.  Both instructions are no-ops in a kernel launched without the attribute (the chunked paths).
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
// the block's tiles are done: the next kernel of the stream may be scheduled (once every block has said so or exited)
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// Device-side timing of one launch (dcb_timing_*): the earliest block start (stored complemented, so that a zeroed entry
// takes it with atomicMax) and the latest block end, in %globaltimer nanoseconds.  Null: the launch is not timed.
struct TierStamp { unsigned long long nstart, end; };
__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ void stamp_start(TierStamp* ts) {
    if (ts && threadIdx.x == 0) atomicMax(&ts->nstart, ~global_ns());
}
__device__ __forceinline__ void stamp_end(TierStamp* ts) {   // block-uniform: called by every thread of the block
    if (!ts) return;
    __syncthreads();
    if (threadIdx.x == 0) atomicMax(&ts->end, global_ns());
}

// Append the reads of this warp that must go to the general kernel: one atomic per warp.
__device__ __forceinline__ void defer_reads(bool defer, uint32_t ri, uint32_t* queue, uint32_t* queue_count) {
    const unsigned m = __ballot_sync(0xFFFFFFFFu, defer);
    if (m) {
        const int lane = threadIdx.x & 31, leader = __ffs(m) - 1;
        uint32_t base = 0;
        if (lane == leader) base = atomicAdd(queue_count, (uint32_t)__popc(m));
        base = __shfl_sync(0xFFFFFFFFu, base, leader);
        if (defer) queue[base + __popc(m & ((1u << lane) - 1u))] = ri;
    }
}

// ------------------------------------------------------------------------------------------------
// exact-tag kernel, generic form: any slot size / seed geometry (reads are walked from shared memory).
// Tables: 0 = V tag records, 1 = J tag records, 2 = V seed index (or the union index), 3 = J seed index.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kExactThreads)
dcb_exact_kernel(BatchDev b, Tables4 tb, DcrParams prm, int both_frames, dcb_result* __restrict__ results,
                 unsigned long long* __restrict__ counters, uint32_t* __restrict__ queue,
                 uint32_t* __restrict__ queue_count, TierStamp* ts) {
    stamp_start(ts);
    extern __shared__ __align__(16) uint32_t smem[];
    const int T = blockDim.x;
    SmemLayout L = carve(smem, tb, (size_t)b.slot_words * T);
    uint32_t* s_rd = L.cols;  // [slot_words][T]
    stage_tables(L, tb);
    pdl_wait();

    const int tid = threadIdx.x;
    const uint32_t n_tiles = (b.n_reads + T - 1) / T;
    for (uint32_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const uint32_t ri = b.first + tile * T + tid;
        const bool live = tile * T + tid < b.n_reads;
        int action = FAST_DONE;
        dcb_result out;
        *reinterpret_cast<uint4*>(&out) = make_uint4(0, 0, 0, 0);
        if (live) {
            const uint4* src = reinterpret_cast<const uint4*>(b.words + (size_t)ri * b.slot_words);
            for (uint32_t k = 0; k < b.slot_words / 4; k++) {
                uint4 v = ldg_stream(src + k);
                s_rd[(4 * k + 0) * T + tid] = v.x;
                s_rd[(4 * k + 1) * T + tid] = v.y;
                s_rd[(4 * k + 2) * T + tid] = v.z;
                s_rd[(4 * k + 3) * T + tid] = v.w;
            }
            const bool flagged = b.n_exc && ((__ldg(b.flags + (ri >> 5)) >> (ri & 31)) & 1u);
            ReadView r;
            r.w = s_rd + tid; r.inv = nullptr; r.stride = T;
            r.n = b.uniform_len ? (int)b.uniform_len : (int)__ldg(b.lens + ri);
            r.nw = (int)b.slot_words;
            r.exc_pos = nullptr; r.exc_kind = nullptr; r.e0 = r.e1 = 0; r.mirror = 0; r.cand = nullptr; r.cand_kq = 0; r.hits = nullptr; r.n_hits = 0;
            uint32_t hand[2];
            action = dcr_exact_read(r, flagged, L.t[0], L.t[1], L.t[2], L.t[3], prm, both_frames, out, L.cnt, false, nullptr, hand);
            if (action == FAST_DEFER)   // for dcb_halftag_kernel
                *reinterpret_cast<uint4*>(results + ri) = make_uint4(hand[0], hand[1], flagged ? exc_first_entry(b, ri) : 0u, 0u);
        }
        defer_reads(live && action == FAST_DEFER, ri, queue, queue_count);
        if (live && action == FAST_DONE) store_result(results + ri, out);
    }
    pdl_launch_dependents();
    flush_counters(L.cnt, counters);
    stamp_end(ts);
}

// ------------------------------------------------------------------------------------------------
// exact-tag kernel, specialised: the read slot (NW words) sits in registers, every sampled seed position is a
// compile-time constant (static funnel shifts, no index arithmetic), and the lanes probe DCB_BLOOM_COPIES private
// copies of the seed filter, interleaved word by word in shared memory (copy c only ever touches banks c, c + 8,
// c + 16, c + 24), so a probe costs one or two shared-memory wavefronts whatever the 32 q-mers are.  (32 copies of a
// 4x smaller filter were conflict-free but let 0.5 false hits per read through to the verification loop.)
//   NW            words per read slot (16 => reads up to 256 nt)
//   QV, SV, WBV   V seed length / stride / log2(filter words);  QJ, SJ, WBJ the same for J
//   UNION         V and J share the seed geometry and are found together through ONE index (table 2)
// One block of up to 1024 threads per SM (the private filters take 128 KB).
// ------------------------------------------------------------------------------------------------
template <int NW, int Q, int S, int WB>
struct SeedScan {
    static constexpr int NPOS = (16 * NW - Q) / S + 1;
    static constexpr int G0 = NPOS < 32 ? NPOS : 32;   // probes collected in the first / second hit word
    static constexpr int G1 = NPOS - G0;
    static constexpr int WLEAD = DCB_IDX_WLEAD(S + Q - 1, Q);
    static constexpr int WMAX = ((NPOS - 1) * S - WLEAD) >> 4;   // first word of the last verification window
    static_assert(NPOS <= 64, "at most 64 sampled positions");
    // Probe the filter at every sampled position.  Probe i of a group of G lands in bit G-1-i of its hit word
    // (each probe shifts the word left by one), so the EARLIEST position is the HIGHEST set bit.
    // bl = shared-space byte address of this lane's copy of the filter: word w at bl + 4 * DCB_BLOOM_COPIES * w.
    static __device__ __forceinline__ void run(const uint32_t (&w)[NW], uint32_t bl, uint32_t& h0, uint32_t& h1) {
        h0 = 0; h1 = 0;
        constexpr uint32_t BMUL = DCB_BLOOM_MUL(Q);
#pragma unroll
        for (int i = 0; i < NPOS; i++) {
            const int p = i * S, a = p >> 4, sh = (p & 15) * 2;
            uint32_t win;   // at least the 2Q key bits of the q-mer at p (higher bits are don't-care)
            if (sh == 0) win = w[a];
            else if (sh + 2 * Q <= 32 || a + 1 >= NW) win = w[a] >> sh;
            else win = __funnelshift_r(w[a], w[a + 1], sh);
            const uint32_t word = lds_u32(mad_copy((win * BMUL) >> (32 - WB), bl));
            const uint32_t top = __funnelshift_l(0u, word, win);          // word << (key & 31): the key's bit -> bit 31
            if (i < 32) h0 = __funnelshift_l(top, h0, 1); else h1 = __funnelshift_l(top, h1, 1);
        }
    }
    // keep the probes whose q-mer lies inside a read of n bases
    static __device__ __forceinline__ void clip(int n, uint32_t& h0, uint32_t& h1) {
        const int nvalid = n >= Q ? (n - Q) / S + 1 : 0;
        if (nvalid < G0) { h0 &= ~((1u << (G0 - nvalid)) - 1u); h1 = 0; }
        else if (G1 > 0 && nvalid - G0 < G1) h1 &= ~((1u << (G1 - (nvalid - G0))) - 1u);
    }
    // earliest remaining probe index (and remove it); call only while (h0 | h1) != 0
    static __device__ __forceinline__ int pop(uint32_t& h0, uint32_t& h1) {
        if (G1 == 0 || h0) { const int b = 31 - __clz(h0); h0 &= ~(1u << b); return G0 - 1 - b; }
        const int b = 31 - __clz(h1); h1 &= ~(1u << b); return G0 + G1 - 1 - b;
    }
    // the 32 bases starting at p - WLEAD, from a column that has a zero row in front and behind
    static __device__ __forceinline__ void window(const uint32_t* col, int T, int p, uint32_t& lo, uint32_t& hi) {
        const int W = p - WLEAD, sh = (W & 15) * 2;
        const uint32_t* c0 = col + (W >> 4) * T;
        const uint32_t a = c0[0], b = c0[T], c = c0[2 * T];
        lo = __funnelshift_r(a, b, sh);
        hi = __funnelshift_r(b, c, sh);
    }
};

// Confirm the filter hits of all 32 reads of a warp.  ONE flat loop over (hit, candidate offset) pairs: on each trip a
// lane either pops its next hit and looks the q-mer up, or -- when that q-mer stands for several tag offsets -- takes
// the next offset, and then checks one candidate.  The warp votes on every trip, so all lanes stay in the same
// instruction stream and the trip count is the LARGEST number of candidates any one read has (not the sum over
// nested per-lane loops).  Must be called by all 32 lanes; `stop` is the hit counter that ends a lane's scan at 2.
template <class Scan, int S>
__device__ __forceinline__ void verify_hits(const ReadView& r, const SeedIdxView& ix, const uint32_t* col, int T, uint32_t lo,
                                            uint32_t hi, FullHit& vh, FullHit& jh, const FullHit& stop) {
    uint32_t offs = 0, wlo = 0, whi = 0;
    int p = 0;
    for (;;) {
        const bool need = offs == 0 && (lo | hi) != 0 && stop.count < 2;
        if (!__any_sync(0xFFFFFFFFu, need || offs != 0)) break;
        if (need) {
            p = Scan::pop(lo, hi) * S;
            Scan::window(col, T, p, wlo, whi);
            offs = fast_class_lookup(ix, wlo, whi);
        }
        __syncwarp();
        if (offs) {
            const int o = 31 - __clz(offs);
            offs ^= 1u << o;
            fast_check_offset(r, ix, p, o, wlo, whi, vh, jh);
        }
        __syncwarp();
    }
}

// What the specialised kernel needs beyond Tables4: the compact filters to replicate.
struct SpecBlooms { const uint32_t* v; const uint32_t* j; };

template <int A, int B> struct StaticMax { static constexpr int value = A > B ? A : B; };

template <int NW, int QV, int SV, int WBV, int QJ, int SJ, int WBJ, bool UNION>
__global__ void __launch_bounds__(1024, 1)
dcb_exact_kernel_spec(BatchDev b, Tables4 tb, SpecBlooms bl, DcrParams prm, int both_frames, dcb_result* __restrict__ results,
                      unsigned long long* __restrict__ counters, uint32_t* __restrict__ queue,
                      uint32_t* __restrict__ queue_count, TierStamp* ts) {
    stamp_start(ts);
    static_assert(!UNION || (QV == QJ && SV == SJ && WBV == WBJ), "union scan needs one seed geometry");
    using ScanV = SeedScan<NW, QV, SV, WBV>;
    using ScanJ = SeedScan<NW, QJ, SJ, WBJ>;
    constexpr int WMAX = UNION ? ScanV::WMAX : StaticMax<ScanV::WMAX, ScanJ::WMAX>::value;
    constexpr int TRAIL = WMAX + 3 - NW > 0 ? WMAX + 3 - NW : 0;   // zero rows behind the read columns
    constexpr int ROWS = 1 + NW + TRAIL;
    extern __shared__ __align__(16) uint32_t smem[];
    const int T = blockDim.x;
    const int tid = threadIdx.x;
    constexpr int BV = DCB_BLOOM_COPIES << WBV, BJ = UNION ? 0 : (DCB_BLOOM_COPIES << WBJ);
    SmemLayout L = carve(smem, tb, (size_t)BV + BJ + (size_t)ROWS * T);
    uint32_t* s_bv = L.cols;
    uint32_t* s_bj = s_bv + BV;
    uint32_t* s_rd = s_bj + BJ;
    for (int i = tid; i < BV; i += T) s_bv[i] = __ldg(bl.v + i / DCB_BLOOM_COPIES);
    for (int i = tid; i < BJ; i += T) s_bj[i] = __ldg(bl.j + i / DCB_BLOOM_COPIES);
    s_rd[tid] = 0u;
    for (int k = 0; k < TRAIL; k++) s_rd[(1 + NW + k) * T + tid] = 0u;
    stage_tables(L, tb);
    pdl_wait();

    const DcbTag* vtags = gene_tags(smem);                       // table 0 starts the dynamic shared memory
    const DcbTag* jtags = gene_tags(smem + tb.words[0]);
    // index views with the geometry pinned to the template constants (lmin = S + Q - 1 for the shipped sets)
    SeedIdxView vix = seed_idx_view(smem + tb.words[0] + tb.words[1]);   // tables are laid out back to back
    vix.q = QV; vix.stride = SV; vix.wlead = ScanV::WLEAD; vix.lmin = SV + QV - 1;
    vix.span = DCB_IDX_SPAN(SV + QV - 1, QV); vix.k = DCB_IDX_K(SV + QV - 1, QV);
    SeedIdxView jix = seed_idx_view(smem + tb.words[0] + tb.words[1] + (UNION ? 0 : tb.words[2]));
    jix.q = QJ; jix.stride = SJ; jix.wlead = ScanJ::WLEAD; jix.lmin = SJ + QJ - 1;
    jix.span = DCB_IDX_SPAN(SJ + QJ - 1, QJ); jix.k = DCB_IDX_K(SJ + QJ - 1, QJ);
    const uint32_t* col = s_rd + T + tid;                 // word k of this thread's read at col[k * T]
    const uint32_t my_bv = smem_u32(s_bv + (tid % DCB_BLOOM_COPIES));
    const uint32_t my_bj = smem_u32(s_bj + (tid % DCB_BLOOM_COPIES));
    const uint32_t n_tiles = (b.n_reads + T - 1) / T;

    for (uint32_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const uint32_t ri = b.first + tile * T + tid;
        const bool live = tile * T + tid < b.n_reads;
        int action = FAST_DONE;
        dcb_result out;
        *reinterpret_cast<uint4*>(&out) = make_uint4(0, 0, 0, 0);
        // Every lane of the warp walks the same instruction stream below (dead and flagged lanes with empty hit
        // masks), so that the verification loop can re-converge the warp with a vote on every trip.
        uint32_t w[NW];
        {
            const uint4* src = reinterpret_cast<const uint4*>(b.words + (size_t)(live ? ri : 0) * NW);
#pragma unroll
            for (int k = 0; k < NW / 4; k++) {
                const uint4 v = ldg_stream(src + k);
                w[4 * k + 0] = v.x; w[4 * k + 1] = v.y; w[4 * k + 2] = v.z; w[4 * k + 3] = v.w;
            }
#pragma unroll
            for (int k = 0; k < NW; k++) s_rd[(1 + k) * T + tid] = w[k];
        }
        const bool flagged = live && b.n_exc && ((__ldg(b.flags + (ri >> 5)) >> (ri & 31)) & 1u);
        const bool scan = live && !flagged;
        ReadView r;
        r.w = col; r.inv = nullptr; r.stride = T;
        r.n = b.uniform_len ? (int)b.uniform_len : (live ? (int)__ldg(b.lens + ri) : 0);
        r.nw = NW;
        r.exc_pos = nullptr; r.exc_kind = nullptr; r.e0 = r.e1 = 0; r.mirror = 0; r.cand = nullptr; r.cand_kq = 0; r.hits = nullptr; r.n_hits = 0;
        FullHit vh, jh;
        vh.count = 0; vh.code = 0;
        jh.count = 0; jh.code = 0;
        uint32_t lo, hi;
        ScanV::run(w, my_bv, lo, hi);
        ScanV::clip(r.n, lo, hi);
        if (!scan) { lo = 0; hi = 0; }
        verify_hits<ScanV, SV>(r, vix, col, T, lo, hi, vh, jh, vh);
        if (!UNION) {
            ScanJ::run(w, my_bj, lo, hi);
            ScanJ::clip(r.n, lo, hi);
            if (!scan || vh.count != 1) { lo = 0; hi = 0; }
            verify_hits<ScanJ, SJ>(r, jix, col, T, lo, hi, vh, jh, jh);
        }
        if (scan) action = dcr_fast_from_hits<true>(r, vtags, jtags, vh, jh, prm, both_frames, out, L.cnt);
        else if (live) action = FAST_DEFER;
        defer_reads(live && action == FAST_DEFER, ri, queue, queue_count);
        if (live && action == FAST_DONE) store_result(results + ri, out);
        else if (live) {
            // hand-over to dcb_halftag_kernel: what the search found; J was only searched for reads with one full V tag
            const uint32_t hj = (!UNION && vh.count != 1) ? DCB_HIT_UNKNOWN : half_word_of(jh);
            // (a read with non-ACGT symbols is not searched here: both genes "unknown", the half-tag kernel searches them itself)
            *reinterpret_cast<uint4*>(results + ri) = scan ? make_uint4(half_word_of(vh), hj, 0u, 0u)
                                                           : make_uint4(DCB_HIT_UNKNOWN, DCB_HIT_UNKNOWN, flagged ? exc_first_entry(b, ri) : 0u, 0u);
        }
    }
    pdl_launch_dependents();
    flush_counters(L.cnt, counters);
    stamp_end(ts);
}

// ------------------------------------------------------------------------------------------------
// exact-tag kernel, flat form (chains whose V and J tags share one seed geometry: every `extended` set).
// Same contract as dcb_exact_kernel_spec -- the read slot in registers, compile-time seed positions, the same finish --
// with a leaner search:
//   1. probe: ONE byte filter (64 KB, one byte per slot) over 13-mers sampled at every 8th base.  A probe is (SHF for
//      the odd positions; the even ones are word-aligned), IMAD (hash), SHF (slot), LDS.U8 and an IMAD that appends the
//      byte to the hit mask: no bit extraction, half the instructions on the FMA pipe.
//   2. confirm: one warp-voted loop; a trip pops a hit (window of 32 bases from shared memory, 13-mer -> offset set by
//      hash-and-displace: two 16-bit reads) and checks ONE offset (perfect-hash prefix table -> whole-tag compare).
//      13-mers are specific enough that the offset set is almost always one offset of one tag, so the trip count of a
//      warp is close to its largest per-read hit count.  A read that already has two distinct V tags is final
//      (multiple_v_matches) and drops its remaining hits.
// No block-wide barrier inside the tile loop: a lane only ever reads the read column it wrote itself.
// ------------------------------------------------------------------------------------------------
struct QTables {
    const uint32_t* vcore; const uint32_t* jcore; const uint32_t* head; const uint32_t* qtab; const uint32_t* bfilter;
    int vcore_words, jcore_words, head_words, qtab_words;
};

__device__ __forceinline__ uint32_t lds_u8(uint32_t addr) {
    uint32_t v;
    asm("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
template <int OFF>
__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {
    uint32_t v;
    asm("ld.shared.u32 %0, [%1+%2];" : "=r"(v) : "r"(addr), "n"(OFF));
    return v;
}
__device__ __forceinline__ uint32_t mad2(uint32_t h, uint32_t bit) {   // 2 * h + bit on the FMA pipe
    uint32_t v;
    asm("mad.lo.u32 %0, %1, 2, %2;" : "=r"(v) : "r"(h), "r"(bit));
    return v;
}

#define WLEAD_OF(S) ((S) - 1)
template <int NW, int Q, int S, int T, bool EXC>
__global__ void __launch_bounds__(T, 1)
dcb_exact_kernel_flat(BatchDev b, QTables qt, DcrParams prm, int both_frames, dcb_result* __restrict__ results,
                      unsigned long long* __restrict__ counters, uint32_t* __restrict__ queue,
                      uint32_t* __restrict__ queue_count, TierStamp* ts) {
    stamp_start(ts);
    static_assert(S == 8, "seeds start at half-word boundaries");
    constexpr int NPOS = (16 * NW - Q) / S + 1;
    constexpr int NA = NPOS < 32 ? NPOS : 32, NB = NPOS - NA;        // probes in the first / second hit word
    static_assert(NB <= 32, "two hit words");
    static_assert(S + Q - 1 <= 32 - WLEAD_OF(S), "the lmin-prefix at every candidate offset lies inside the window");
    constexpr int WLEAD = S - 1;                                     // the verification window starts at the earliest possible tag start
    constexpr int WMAX = ((NPOS - 1) * S - WLEAD) >> 4;
    constexpr int TRAIL = WMAX + 3 - NW > 1 ? WMAX + 3 - NW : 1;    // zero rows behind the read columns
    constexpr int ROWS = 1 + NW + TRAIL;
    constexpr int FBYTES = 1 << DCB_FBITS;
    constexpr uint32_t FMUL = DCB_BLOOM_MUL(Q);
    extern __shared__ __align__(16) uint32_t smem[];
    const int tid = threadIdx.x;
    // layout: [byte filter][read columns][V tags][J tags][index head][offset table + tag slots][counters][mbarrier]
    // (kept as small as it is: shared memory is carved out of the L1, and a 204 KB layout measured 20 % slower in the
    // phases that touch global memory than this 160 KB one)
    uint32_t* s_filt = smem;
    uint32_t* s_rd = s_filt + FBYTES / 4;
    uint32_t* s_vcore = s_rd + ROWS * T;
    uint32_t* s_jcore = s_vcore + qt.vcore_words;
    uint32_t* s_head = s_jcore + qt.jcore_words;
    uint32_t* s_qtab = s_head + qt.head_words;
    dcb_cnt_t* s_cnt = s_qtab + qt.qtab_words;
    uint64_t* bar = reinterpret_cast<uint64_t*>(s_cnt + ((DCB_NCOUNTERS + 3) & ~3));
    uint32_t* s_x = reinterpret_cast<uint32_t*>(bar + 2);            // [T] EXC only: where each read's exception entries sit in its warp's run

    s_rd[tid] = 0u;
    for (int k = 0; k < TRAIL; k++) s_rd[(1 + NW + k) * T + tid] = 0u;
    tma_stage_begin(bar, (uint32_t)(FBYTES + 4 * (qt.vcore_words + qt.jcore_words + qt.head_words + qt.qtab_words)));
    tma_stage_copy(bar, s_filt, qt.bfilter, FBYTES);
    tma_stage_copy(bar, s_vcore, qt.vcore, 4u * qt.vcore_words);
    tma_stage_copy(bar, s_jcore, qt.jcore, 4u * qt.jcore_words);
    tma_stage_copy(bar, s_head, qt.head, 4u * qt.head_words);
    tma_stage_copy(bar, s_qtab, qt.qtab, 4u * qt.qtab_words);
    if (tid < DCB_NCOUNTERS) s_cnt[tid] = 0;
    tma_stage_wait(bar);
    __syncthreads();
    pdl_wait();

    const DcbTag* vtags = gene_tags(s_vcore);
    const DcbTag* jtags = gene_tags(s_jcore);
    QIdxView ix = q_idx_view(s_head, s_qtab);
    ix.q = Q; ix.stride = S; ix.wlead = WLEAD; ix.lmin = S + Q - 1;       // geometry pinned to the template constants
    const uint32_t* col = s_rd + T + tid;                 // word k of this thread's read at col[k * T]
    const uint32_t col_addr = smem_u32(col);
    const uint32_t filt = smem_u32(s_filt);
    const uint32_t n_tiles = (b.n_reads + T - 1) / T;

    for (uint32_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const uint32_t ri = b.first + tile * T + tid;
        const bool live = tile * T + tid < b.n_reads;
        int action = FAST_DONE;
        dcb_result out;
        *reinterpret_cast<uint4*>(&out) = make_uint4(0, 0, 0, 0);
        uint32_t w[NW];
        {
            const uint4* src = reinterpret_cast<const uint4*>(b.words + (size_t)(live ? ri : 0) * NW);
#pragma unroll
            for (int k = 0; k < NW / 4; k++) {
                const uint4 v = ldg_stream(src + k);
                w[4 * k + 0] = v.x; w[4 * k + 1] = v.y; w[4 * k + 2] = v.z; w[4 * k + 3] = v.w;
            }
#pragma unroll
            for (int k = 0; k < NW; k++) s_rd[(1 + k) * T + tid] = w[k];
        }
        // EXC: the batch has reads with non-ACGT symbols (its own instantiation, so that the clean path carries none of it)
        const bool flagged = live && b.n_exc && ((__ldg(b.flags + (ri >> 5)) >> (ri & 31)) & 1u);
        ExcProbe xp = exc_probe_none();
        if (EXC) {
            // The warp's 32 reads are 32 consecutive read indices (b.first and T are multiples of 32): their non-ACGT symbols
            // are ONE run of the sorted exception list.  Lane k fetches entry k of the run; every read's entries (a short
            // sub-run) then come to its lane by shuffle -- no per-read scans of the list in global memory.
            const int lane = tid & 31;
            const uint32_t g = ri >> 5;
            const bool wlive = tile * T + (tid & ~31) < b.n_reads;          // the warp has a live lane: g is a group of the batch
            const uint32_t eb = wlive ? __ldg(b.exc_index + g) : 0u, ee = wlive ? __ldg(b.exc_index + g + 1) : 0u;
            const uint32_t k = eb + lane;
            const bool have = k < ee;
            const uint32_t rd = have ? __ldg(b.exc_read + k) : 0u;
            const uint32_t ps = have ? (uint32_t)__ldg(b.exc_pos + k) : 0u, kd = have ? (uint32_t)__ldg(b.exc_kind + k) : 3u;
            const uint32_t same = __match_any_sync(0xFFFFFFFFu, have ? (rd & 31u) : 32u + lane);   // the lanes holding one read's entries
            s_x[tid] = 0u;
            __syncwarp();
            if (have && lane == __ffs(same) - 1) s_x[(tid & ~31) + (rd & 31u)] = (uint32_t)lane | ((uint32_t)__popc(same) << 8);
            __syncwarp();
            const uint32_t info = s_x[tid];
            const int first = (int)(info & 255u), cnt = (int)(info >> 8);
            int nx = 0;
#pragma unroll
            for (int s2 = 0; s2 < 4; s2++) {
                const uint32_t p2 = __shfl_sync(0xFFFFFFFFu, ps, (first + s2) & 31), k2 = __shfl_sync(0xFFFFFFFFu, kd, (first + s2) & 31);
                if (s2 < cnt && k2 != 3u) { exc_probe_add(xp, nx, p2); nx++; }
            }
            xp.e0 = eb + (uint32_t)first;
            // more than four symbols, or a run that does not fit in the 32 entries fetched: not searched here
            xp.over = flagged && (cnt > 4 || cnt == 0 || (ee - eb > 32u && first + cnt >= 32));
        }
        const bool scan = EXC ? (live && !xp.over) : (live && !flagged);   // EXC: reads with non-ACGT symbols too, see ExcProbe
        ReadView r;
        r.w = col; r.inv = nullptr; r.stride = T;
        r.n = b.uniform_len ? (int)b.uniform_len : (live ? (int)__ldg(b.lens + ri) : 0);
        r.nw = NW;
        r.exc_pos = nullptr; r.exc_kind = nullptr; r.e0 = r.e1 = 0; r.mirror = 0; r.cand = nullptr; r.cand_kq = 0; r.hits = nullptr; r.n_hits = 0;

        // 1. probe: bit NPOS-1-i of h <=> the seed at i * S may be indexed.  The slot must hash the WHOLE seed: reads are
        //    full of 8-mers that homologous genes share with a tag (measured: slot = the seed's first 8 bases costs 0.8
        //    trips more than it saves in probe instructions).  Even probes are word-aligned (no extraction).
        //    Probe i < NA is bit NA-1-i of h, probe i >= NA (reads longer than 256 nt) bit NPOS-1-i of hb.
        uint32_t h = 0, hb = 0;
#pragma unroll
        for (int i = 0; i < NPOS; i++) {
            const uint32_t win = (i & 1) ? __funnelshift_r(w[i >> 1], (i >> 1) + 1 < NW ? w[(i >> 1) + 1] : 0u, 16) : w[i >> 1];
            const uint32_t byte = lds_u8(filt + ((win * FMUL) >> (32 - DCB_FBITS)));
            if (i < NA) h = mad2(h, byte);
            else hb = mad2(hb, byte);
        }
        {
            const int nvalid = r.n >= Q ? (r.n - Q) / S + 1 : 0;     // probes whose seed lies inside the read
            if (nvalid < NA) h &= ~((1u << (NA - nvalid)) - 1u);
            if (NB > 0) {
                const int nvb = nvalid > NA ? nvalid - NA : 0;
                if (nvb < NB) hb &= ~((1u << (NB - nvb)) - 1u);
            }
            if (!scan) { h = 0; hb = 0; }
        }
        // this lane's column is read back below by this lane only: program order suffices, no barrier
#ifndef DCB_VAR_PREFETCH
#define DCB_VAR_PREFETCH 2   // measured: +1 % (L1 or L2 alike)
#endif
#if DCB_VAR_PREFETCH
        {   // the next tile's slot of this lane: in flight while this tile is confirmed and finished
            const uint32_t nt = tile + gridDim.x;
            if (nt < n_tiles) {
                const uint32_t* nx = b.words + (size_t)min(b.first + nt * T + tid, b.first + b.n_reads - 1) * NW;
#if DCB_VAR_PREFETCH == 1
                asm volatile("prefetch.global.L1 [%0];" ::"l"(nx));
                if (NW > 32) asm volatile("prefetch.global.L1 [%0];" ::"l"(nx + 32));
#else
                asm volatile("prefetch.global.L2 [%0];" ::"l"(nx));
#endif
            }
        }
#endif

        // 2. confirm, one (hit, offset) candidate per trip
        HitWordsX hwx;                                               // EXC: occurrences over a non-ACGT symbol are dropped
        HitWords& hw = hwx.hw;
        hw.v = 0; hw.j = 0; hw.n_v = ix.n_v;
        hwx.xp = (EXC && flagged) ? &xp : nullptr; hwx.utag = ix.utag;
        uint32_t offs = 0, wlo = 0, whi = 0;
        int p = 0;
        for (;;) {
            const bool need = offs == 0u && (h | hb) != 0u;
            if (!__any_sync(0xFFFFFFFFu, need || offs != 0u)) break;
            if (need) {
                int i;                                               // the probe popped: lowest position first
                if (NB == 0 || h) { const int bit = 31 - __clz(h); h ^= 1u << bit; i = NA - 1 - bit; }
                else { const int bit = 31 - __clz(hb); hb ^= 1u << bit; i = NPOS - 1 - bit; }
                // bit position of the window start i * S - WLEAD; its word row is (i - 1) >> 1
                const int wb = 2 * (S * i - WLEAD);
                p = S * i;
                const uint32_t a0 = col_addr - (T * 4) + (uint32_t)(((i + 1) >> 1) * (T * 4));
                const uint32_t x = lds_u32<0>(a0), y = lds_u32<T * 4>(a0), zz = lds_u32<2 * T * 4>(a0);
                wlo = __funnelshift_r(x, y, wb);                     // the shift wraps modulo 32
                whi = __funnelshift_r(y, zz, wb);
                offs = q_offsets(ix, __funnelshift_r(wlo, whi, 2 * WLEAD));
            }
            if (offs) {
                const int o = 31 - __clz(offs);
                offs ^= 1u << o;
                if (EXC) q_check_offset<true>(r, ix, p, o, wlo, whi, hwx);
                else q_check_offset<true>(r, ix, p, o, wlo, whi, hw);
                if (hw.v == DCB_HIT_MULTI) { h = 0u; hb = 0u; offs = 0u; }   // final whatever else is found (decombine.py:278-280)
            }
        }
        if (EXC) hwx.finish();
        FullHit vh, jh;
        hw.decode(vh, jh);
        if (EXC) {
            if (scan) action = dcr_fast_from_hits<true>(r, vtags, jtags, vh, jh, prm, both_frames, out, s_cnt, flagged, xp);
            else if (live) action = FAST_DEFER;
        } else {
            if (scan) action = dcr_fast_from_hits<true>(r, vtags, jtags, vh, jh, prm, both_frames, out, s_cnt);
            else if (live) action = FAST_DEFER;
        }
        defer_reads(live && action == FAST_DEFER, ri, queue, queue_count);
        if (live && action == FAST_DONE) store_result(results + ri, out);
        else if (live) {
            // hand-over to dcb_halftag_kernel in the read's (still unused) result slot: what the search found, one word
            // per gene with the tag numbered inside its gene; "several" for a read that was not searched
            const bool one_j = hw.j != 0u && hw.j != DCB_HIT_MULTI;
            const uint4 hand = make_uint4(scan ? hw.v : DCB_HIT_MULTI, scan ? (one_j ? hw.j - ((uint32_t)ix.n_v << 16) : hw.j) : DCB_HIT_MULTI,
                                          xp.e0, 0u);
            *reinterpret_cast<uint4*>(results + ri) = hand;
        }
    }
    pdl_launch_dependents();
    flush_counters(s_cnt, counters);
    stamp_end(ts);
}

// ------------------------------------------------------------------------------------------------
// half-tag kernel: the reads the flat exact-tag kernel queued (compacted, so warps are dense), one thread per read.
// Almost all of them lack ONE full tag because of a substitution or an N in it.  The flat kernel left what it found in
// the read's result slot; here the half keywords of the missing gene(s) are found through the sampled half-tag index
// (DcbHalfIndex: a direct-indexed 16-bit entry per 7-mer, probed at every 4th base from registers), every occurrence
// is confirmed in one warp-voted loop and expanded into (tag, start) candidates kept in the reference's order, and the
// candidates are tried in turn: Hamming <= 1, counter, bit-parallel deletion walk, the four filters (dcr_core.cuh,
// "Half-tag path").  Counters stay pending in a register until the read is decided; a read outside the interior case
// (several full-tag candidates in a read with non-ACGT symbols, a tag window or a deletion walk that leaves the read or
// the 32-base window, more than DCB_HALF_CAP candidates) goes on to the general kernel through a second queue, uncounted.
// Tables: 0 = V tag records, 1 = J tag records, 2 = half-tag index.
// ------------------------------------------------------------------------------------------------
// The three capacities can be set at compile time (-D...): the test suite builds variants with tiny lists, in which nearly
// every warp overflows every list, to run the pass-on branches on ordinary data (build.py variant, VARIANTS).
#ifndef DCB_HALF_CAP
#define DCB_HALF_CAP 12         // candidates of one read
#endif
#ifndef DCB_HALF_WCAP
#define DCB_HALF_WCAP 192       // probe hits of one warp's 32 reads that are confirmed here; reads beyond pass on
#endif
#ifndef DCB_HALF_WCAP2
#define DCB_HALF_WCAP2 126      // prefix hits, and (occurrence, tag) pairs, of one warp's 32 reads
#endif
static_assert(DCB_HALF_WCAP % 2 == 0, "s_work holds 16-bit entries and is carved in 32-bit words");
static_assert(DCB_HALF_WCAP2 >= 3, "a J-scan round takes reads until WCAP2 / 3 prefix hits");
static_assert(DCB_HALF_CAP >= 1 && DCB_HALF_CAP <= 4095, "the candidate count of DCB_HALF_COUNT has 12 bits");
template <int NW, int T>
__global__ void __launch_bounds__(T, 1)
dcb_halftag_kernel(BatchDev b, Tables4 tb, DcrParams prm, dcb_result* __restrict__ results,
                   unsigned long long* __restrict__ counters, const uint32_t* __restrict__ queue,
                   const uint32_t* __restrict__ queue_count, uint32_t* __restrict__ queue2, uint32_t* __restrict__ queue2_count,
                   TierStamp* ts) {
    constexpr int ROWS = NW + 3;                                    // a zero row in front of the read's words, two behind
    constexpr int NPOS = (16 * NW - DCB_HALF_Q) / DCB_HALF_STRIDE + 1;
    constexpr int NM = (NPOS + 31) / 32;                            // probe-hit mask words
    static_assert(NM <= 3 && NPOS <= 255, "three mask words, probe index in 8 bits");
    stamp_start(ts);
    pdl_wait();
    const uint32_t n_items = *queue_count;
    const uint32_t n_tiles = (n_items + T - 1) / T;
    if (blockIdx.x >= n_tiles) { stamp_end(ts); return; }          // nothing queued for this block: do not even stage the tables
    extern __shared__ __align__(16) uint32_t smem[];
    const int tid = threadIdx.x, lane = tid & 31, wbase = tid - lane;
    SmemLayout L = carve(smem, tb, (size_t)(2 * ROWS + DCB_HALF_CAP + 1) * T + (size_t)(T / 32) * (DCB_HALF_WCAP / 2 + 2 * DCB_HALF_WCAP2 + 2));
    uint32_t* s_rd = L.cols;                      // [ROWS][T]
    uint32_t* s_inv = s_rd + (size_t)ROWS * T;    // [ROWS][T] invalid-base column, 01 per non-ACGT symbol
    uint32_t* s_cand = s_inv + (size_t)ROWS * T;  // [DCB_HALF_CAP][T]
    uint32_t* s_n = s_cand + (size_t)DCB_HALF_CAP * T;   // [T] candidates appended per read
    uint16_t* s_work = reinterpret_cast<uint16_t*>(s_n + T) + (size_t)(tid >> 5) * DCB_HALF_WCAP;   // this warp's probe hits: lane << 8 | probe
    uint32_t* s_work2 = s_n + T + (size_t)(T / 32) * (DCB_HALF_WCAP / 2) + (size_t)(tid >> 5) * (2 * DCB_HALF_WCAP2 + 2);   // prefix hits: lane | P << 5 | set << 15
    uint32_t* s_work3 = s_work2 + DCB_HALF_WCAP2;             // (occurrence, tag) pairs: lane | P << 5 | keyword << 15 | tag index << 23
    uint32_t* s_n2 = s_work3 + DCB_HALF_WCAP2;                // lengths of the two lists
    s_rd[tid] = 0u; s_rd[(NW + 1) * T + tid] = 0u; s_rd[(NW + 2) * T + tid] = 0u;
    s_inv[tid] = 0u; s_inv[(NW + 1) * T + tid] = 0u; s_inv[(NW + 2) * T + tid] = 0u;
    stage_tables(L, tb);
    const DcbTag* vtags = gene_tags(L.t[0]);
    const DcbTag* jtags = gene_tags(L.t[1]);
    const HalfView hx = half_view(L.t[2]);
    const uint32_t t7 = smem_u32(hx.t);
    uint32_t* col = s_rd + T + tid;               // word k of this thread's read at col[k * T]
    uint32_t* icol = s_inv + T + tid;

    ExcList ex;
    ex.read = b.exc_read; ex.pos = b.exc_pos; ex.kind = b.exc_kind; ex.n = b.n_exc;
    for (uint32_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const uint32_t item = tile * T + tid;
        const bool live = item < n_items;
        const uint32_t ri = live ? __ldg(queue + item) : b.first;
        uint32_t w[NW];
        {
            const uint4* src = reinterpret_cast<const uint4*>(b.words + (size_t)ri * NW);
#pragma unroll
            for (int k = 0; k < NW / 4; k++) {
                const uint4 v = ldg_stream(src + k);
                w[4 * k + 0] = v.x; w[4 * k + 1] = v.y; w[4 * k + 2] = v.z; w[4 * k + 3] = v.w;
            }
#pragma unroll
            for (int k = 0; k < NW; k++) col[k * T] = w[k];
        }
        const uint4 hand = *reinterpret_cast<const uint4*>(results + ri);
        uint32_t hv = hand.x, hj = hand.y, need = 0;
        ReadView r;
        r.w = col; r.stride = T; r.nw = NW;
        r.n = b.uniform_len ? (int)b.uniform_len : (int)__ldg(b.lens + ri);
        const uint32_t* inv2 = nullptr;
        bool act = live;                          // still being decided here; live && !act: passed on
        if (live) {
            const bool flagged = b.n_exc && ((__ldg(b.flags + (ri >> 5)) >> (ri & 31)) & 1u);
            const uint32_t e0 = hand.z;           // the read's first entry in the exception list, from the exact-tag kernel
            ExcList exr = ex;
            if (flagged) exr.n = __ldg(b.exc_index + (ri >> 5) + 1);   // its entries end inside its 32-read group's run
            act = half_begin(r, inv2, flagged, exr, e0, icol, vtags, jtags, hv, hj, need, hx.j_ok != 0);
        }
        if (!act) need = 0;
        s_n[tid] = 0u;
        // 1. probe: bit i of the mask <=> the 7-mer at base 4 i occurs, at an offset < 4, in a half keyword of a gene that
        //    is still missing
        uint32_t cm[NM];
#pragma unroll
        for (int m = 0; m < NM; m++) cm[m] = 0u;
        if (__any_sync(0xFFFFFFFFu, need != 0u)) {
#pragma unroll
            for (int i = 0; i < NPOS; i++) {
                const int a = i >> 2, sh = (i & 3) * 8;
                const uint32_t win = sh <= 16 ? (w[a] >> sh) : __funnelshift_r(w[a], a + 1 < NW ? w[a + 1] : 0u, sh);
                uint32_t e;
                asm("ld.shared.u16 %0, [%1];" : "=r"(e) : "r"(t7 + ((win & 0x3FFFu) << 1)));
                cm[i >> 5] |= ((e & need) ? 1u : 0u) << (i & 31);
            }
            const int nvalid = r.n >= DCB_HALF_Q ? (r.n - DCB_HALF_Q) / DCB_HALF_STRIDE + 1 : 0;   // probes inside the read
#pragma unroll
            for (int m = 0; m < NM; m++) {
                const int keep = nvalid - 32 * m;
                if (keep < 32) cm[m] &= keep > 0 ? ((1u << keep) - 1u) : 0u;
            }
        }
        // 2. pool the probe hits of the warp's 32 reads in one list, so that confirming them keeps all lanes busy whatever
        //    their distribution over the reads (measured before: 6 of 32 lanes active when every lane confirmed its own)
        int mine = 0;
#pragma unroll
        for (int m = 0; m < NM; m++) mine += __popc(cm[m]);
        int incl = mine;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int t = __shfl_up_sync(0xFFFFFFFFu, incl, d);
            if (lane >= d) incl += t;
        }
        int at = incl - mine;
        const bool fits = incl <= DCB_HALF_WCAP;
        const int n_work = __reduce_max_sync(0xFFFFFFFFu, fits ? incl : 0);
        if (mine && !fits) act = false;
        if (fits) {
#pragma unroll
            for (int m = 0; m < NM; m++)
                for (uint32_t c = cm[m]; c; c &= c - 1u) s_work[at++] = (uint16_t)((lane << 8) | (32 * m + __ffs(c) - 1));
        }
        __syncwarp();
        // 3. confirm, in three flat stages with all lanes busy in each:
        //    a. lane k takes probe hit k of the list -- another lane's read as a rule -- and looks the keyword prefix of
        //       every (set, offset) the probe entry names up; a prefix that exists goes on the warp's second list
        if (lane == 0) { s_n2[0] = 0u; s_n2[1] = 0u; }
        __syncwarp();
        for (int k0 = 0; k0 < n_work; k0 += 32) {
            const bool has = k0 + lane < n_work;
            const uint32_t it = has ? s_work[k0 + lane] : (uint32_t)(lane << 8);
            const int src = (int)(it >> 8), p = DCB_HALF_STRIDE * (int)(it & 255u);
            const uint32_t need_s = __shfl_sync(0xFFFFFFFFu, need, src);
            const int n_s = __shfl_sync(0xFFFFFFFFu, r.n, src);
            if (has) {
                ReadView rs;
                rs.w = s_rd + T + wbase + src; rs.stride = T; rs.nw = NW; rs.n = n_s;
                const uint32_t* c0 = rs.w + (p >> 4) * T;
                const uint32_t win = __funnelshift_r(c0[0], c0[T], (p & 15) * 2);
                for (uint32_t e = hx.t[win & 0x3FFFu] & need_s; e; e &= e - 1u) {
                    const int bit = __ffs(e) - 1, P = p - (bit & 3);
                    if (half_prefix<true>(rs, hx, bit >> 2, P)) {
                        const uint32_t at = atomicAdd(s_n2, 1u);
                        if (at < DCB_HALF_WCAP2) s_work2[at] = (uint32_t)src | ((uint32_t)P << 5) | ((uint32_t)(bit >> 2) << 15);
                        else atomicAdd(s_n + wbase + src, DCB_HALF_BAIL);                          // list full: pass the read on
                    }
                }
            }
        }
        __syncwarp();
        //    Round 0: the prefix hits of the sampled index.  Rounds 1, 2, ..., only for chains whose J halves are below the sampled
        //    index (j_short: 12-nt J tags): a read whose V is assigned and whose J is missing is probed with the 6-mer table at
        //    every base, the warp's lanes taking 8 bases each; the occurrences go on the (empty again) second list and through
        //    the same two stages, a few reads per round.  Where the exact-tag kernel did not search J, the full J tags are
        //    compared as well.
        uint32_t mw = 0;                                        // reads of this warp still to be scanned (rounds 1, 2, ...)
        for (int round = 0;; round++) {
            if (round >= 1) {
                if (round == 1) {
                    if (!hx.j_short) break;
                    mw = __ballot_sync(0xFFFFFFFFu, act && half_jshort_ok(hx, hv, hj, s_cand + tid, T, DCB_HALF_CAP, s_n[tid]));
                }
                if (!mw) break;
                if (lane == 0) { s_n2[0] = 0u; s_n2[1] = 0u; }
                __syncwarp();
                while (mw) {                                    // as many reads per round as the lists take comfortably
                    const int src = __ffs(mw) - 1;
                    mw &= mw - 1u;
                    const int n_s = __shfl_sync(0xFFFFFFFFu, r.n, src);
                    const uint32_t* cs = s_rd + T + wbase + src;
                    for (int base = 0; base + DCB_HALF_JQ <= n_s; base += 256) {
                        const int p0 = base + 8 * lane;
                        uint32_t found = 0;                     // bit k: a J half keyword may start at p0 + k
                        if (p0 + DCB_HALF_JQ <= n_s) {
                            const uint32_t* c0 = cs + (p0 >> 4) * T;
                            const uint64_t w64 = (((uint64_t)c0[T] << 32) | c0[0]) >> ((p0 & 15) * 2);
#pragma unroll
                            for (int k = 0; k < 8; k++)
                                found |= (hx.jt[(uint32_t)(w64 >> (2 * k)) & 0xFFFu] != 0 && p0 + k + DCB_HALF_JQ <= n_s ? 1u : 0u) << k;
                        }
                        for (; found; found &= found - 1u) {
                            const uint32_t at = atomicAdd(s_n2, 1u);
                            if (at < DCB_HALF_WCAP2) s_work2[at] = (uint32_t)src | ((uint32_t)(p0 + __ffs(found) - 1) << 5) | (1u << 17);
                            else atomicAdd(s_n + wbase + src, DCB_HALF_BAIL);               // list full: pass the read on
                        }
                    }
                    __syncwarp();
                    if (s_n2[0] >= DCB_HALF_WCAP2 / 3) break;
                }
            }
            //    a'. lane k takes prefix hit k: the keywords with that prefix are compared with the read as a whole; an occurrence
            //       puts one item per tag that has this half on the third list
            const int n_pre = (int)min(s_n2[0], (uint32_t)DCB_HALF_WCAP2);
            for (int k0 = 0; k0 < n_pre; k0 += 32) {
                const bool has = k0 + lane < n_pre;
                const uint32_t it = has ? s_work2[k0 + lane] : (uint32_t)lane;
                const int src = (int)(it & 31u), P = (int)((it >> 5) & 1023u), set = (int)((it >> 15) & 3u);
                const int n_s = __shfl_sync(0xFFFFFFFFu, r.n, src);
                const int flg_s = __shfl_sync(0xFFFFFFFFu, inv2 != nullptr ? 1 : 0, src);
                const uint32_t fu_s = __shfl_sync(0xFFFFFFFFu, DCB_FU_OF(hv, hj), src);   // genes whose full tags are not searched yet
                if (has) {
                    ReadView rs;
                    rs.w = s_rd + T + wbase + src; rs.stride = T; rs.nw = NW; rs.n = n_s;
                    struct Sink {
                        uint32_t* list; uint32_t* n3; uint32_t* n_src; uint32_t base;
                        __device__ __forceinline__ void operator()(int id, int n_tags) {
                            const uint32_t at = atomicAdd(n3, (uint32_t)n_tags);
                            if (at + n_tags > DCB_HALF_WCAP2) {             // list full: pass the read on; what was reserved is void
                                atomicAdd(n_src, DCB_HALF_BAIL);
                                for (uint32_t q = at; q < DCB_HALF_WCAP2; q++) list[q] = 0xFFFFFFFFu;
                                return;
                            }
                            for (int ti = 0; ti < n_tags; ti++) list[at + ti] = base | ((uint32_t)id << 15) | ((uint32_t)ti << 23);
                        }
                    } sink{s_work3, s_n2 + 1, s_n + wbase + src, (uint32_t)src | ((uint32_t)P << 5) | (fu_s << 27)};
                    uint32_t meta;
                    if ((it >> 17) & 1u) {                          // a 6-mer hit of the J scan
                        uint32_t lo, hi;
                        rd_win32x<true>(rs, P, lo, hi);
                        meta = hx.jt[lo & 0xFFFu];
                    } else {
                        meta = half_prefix<true>(rs, hx, set, P);
                    }
                    half_keywords<true>(rs, flg_s ? s_inv + T + wbase + src : nullptr, hx, meta, P, sink);
                }
            }
            __syncwarp();
            //    b. lane k takes item k of the third list: one (occurrence, tag) pair -> length guard, Hamming <= 1, the
            //       candidate appended to its read's list
            const int n_work2 = (int)min(s_n2[1], (uint32_t)DCB_HALF_WCAP2);
            for (int k0 = 0; k0 < n_work2; k0 += 32) {
                uint32_t it = k0 + lane < n_work2 ? s_work3[k0 + lane] : 0xFFFFFFFFu;
                const bool has = it != 0xFFFFFFFFu;
                if (!has) it = (uint32_t)lane;
                const int src = (int)(it & 31u);
                const int n_s = __shfl_sync(0xFFFFFFFFu, r.n, src);
                const int flg_s = __shfl_sync(0xFFFFFFFFu, inv2 != nullptr ? 1 : 0, src);
                if (has) {
                    ReadView rs;
                    rs.w = s_rd + T + wbase + src; rs.stride = T; rs.nw = NW; rs.n = n_s;
                    const uint32_t* inv_s = flg_s ? s_inv + T + wbase + src : nullptr;
                    const int id = (int)((it >> 15) & 255u), ti = (int)((it >> 23) & 15u), P = (int)((it >> 5) & 1023u);
                    half_candidate<true>(rs, inv_s, hx, vtags, jtags, id, ti, P, s_cand + wbase + src, DCB_HALF_CAP, s_n + wbase + src);
                    if ((it >> 27) & 3u)
                        half_full_candidate<true>(rs, inv_s, hx, vtags, jtags, id, ti, P, (it >> 27) & 3u, s_cand + wbase + src, DCB_HALF_CAP, s_n + wbase + src);
                }
            }
            __syncwarp();
        }
        // 4. decide: the candidates in the reference's order
        bool pass_on = live && !act;
        if (act) {
            dcb_result out;
            *reinterpret_cast<uint4*>(&out) = make_uint4(0, 0, 0, 0);
            uint32_t pend = 0;
            if (half_run<true>(r, inv2, hx, vtags, jtags, hv, hj, s_cand + tid, DCB_HALF_CAP, s_n[tid], prm, out, pend)) {
                store_result(results + ri, out);
                half_commit(pend, L.cnt);
            } else {
                pass_on = true;
            }
        }
        defer_reads(pass_on, ri, queue2, queue2_count);
        __syncwarp();
    }
    pdl_launch_dependents();
    flush_counters(L.cnt, counters);
    stamp_end(ts);
}

// ------------------------------------------------------------------------------------------------
// general kernel (queued reads, or every read when queue == nullptr)
// ------------------------------------------------------------------------------------------------
#ifndef DCB_GENERAL_MIN_SPREAD
#define DCB_GENERAL_MIN_SPREAD 4
#endif
__global__ void __launch_bounds__(kGeneralThreads, DCB_GENERAL_BLOCKS)
dcb_general_kernel(BatchDev b, Tables4 tb, DcrParams prm, int both_frames, dcb_result* __restrict__ results,
                   unsigned long long* __restrict__ counters, const uint32_t* __restrict__ queue,
                   const uint32_t* __restrict__ queue_count, uint32_t* __restrict__ zero_next, TierStamp* ts) {
    extern __shared__ __align__(16) uint32_t smem[];
    const int T = blockDim.x;
    stamp_start(ts);
    pdl_wait();
    // the last kernel of a resident step clears the counter set of the NEXT step (dcb_run_resident): every kernel that
    // used that set -- the previous step's -- has completed by now, and the next step's kernels wait for this one
    if (zero_next && blockIdx.x == 0)
        for (int i = threadIdx.x; i < (int)kCounterSetWords; i += T) zero_next[i] = 0u;
    // A short queue is spread thinly: S reads per warp (lanes 0 .. S-1), so that all of it runs in one wave of warps and a
    // warp serialises S divergent paths instead of 32 -- the reads that get here are the odd ones, each on a path of its
    // own, and a tile's latency is its slowest warp's (measured on configs[2]: 9 k reads took 0.16 ms at 32 per warp).
    const uint32_t n_items = queue ? *queue_count : b.n_reads;
    uint32_t S = 32;
    {
        const uint64_t warps = (uint64_t)gridDim.x * (uint32_t)(T >> 5);
        while (S > DCB_GENERAL_MIN_SPREAD && (uint64_t)n_items <= warps * (S >> 1)) S >>= 1;
    }
    const uint32_t per_tile = (uint32_t)(T >> 5) * S;
    const uint32_t n_tiles = (n_items + per_tile - 1) / per_tile;
    if (blockIdx.x >= n_tiles) { stamp_end(ts); return; }   // nothing for this block: do not even stage the tables
    const int nw = (int)b.slot_words, nwi = (nw + 1) / 2;
    SmemLayout L = carve(smem, tb, (size_t)(nw + nwi) * T * (both_frames ? 2 : 1) + (size_t)(nwi + DCB_HITS_CAP + 6) * T + 20);
    uint32_t* s_rd = L.cols;                      // [nw][T]
    uint32_t* s_inv = s_rd + (size_t)nw * T;      // [nwi][T]
    uint32_t* s_cand = s_inv + (size_t)nwi * T;   // [nwi][T] candidate keyword positions
    uint32_t* s_hits = s_cand + (size_t)nwi * T;  // [DCB_HITS_CAP][T] keyword occurrences
    uint32_t* s_meta = s_hits + (size_t)DCB_HITS_CAP * T;  // [5][T] read index, length, exception range, view flags
    uint16_t* s_perm = reinterpret_cast<uint16_t*>(s_meta + (size_t)5 * T);   // [T] column of the t-th read after regrouping
    uint32_t* s_cls = s_meta + (size_t)5 * T + (T + 1) / 2;        // [18] class counters / offsets
    uint32_t* s_rd1 = s_cls + 20;                 // second frame (only when both_frames)
    uint32_t* s_inv1 = s_rd1 + (size_t)nw * T;
    stage_tables(L, tb);
    const uint32_t* vblob = L.t[0];
    const uint32_t* jblob = L.t[1];
    const uint32_t* sfilt = tb.words[2] ? L.t[2] : nullptr;      // union suffix filter

    const int tid = threadIdx.x;
    const uint32_t slot = (uint32_t)(tid >> 5) * S + (uint32_t)(tid & 31);   // this thread's place among the tile's reads
    const bool placed = (uint32_t)(tid & 31) < S;
    ExcList ex;
    ex.read = b.exc_read; ex.pos = b.exc_pos; ex.kind = b.exc_kind; ex.n = b.n_exc;
    for (uint32_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        // ---- step 1: thread t prepares the read in column t (marks, invalid-base mask, hit list) and classifies it
        const uint32_t item = tile * per_tile + slot;
        const bool live = placed && item < n_items;
        int cls = 16;                                      // dead column (past the end of the queue)
        __syncthreads();                                   // the previous tile is done with the columns and s_cls
        if (tid < 18) s_cls[tid] = 0u;
        __syncthreads();
        if (live) {
            const uint32_t ri = queue ? queue[item] : b.first + item;
            const uint4* src = reinterpret_cast<const uint4*>(b.words + (size_t)ri * b.slot_words);
            for (int k = 0; k < nw / 4; k++) {
                uint4 v = __ldg(src + k);
                s_rd[(4 * k + 0) * T + tid] = v.x;
                s_rd[(4 * k + 1) * T + tid] = v.y;
                s_rd[(4 * k + 2) * T + tid] = v.z;
                s_rd[(4 * k + 3) * T + tid] = v.w;
            }
            ReadView r;
            r.w = s_rd + tid; r.stride = T;
            r.n = b.uniform_len ? (int)b.uniform_len : (int)__ldg(b.lens + ri);
            r.nw = nw;
            const bool flagged = b.n_exc && ((__ldg(b.flags + (ri >> 5)) >> (ri & 31)) & 1u);
            ExcList exr = ex;                          // the read's entries lie inside its 32-read group's run of the list
            if (flagged) { exr.lo = __ldg(b.exc_index + (ri >> 5)); exr.n = __ldg(b.exc_index + (ri >> 5) + 1); }
            cls = dcr_general_prepare(r, ri, flagged, exr, s_inv + tid, vblob, jblob, sfilt, s_cand + tid, s_hits + tid);
            uint32_t* m = s_meta + tid;                    // what step 2 needs to rebuild the view of this column
            m[0] = ri; m[T] = (uint32_t)r.n; m[2 * T] = (uint32_t)r.e0; m[3 * T] = (uint32_t)r.e1;
            m[4 * T] = (uint32_t)r.n_hits | (r.hits ? 0x100u : 0u) | (r.inv ? 0x200u : 0u) | (r.cand ? 0x400u : 0u) |
                       ((uint32_t)r.cand_kq << 16);
        }
        // ---- regroup: counting sort of the columns by class, so that a warp of step 2 runs mostly one path
        const uint32_t rank = atomicAdd(&s_cls[cls], 1u);  // shared-memory atomics, 17 counters
        __syncthreads();
        if (tid == 0) {
            uint32_t acc = 0;
            for (int k = 0; k < 17; k++) { const uint32_t c = s_cls[k]; s_cls[k] = acc; acc += c; }
            s_cls[17] = acc;
        }
        __syncthreads();
        s_perm[s_cls[cls] + rank] = (uint16_t)tid;
        __syncthreads();
        // ---- step 2: thread t analyses column s_perm[t] (dead columns sort last)
        const int col = s_perm[placed ? slot : 0];
        if (placed && slot < s_cls[16]) {                  // live columns: classes 0..15
            const uint32_t* m = s_meta + col;
            const uint32_t ri = m[0], fl = m[4 * T];
            ReadView r;
            r.w = s_rd + col; r.stride = T; r.n = (int)m[T]; r.nw = nw;
            r.exc_pos = ex.pos; r.exc_kind = ex.kind; r.e0 = (int)m[2 * T]; r.e1 = (int)m[3 * T]; r.mirror = 0;
            r.inv = (fl & 0x200u) ? s_inv + col : nullptr;
            r.cand = (fl & 0x400u) ? s_cand + col : nullptr; r.cand_kq = (int)(fl >> 16);
            r.hits = (fl & 0x100u) ? s_hits + col : nullptr; r.n_hits = (int)(fl & 0xFFu);
            dcb_result out;
            *reinterpret_cast<uint4*>(&out) = make_uint4(0, 0, 0, 0);
            dcr_general_run(r, ex, s_rd1 + col, s_inv1 + col, vblob, jblob, prm, both_frames, out, L.cnt, sfilt,
                            s_cand + col, s_hits + col);
            store_result(results + ri, out);
        }
    }
    pdl_launch_dependents();
    flush_counters(L.cnt, counters);
    stamp_end(ts);
}

#include "pack_device.cuh"

// ------------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------------
#define CUDA_TRY(expr)                                                                          \
    do {                                                                                        \
        cudaError_t e__ = (expr);                                                               \
        if (e__ != cudaSuccess) {                                                               \
            dcb_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
            return DCB_ENOGPU;                                                                  \
        }                                                                                       \
    } while (0)

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return DCB_OK;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        if (cudaMalloc(&p, want) != cudaSuccess) {
            dcb_set_error("cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(cudaGetLastError()));
            return DCB_ENOMEM;
        }
        cap = want;
        return DCB_OK;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

struct dcb_ctx {
    int device = 0;
    int n_sms = 0;
    dcb_params params{};
    cudaStream_t own_stream = nullptr, stream = nullptr, stream2 = nullptr;
    cudaEvent_t ev_ready = nullptr, ev_done = nullptr;
    // device copies of the table blobs: general (V, J), tag records (V, J), seed indexes (V, J, union of both)
    uint32_t *d_vgen = nullptr, *d_jgen = nullptr, *d_vcore = nullptr, *d_jcore = nullptr;
    uint32_t *d_vidx = nullptr, *d_jidx = nullptr, *d_uidx = nullptr;
    uint32_t* d_sfilt = nullptr;   // union suffix filter of the general kernel
    int sfilt_words = 0;
    uint32_t* d_half = nullptr;    // sampled half-tag index (null: the chain has half tags too short for it)
    int half_words = 0;
    void* half_fn = nullptr;       // half-tag kernel picked for the resident batch, or null
    int half_grid = 0, half_threads = 0;
    size_t half_smem = 0;
    DevBuf queue2;                 // reads the half-tag kernel passes on to the general kernel
    // device-side packing (dcb_decombine_ascii / dcb_pack_device): text and per-read offsets / lengths of the chunk in
    // flight on each of the two streams, exception counts per 32-read group, the running total of the exception list
    DevBuf text[2], roff[2], rlen[2], group_count;
    uint32_t* d_exc_total = nullptr;
    cudaEvent_t ev_scan[2] = {nullptr, nullptr};
    // page-locked staging for text that arrives in pageable memory (a memory-mapped FASTQ file): host threads copy the
    // chunk in, the copy engine takes it from there at link speed while the threads fill the other buffer
    char* stage[2] = {nullptr, nullptr};
    size_t stage_cap[2] = {0, 0};
    cudaEvent_t ev_stage[2] = {nullptr, nullptr};
    // pageable text in dcb_decombine_ascii: chunks of clean reads packed by the host threads (dcb_pack_words) into
    // page-locked buffers, two so that the threads fill one while the copy engine takes the other
    uint32_t* hwords[2] = {nullptr, nullptr};
    size_t hwords_cap[2] = {0, 0};
    cudaEvent_t ev_hw[2] = {nullptr, nullptr};
    uint32_t host_chunks = 0, device_chunks = 0;   // of the last dcb_decombine_ascii call
    // two-ended sharing (ascii_two_ended): the device takes the chunks from the front, a host thread packs chunks from the
    // back into ONE page-locked region (slot i = the i-th chunk from the end) until the two meet
    char* hstage = nullptr;
    size_t hstage_cap = 0;
    cudaEvent_t ev_text[2] = {nullptr, nullptr};   // the text copy of the last device chunk of each parity
    cudaStream_t stream3 = nullptr;                // the worker's copies of the chunks it packed
    std::vector<cudaEvent_t> ev_hcopy;             // one per chunk: its packed words have arrived
    bool text_pending[2] = {false, false};
    double pack_ms = 0;            // device time of the pack kernels of the last dcb_pack_device call (CUDA events)
    int vgen_words = 0, jgen_words = 0, vcore_words = 0, jcore_words = 0, vidx_words = 0, jidx_words = 0, uidx_words = 0;
    DevBuf words, lens, flags, exc_read, exc_pos, exc_kind, exc_index, results, queue;
    std::vector<uint32_t> h_exc_index;   // host copy of exc_index while its upload is in flight
    uint32_t exc_cap = 0;                // entries of the device-side exception list of the batch being packed on the device
    uint32_t* d_queue_count = nullptr;   // two counter sets of kCounterSetWords (dcb_run_resident alternates them)
    int set_last = 0, set_next = 0;      // the set the last run used; the (zeroed) set the next resident step uses
    BatchDev batch{};
    bool have_batch = false, ran = false;
    bool timing = false;
    TierStamp* d_stamps = nullptr;       // one entry per timed launch since the last collection
    std::vector<int> stamp_slot;         // the timer slot of each entry in use
    double ms[DCB_NTIMERS] = {0, 0, 0, 0};
    uint64_t launches[DCB_NTIMERS] = {0, 0, 0, 0};
    int exact_grid = 0, general_grid = 0, exact_threads = kExactThreads, general_threads = kGeneralThreads;
    size_t exact_smem = 0, general_smem = 0;
    // seed geometry of the two genes and the union bitmap (built when they agree)
    int qv = 0, sv = 0, qj = 0, sj = 0, lminv = 0, lminj = 0;
    int vhead = 0, jhead = 0, uhead = 0, vbloom = 0, jbloom = 0, ubloom = 0;   // head_words / bloom_off of the three indexes
    void* spec_fn = nullptr;   // specialised exact kernel picked for the resident batch, or null
    void* q_fn = nullptr;      // flat kernel picked for the resident batch, or null (then spec_fn / the generic kernel run)
    int ulegacy = 0, uqtab_off = 0, uqtab_words = 0, ubfilter_off = 0, ufbits = 0, uqq = 0, uqs = 0, utqbits = 0;
    int vlegacy = 0, jlegacy = 0;
    bool spec_union = false;
};

typedef void (*exact_spec_fn)(BatchDev, Tables4, SpecBlooms, DcrParams, int, dcb_result*, unsigned long long*, uint32_t*, uint32_t*, TierStamp*);

// Specialisations compiled in: V seeds (q=9, stride 12) -- every shipped V tag set has 20-nt minimum tags --
// with J either sharing that geometry (20-nt J tags: one union index) or using (q=8, stride 5) (12-nt J tags).
static exact_spec_fn pick_spec(int nw, int qv, int sv, int lminv, int qj, int sj, int lminj, bool* is_union) {
    if (qv != 9 || sv != 12 || lminv != 20) return nullptr;
    const bool uni = (qj == 9 && sj == 12 && lminj == 20), sep = (qj == 8 && sj == 5 && lminj == 12);
    if (!uni && !sep) return nullptr;
    *is_union = uni;
#define DCB_SPEC(NW) (uni ? dcb_exact_kernel_spec<NW, 9, 12, DCB_WBITS_UNION, 9, 12, DCB_WBITS_UNION, true> \
                          : dcb_exact_kernel_spec<NW, 9, 12, DCB_WBITS_SINGLE, 8, 5, DCB_WBITS_SINGLE, false>)
    switch (nw) {
        case 8:  return DCB_SPEC(8);
        case 12: return DCB_SPEC(12);
        case 16: return DCB_SPEC(16);
        case 20: return DCB_SPEC(20);
        default: return nullptr;
    }
#undef DCB_SPEC
}
// Flat kernel: chains whose V and J tags share one index with 20-nt minimum tags (13-mer seeds at stride 8), read slots
// up to 20 words (320 nt: two hit words).
typedef void (*exact_q_fn)(BatchDev, QTables, DcrParams, int, dcb_result*, unsigned long long*, uint32_t*, uint32_t*, TierStamp*);
static constexpr int kQThreads = 1024;
static exact_q_fn pick_q(int nw, int qq, int qs, int lmin, bool exc) {
    if (qq != 13 || qs != 8 || lmin != 20) return nullptr;
#define DCB_FLAT(NW) (exc ? dcb_exact_kernel_flat<NW, 13, 8, kQThreads, true> : dcb_exact_kernel_flat<NW, 13, 8, kQThreads, false>)
    switch (nw) {
        case 8:  return DCB_FLAT(8);
        case 12: return DCB_FLAT(12);
        case 16: return DCB_FLAT(16);
        case 20: return DCB_FLAT(20);
        default: return nullptr;
    }
#undef DCB_FLAT
}
static int q_rows(int nw) {   // must match the kernel's ROWS
    const int npos = (16 * nw - 13) / 8 + 1, wmax = ((npos - 1) * 8 - 7) >> 4;
    const int trail = wmax + 3 - nw > 1 ? wmax + 3 - nw : 1;
    return 1 + nw + trail;
}

typedef void (*halftag_fn)(BatchDev, Tables4, DcrParams, dcb_result*, unsigned long long*, const uint32_t*, const uint32_t*, uint32_t*, uint32_t*,
                           TierStamp*);
// block width per slot size: as wide as the read / invalid-base / candidate columns leave room for beside the tables
static halftag_fn pick_half(int nw, int attempt, int* threads) {
    // widest first; the later attempts are for tag sets whose tables leave less room
#define DCB_HALF_PICK(NW_, T_) { *threads = T_; return dcb_halftag_kernel<NW_, T_>; }
    switch (nw * 4 + attempt) {
        case 32: DCB_HALF_PICK(8, 768)
        case 33: DCB_HALF_PICK(8, 640)
        case 48: DCB_HALF_PICK(12, 768)
        case 49: DCB_HALF_PICK(12, 640)
        case 64: DCB_HALF_PICK(16, 736)
        case 65: DCB_HALF_PICK(16, 672)
        case 66: DCB_HALF_PICK(16, 608)
        case 80: DCB_HALF_PICK(20, 608)
        case 81: DCB_HALF_PICK(20, 544)
        default: return nullptr;
    }
#undef DCB_HALF_PICK
}

// rows of shared memory per read column in the specialised kernel (must match the kernel's ROWS)
static int spec_rows(int nw, bool uni) {
    auto wmax = [&](int q, int s) { const int npos = (16 * nw - q) / s + 1; return ((npos - 1) * s - (s)) >> 4; };  // wlead == stride
    const int wm = uni ? wmax(9, 12) : std::max(wmax(9, 12), wmax(8, 5));
    const int trail = wm + 3 - nw > 0 ? wm + 3 - nw : 0;
    return 1 + nw + trail;
}

static int upload_blob(const std::vector<uint32_t>& v, uint32_t** d, int* words) {
    CUDA_TRY(cudaMalloc((void**)d, v.size() * 4));
    CUDA_TRY(cudaMemcpy(*d, v.data(), v.size() * 4, cudaMemcpyHostToDevice));
    *words = (int)v.size();
    return DCB_OK;
}

// Per-launch timing without host events between the launches (they would end the programmatic overlap of a resident
// step): each timed kernel stamps its entry of d_stamps itself (TierStamp); the entries are added up, and zeroed for
// reuse, when they are collected -- by dcb_timing_get / dcb_timing_reset, or when every entry is in use.
static constexpr int kStamps = 4096;
static int timing_collect(dcb_ctx* c) {
    if (c->stamp_slot.empty()) return DCB_OK;
    std::vector<TierStamp> h(c->stamp_slot.size());
    CUDA_TRY(cudaMemcpyAsync(h.data(), c->d_stamps, h.size() * sizeof(TierStamp), cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaMemsetAsync(c->d_stamps, 0, h.size() * sizeof(TierStamp), c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    for (size_t i = 0; i < h.size(); i++) {
        const unsigned long long t0 = ~h[i].nstart;
        if (h[i].nstart == 0 || h[i].end < t0) continue;   // not stamped (a launch that failed)
        c->ms[c->stamp_slot[i]] += (double)(h[i].end - t0) * 1e-6;
        c->launches[c->stamp_slot[i]] += 1;
    }
    c->stamp_slot.clear();
    return DCB_OK;
}
// The entry a timed launch of timer `slot` stamps, or null when timing is off.
static int timing_entry(dcb_ctx* c, int slot, bool timed, TierStamp** ts) {
    *ts = nullptr;
    if (!timed || !c->timing) return DCB_OK;
    if ((int)c->stamp_slot.size() == kStamps) {
        int rc;
        if ((rc = timing_collect(c))) return rc;
    }
    *ts = c->d_stamps + c->stamp_slot.size();
    c->stamp_slot.push_back(slot);
    return DCB_OK;
}

// A kernel launch; pdl: with the programmatic stream serialization attribute (see pdl_wait).
template <typename... P, typename... A>
static cudaError_t launch(bool pdl, void (*fn)(P...), int grid, int threads, size_t smem, cudaStream_t s, A... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3((unsigned)threads); cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, fn, args...);
}

extern "C" {

dcb_ctx* dcb_ctx_create(int device, const dcb_tagset* v, const dcb_tagset* j, const dcb_params* p) {
    if (!v || !j || !p) { dcb_set_error("dcb_ctx_create: null argument"); return nullptr; }
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0) {
        (void)cudaGetLastError();
        dcb_set_error("dcb_ctx_create: no CUDA device available (there is no CPU fallback)");
        return nullptr;
    }
    if (device < 0 || device >= n_dev) { dcb_set_error("dcb_ctx_create: device %d out of range", device); return nullptr; }
    if (cudaSetDevice(device) != cudaSuccess) { dcb_set_error("cudaSetDevice failed"); return nullptr; }
    dcb_ctx* c = new dcb_ctx();
    c->device = device;
    c->params = *p;
    auto fail = [&](const char* what) -> dcb_ctx* {
        if (what) dcb_set_error("dcb_ctx_create: %s: %s", what, cudaGetErrorString(cudaGetLastError()));
        dcb_ctx_destroy(c);
        return nullptr;
    };
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return fail("cudaGetDeviceProperties");
    c->n_sms = prop.multiProcessorCount;
    if (cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking) != cudaSuccess) return fail("cudaStreamCreate");
    c->stream = c->own_stream;
    if (cudaStreamCreateWithFlags(&c->stream2, cudaStreamNonBlocking) != cudaSuccess) return fail("cudaStreamCreate");
    if (cudaEventCreateWithFlags(&c->ev_ready, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&c->ev_done, cudaEventDisableTiming) != cudaSuccess) return fail("cudaEventCreate");
    if (upload_blob(v->general, &c->d_vgen, &c->vgen_words) || upload_blob(j->general, &c->d_jgen, &c->jgen_words) ||
        upload_blob(v->core, &c->d_vcore, &c->vcore_words) || upload_blob(j->core, &c->d_jcore, &c->jcore_words) ||
        upload_blob(v->index, &c->d_vidx, &c->vidx_words) || upload_blob(j->index, &c->d_jidx, &c->jidx_words))
        return fail(nullptr);
    {
        const DcbSeedIndex& iv = *reinterpret_cast<const DcbSeedIndex*>(v->index.data());
        const DcbSeedIndex& ij = *reinterpret_cast<const DcbSeedIndex*>(j->index.data());
        c->qv = iv.q; c->sv = iv.stride; c->qj = ij.q; c->sj = ij.stride; c->lminv = iv.lmin; c->lminj = ij.lmin;
        c->vhead = iv.head_words; c->vbloom = iv.bloom_off; c->jhead = ij.head_words; c->jbloom = ij.bloom_off;
        c->vlegacy = iv.legacy_words; c->jlegacy = ij.legacy_words;
        if (v->lmin == j->lmin) {  // same seed geometry: one index (and one filter) finds both genes
            std::vector<uint32_t> u;
            if (dcb_build_seed_index(&v->tags, &j->tags, v->lmin, DCB_WBITS_UNION, u)) {
                const DcbSeedIndex& iu = *reinterpret_cast<const DcbSeedIndex*>(u.data());
                c->uhead = iu.head_words; c->ubloom = iu.bloom_off; c->ulegacy = iu.legacy_words;
                c->uqtab_off = iu.qtab_off; c->uqtab_words = iu.qtab_words; c->ubfilter_off = iu.bfilter_off; c->ufbits = iu.fbits;
                c->uqq = iu.qq; c->uqs = iu.qstride; c->utqbits = iu.tq_bits;
                if (upload_blob(u, &c->d_uidx, &c->uidx_words)) return fail(nullptr);
            }
        }
    }
    {   // union suffix filter: the general kernel marks candidate keyword positions with it
        size_t nwf = 0;
        if (dcb_tagset_suffix_filter(v, j, nullptr, 0, &nwf) == DCB_OK) {
            std::vector<uint32_t> sf(nwf);
            if (dcb_tagset_suffix_filter(v, j, sf.data(), sf.size(), &nwf) == DCB_OK)
                if (upload_blob(sf, &c->d_sfilt, &c->sfilt_words)) return fail(nullptr);
        }
    }
    {   // sampled half-tag index: what the half-tag kernel finds the half keywords with
        std::vector<uint32_t> hb;
        if (dcb_build_half_index(v, j, hb))
            if (upload_blob(hb, &c->d_half, &c->half_words)) return fail(nullptr);
    }
    // queue counters and reference counters in ONE block (both counter sets): one memset clears them all
    if (cudaMalloc((void**)&c->d_queue_count, kZeroBlockBytes) != cudaSuccess) return fail("cudaMalloc");
    if (cudaMemsetAsync(c->d_queue_count, 0, kZeroBlockBytes, c->own_stream) != cudaSuccess ||
        cudaStreamSynchronize(c->own_stream) != cudaSuccess) return fail("cudaMemset");
    if (cudaMalloc((void**)&c->d_exc_total, 16) != cudaSuccess) return fail("cudaMalloc");
    for (int i = 0; i < 2; i++)
        if (cudaEventCreateWithFlags(&c->ev_scan[i], cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&c->ev_stage[i], cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&c->ev_hw[i], cudaEventDisableTiming) != cudaSuccess) return fail("cudaEventCreate");
    for (int i = 0; i < 2; i++)
        if (cudaEventCreateWithFlags(&c->ev_text[i], cudaEventDisableTiming) != cudaSuccess) return fail("cudaEventCreate");
    return c;
}

void dcb_ctx_destroy(dcb_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->own_stream) { cudaStreamSynchronize(c->own_stream); cudaStreamDestroy(c->own_stream); }
    if (c->stream2) { cudaStreamSynchronize(c->stream2); cudaStreamDestroy(c->stream2); }
    if (c->ev_ready) cudaEventDestroy(c->ev_ready);
    if (c->ev_done) cudaEventDestroy(c->ev_done);
    cudaFree(c->d_vgen); cudaFree(c->d_jgen); cudaFree(c->d_vcore); cudaFree(c->d_jcore);
    cudaFree(c->d_vidx); cudaFree(c->d_jidx); cudaFree(c->d_uidx); cudaFree(c->d_sfilt); cudaFree(c->d_half);
    cudaFree(c->d_queue_count);   // the reference counters live in the same block
    cudaFree(c->d_stamps);
    c->words.release(); c->lens.release(); c->flags.release(); c->exc_read.release(); c->exc_pos.release(); c->exc_index.release();
    c->exc_kind.release(); c->results.release(); c->queue.release(); c->queue2.release();
    for (int i = 0; i < 2; i++) {
        c->text[i].release(); c->roff[i].release(); c->rlen[i].release();
        if (c->ev_scan[i]) cudaEventDestroy(c->ev_scan[i]);
        if (c->ev_stage[i]) cudaEventDestroy(c->ev_stage[i]);
        if (c->stage[i]) cudaFreeHost(c->stage[i]);
        if (c->ev_hw[i]) cudaEventDestroy(c->ev_hw[i]);
        if (c->hwords[i]) cudaFreeHost(c->hwords[i]);
    }
    for (int i = 0; i < 2; i++) if (c->ev_text[i]) cudaEventDestroy(c->ev_text[i]);
    if (c->hstage) cudaFreeHost(c->hstage);
    if (c->stream3) { cudaStreamSynchronize(c->stream3); cudaStreamDestroy(c->stream3); }
    for (cudaEvent_t e : c->ev_hcopy) cudaEventDestroy(e);
    c->group_count.release();
    cudaFree(c->d_exc_total);
    delete c;
}

int dcb_ctx_set_stream(dcb_ctx* c, void* cuda_stream) {
    if (!c) return DCB_EINVAL;
    c->stream = cuda_stream ? (cudaStream_t)cuda_stream : c->own_stream;
    return DCB_OK;
}

// Size the device buffers for batch P, point the BatchDev at them and pick the launch geometry.  No copies.
static int prepare_batch(dcb_ctx* c, const dcb_packed* P, size_t exc_cap = 0) {
    if (P->n_reads >= 0xFFFFFFFFull) { dcb_set_error("batch too large"); return DCB_EINVAL; }
    const size_t n = P->n_reads, sw = P->slot_words;
    if (sw == 0 || sw % 4) { dcb_set_error("slot_words must be a positive multiple of 4"); return DCB_EINVAL; }
    int rc;
    if ((rc = c->words.ensure(n * sw * 4 + 16)) || (rc = c->lens.ensure(n * 2 + 16)) ||
        (rc = c->flags.ensure(((n + 31) / 32) * 4 + 16)) || (rc = c->exc_read.ensure(std::max<size_t>(P->n_exc, exc_cap) * 4 + 16)) ||
        (rc = c->exc_pos.ensure(std::max<size_t>(P->n_exc, exc_cap) * 2 + 16)) || (rc = c->exc_kind.ensure(std::max<size_t>(P->n_exc, exc_cap) + 16)) ||
        (rc = c->exc_index.ensure(((n + 31) / 32 + 2) * 4 + 16)) ||
        (rc = c->results.ensure(n * sizeof(dcb_result) + 16)) || (rc = c->queue.ensure(n * 4 + 16)) ||
        (rc = c->queue2.ensure(n * 4 + 16)))
        return rc;
    BatchDev& b = c->batch;
    b.words = (const uint32_t*)c->words.p; b.lens = (const uint16_t*)c->lens.p; b.flags = (const uint32_t*)c->flags.p;
    b.exc_read = (const uint32_t*)c->exc_read.p; b.exc_pos = (const uint16_t*)c->exc_pos.p;
    b.exc_kind = (const uint8_t*)c->exc_kind.p; b.exc_index = (const uint32_t*)c->exc_index.p;
    b.n_reads = (uint32_t)n; b.slot_words = (uint32_t)sw; b.uniform_len = P->uniform_len; b.n_exc = P->n_exc;
    b.first = 0;
    c->have_batch = true; c->ran = false;

    // launch geometry: persistent blocks, a whole number of blocks per SM; long reads get narrower blocks
    const size_t tail = (((DCB_NCOUNTERS + 3) & ~3) + 4) * 4;
    const size_t kMaxSmem = 227 * 1024;
    const size_t nwi = (sw + 1) / 2;
    // exact-tag tables: tag records of both genes + either the union index or the two per-gene indexes
    const bool have_union = c->d_uidx != nullptr;
    const size_t tbl_e = (size_t)c->vcore_words + c->jcore_words + (have_union ? (size_t)c->ulegacy : (size_t)c->vlegacy + c->jlegacy);
    bool is_union = false;
    exact_spec_fn spec = c->params.force_general == 1 ? nullptr
                                                 : pick_spec((int)sw, c->qv, c->sv, c->lminv, c->qj, c->sj, c->lminj, &is_union);
    if (spec && is_union != have_union) spec = nullptr;
    c->spec_fn = (void*)spec; c->spec_union = have_union;
    int occ_e = 0, occ_g = 0;
    exact_q_fn qfn = nullptr;
    if (have_union && (c->params.force_general == 0 || c->params.force_general == 3) && c->ufbits == DCB_FBITS && c->utqbits > 0)
        qfn = pick_q((int)sw, c->uqq, c->uqs, c->lminv, P->n_exc != 0);
    if (qfn) {
        c->exact_smem = ((size_t)1 << DCB_FBITS) + ((size_t)q_rows((int)sw) * kQThreads +
                         c->vcore_words + c->jcore_words + c->uhead + c->uqtab_words) * 4 + tail + (P->n_exc ? kQThreads * 4 : 0);
        if (c->exact_smem > kMaxSmem) qfn = nullptr;
    }
    c->q_fn = (void*)qfn;
    if (qfn) {
        spec = nullptr; c->spec_fn = nullptr;
        c->exact_threads = kQThreads;
        CUDA_TRY(cudaFuncSetAttribute(qfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c->exact_smem));
        CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_e, qfn, c->exact_threads, c->exact_smem));
    } else if (spec) {
        // tables (index heads only) + the private copies of the filter(s) + the read columns of as wide a block as fits
        const size_t tbl_s = (size_t)c->vcore_words + c->jcore_words + (have_union ? (size_t)c->uhead : (size_t)c->vhead + c->jhead);
        const size_t blooms = have_union ? ((size_t)DCB_BLOOM_COPIES << DCB_WBITS_UNION) : 2 * ((size_t)DCB_BLOOM_COPIES << DCB_WBITS_SINGLE);
        const size_t rows = (size_t)spec_rows((int)sw, have_union);
        int T = 1024;
        for (; T >= 256; T -= 128) {
            c->exact_smem = (tbl_s + blooms + rows * T) * 4 + tail;
            if (c->exact_smem <= kMaxSmem) break;
        }
        if (T < 256) { spec = nullptr; c->spec_fn = nullptr; }
        else c->exact_threads = T;
    }
    if (qfn) {
    } else if (spec) {
        CUDA_TRY(cudaFuncSetAttribute(spec, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c->exact_smem));
        CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_e, spec, c->exact_threads, c->exact_smem));
    } else {
        int T = kExactThreads;
        for (; T >= 32; T >>= 1) {
            c->exact_smem = (tbl_e + sw * T) * 4 + tail;
            if (c->exact_smem <= kMaxSmem) break;
        }
        if (T < 32) { dcb_set_error("tag tables + %u-nt reads do not fit in shared memory", P->max_len); return DCB_EUNSUPPORTED; }
        c->exact_threads = T;
        CUDA_TRY(cudaFuncSetAttribute(dcb_exact_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c->exact_smem));
        CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_e, dcb_exact_kernel, T, c->exact_smem));
    }
    {
        int T = kGeneralThreads;
        for (; T >= 32; T -= (T > 64 ? 64 : 32)) {
            c->general_smem = ((size_t)c->vgen_words + c->jgen_words + c->sfilt_words + (sw + nwi) * T * (c->params.both_frames ? 2 : 1) + (nwi + DCB_HITS_CAP + 6) * T + 20) * 4 + tail;
            if (c->general_smem <= kMaxSmem) break;
        }
        if (T < 32) { dcb_set_error("tag tables + %u-nt reads do not fit in shared memory", P->max_len); return DCB_EUNSUPPORTED; }
        c->general_threads = T;
        CUDA_TRY(cudaFuncSetAttribute(dcb_general_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c->general_smem));
        CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_g, dcb_general_kernel, T, c->general_smem));
    }
    // half-tag kernel: between the flat kernel and the general kernel, for chains with a half-tag index (one frame only)
    c->half_fn = nullptr;
    if (c->d_half && !c->params.both_frames && c->params.force_general == 0) {
        for (int attempt = 0; attempt < 4 && !c->half_fn; attempt++) {
            int ht = 0;
            halftag_fn hf = pick_half((int)sw, attempt, &ht);
            if (!hf) break;
            const size_t smem = ((size_t)c->vcore_words + c->jcore_words + c->half_words + (2 * (sw + 3) + DCB_HALF_CAP + 1) * ht +
                                 (ht / 32) * (DCB_HALF_WCAP / 2 + 2 * DCB_HALF_WCAP2 + 2)) * 4 + tail;
            if (smem > kMaxSmem) continue;
            int occ_h = 0;
            CUDA_TRY(cudaFuncSetAttribute(hf, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_h, hf, ht, smem));
            if (occ_h >= 1) { c->half_fn = (void*)hf; c->half_grid = c->n_sms * occ_h; c->half_threads = ht; c->half_smem = smem; }
        }
    }
    if (occ_e < 1 || occ_g < 1) { dcb_set_error("kernel does not fit on an SM"); return DCB_EUNSUPPORTED; }
    const uint32_t tiles_e = (uint32_t)((n + c->exact_threads - 1) / c->exact_threads);
    const uint32_t tiles_g = (uint32_t)((n + c->general_threads - 1) / c->general_threads);
    c->exact_grid = (int)std::max<uint32_t>(1, std::min<uint32_t>(tiles_e, (uint32_t)(c->n_sms * occ_e)));
    c->general_grid = (int)std::max<uint32_t>(1, std::min<uint32_t>(tiles_g, (uint32_t)(c->n_sms * occ_g)));
    return DCB_OK;
}

// lens (unless every read has the same length), flag bits and the sparse exception list: everything but the words
static int copy_side_arrays(dcb_ctx* c, const dcb_packed* P, cudaStream_t s) {
    const size_t n = P->n_reads;
    if (n && !P->uniform_len) CUDA_TRY(cudaMemcpyAsync(c->lens.p, P->lens, n * 2, cudaMemcpyHostToDevice, s));
    if (n && P->n_exc) CUDA_TRY(cudaMemcpyAsync(c->flags.p, P->flags, ((n + 31) / 32) * 4, cudaMemcpyHostToDevice, s));
    if (P->n_exc) {
        CUDA_TRY(cudaMemcpyAsync(c->exc_read.p, P->exc_read, (size_t)P->n_exc * 4, cudaMemcpyHostToDevice, s));
        CUDA_TRY(cudaMemcpyAsync(c->exc_pos.p, P->exc_pos, (size_t)P->n_exc * 2, cudaMemcpyHostToDevice, s));
        CUDA_TRY(cudaMemcpyAsync(c->exc_kind.p, P->exc_kind, (size_t)P->n_exc, cudaMemcpyHostToDevice, s));
        // the list's end marker and the per-32-reads index the exact kernel enters the list through
        CUDA_TRY(cudaMemsetAsync((char*)c->exc_read.p + (size_t)P->n_exc * 4, 0xFF, 4, s));
        const size_t nb = (n + 31) / 32 + 1;
        c->h_exc_index.assign(nb, P->n_exc);
        uint32_t e = 0;
        for (size_t k = 0; k < nb; k++) {
            while (e < P->n_exc && P->exc_read[e] < 32 * k) e++;
            c->h_exc_index[k] = e;
        }
        CUDA_TRY(cudaMemcpyAsync(c->exc_index.p, c->h_exc_index.data(), nb * 4, cudaMemcpyHostToDevice, s));
    }
    return DCB_OK;
}

static uint32_t* counter_set(dcb_ctx* c, int set) { return c->d_queue_count + (size_t)set * kCounterSetWords; }
static unsigned long long* ref_counters(dcb_ctx* c, int set) {
    return reinterpret_cast<unsigned long long*>(counter_set(c, set) + 2 * kMaxChunks);
}

// The kernels over reads [first, first + count) of the resident batch, on stream s.  set, slot: which counter set and
// which queue counters in it.  zero_next: the counter set the general kernel clears for the next step (or null).  pdl:
// every launch with the programmatic stream serialization attribute (dcb_run_resident).
static int launch_range(dcb_ctx* c, cudaStream_t s, uint32_t first, uint32_t count, int set, int slot, uint32_t* zero_next,
                        bool timed, bool pdl) {
    if (count == 0) return DCB_OK;
    BatchDev b = c->batch;
    b.first = first; b.n_reads = count;
    uint32_t* qcount = counter_set(c, set) + slot;
    unsigned long long* counters = ref_counters(c, set);
    uint32_t* queue = (uint32_t*)c->queue.p + first;
    dcb_result* results = (dcb_result*)c->results.p;
    DcrParams prm;
    prm.allow_ns = c->params.allow_ns; prm.lenthreshold = c->params.lenthreshold;
    const uint32_t tiles_e = (count + c->exact_threads - 1) / c->exact_threads;
    const uint32_t tiles_g = (count + c->general_threads - 1) / c->general_threads;
    const int grid_e = (int)std::max<uint32_t>(1, std::min<uint32_t>(tiles_e, (uint32_t)c->exact_grid));
    const int grid_g = (int)std::max<uint32_t>(1, std::min<uint32_t>(tiles_g, (uint32_t)c->general_grid));
    const int both = c->params.both_frames;
    TierStamp* ts;
    int rc;
    if (c->params.force_general != 1) {
        if ((rc = timing_entry(c, 0, timed, &ts))) return rc;
        Tables4 te;
        te.g[0] = c->d_vcore; te.words[0] = c->vcore_words;
        te.g[1] = c->d_jcore; te.words[1] = c->jcore_words;
        if (c->spec_union) { te.g[2] = c->d_uidx; te.words[2] = c->ulegacy; te.g[3] = nullptr; te.words[3] = 0; }
        else { te.g[2] = c->d_vidx; te.words[2] = c->vlegacy; te.g[3] = c->d_jidx; te.words[3] = c->jlegacy; }
        if (c->q_fn) {
            QTables qt;
            qt.vcore = c->d_vcore; qt.jcore = c->d_jcore; qt.head = c->d_uidx; qt.qtab = c->d_uidx + c->uqtab_off;
            qt.bfilter = c->d_uidx + c->ubfilter_off;
            qt.vcore_words = c->vcore_words; qt.jcore_words = c->jcore_words; qt.head_words = c->uhead; qt.qtab_words = c->uqtab_words;
            CUDA_TRY(launch(pdl, (exact_q_fn)c->q_fn, grid_e, c->exact_threads, c->exact_smem, s, b, qt, prm, both, results, counters,
                            queue, qcount, ts));
        } else if (c->spec_fn) {
            SpecBlooms sb;
            if (c->spec_union) { te.words[2] = c->uhead; sb.v = c->d_uidx + c->ubloom; sb.j = nullptr; }
            else { te.words[2] = c->vhead; te.words[3] = c->jhead; sb.v = c->d_vidx + c->vbloom; sb.j = c->d_jidx + c->jbloom; }
            CUDA_TRY(launch(pdl, (exact_spec_fn)c->spec_fn, grid_e, c->exact_threads, c->exact_smem, s, b, te, sb, prm, both, results,
                            counters, queue, qcount, ts));
        } else {
            CUDA_TRY(launch(pdl, dcb_exact_kernel, grid_e, c->exact_threads, c->exact_smem, s, b, te, prm, both, results, counters,
                            queue, qcount, ts));
        }
    }
    Tables4 tg;
    tg.g[3] = nullptr; tg.words[3] = 0;
    if (c->half_fn) {   // the queued reads through the half-tag kernel; what it passes on is the general kernel's queue
        if ((rc = timing_entry(c, 2, timed, &ts))) return rc;
        uint32_t* qcount2 = counter_set(c, set) + kMaxChunks + slot;
        uint32_t* queue2 = (uint32_t*)c->queue2.p + first;
        tg.g[0] = c->d_vcore; tg.words[0] = c->vcore_words; tg.g[1] = c->d_jcore; tg.words[1] = c->jcore_words;
        tg.g[2] = c->d_half; tg.words[2] = c->half_words;
        const uint32_t tiles_h = (count + c->half_threads - 1) / c->half_threads;
        const int grid_h = (int)std::max<uint32_t>(1, std::min<uint32_t>(tiles_h, (uint32_t)c->half_grid));
        CUDA_TRY(launch(pdl, (halftag_fn)c->half_fn, grid_h, c->half_threads, c->half_smem, s, b, tg, prm, results, counters,
                        (const uint32_t*)queue, (const uint32_t*)qcount, queue2, qcount2, ts));
        queue = queue2; qcount = qcount2;
    }
    if ((rc = timing_entry(c, 1, timed, &ts))) return rc;
    tg.g[0] = c->d_vgen; tg.words[0] = c->vgen_words; tg.g[1] = c->d_jgen; tg.words[1] = c->jgen_words;
    tg.g[2] = c->d_sfilt; tg.words[2] = c->sfilt_words;
    CUDA_TRY(launch(pdl, dcb_general_kernel, grid_g, c->general_threads, c->general_smem, s, b, tg, prm, both, results, counters,
                    c->params.force_general == 1 ? nullptr : (const uint32_t*)queue, (const uint32_t*)qcount, zero_next, ts));
    return DCB_OK;
}

// Clear both counter sets on stream s: the chunked paths count in set 0, the next resident step in set 1.
static int reset_counter_sets(dcb_ctx* c, cudaStream_t s) {
    CUDA_TRY(cudaMemsetAsync(c->d_queue_count, 0, kZeroBlockBytes, s));
    c->set_last = 0; c->set_next = 1;
    return DCB_OK;
}

static int read_counters(dcb_ctx* c, cudaStream_t s, uint64_t* counters) {
    unsigned long long h[DCB_NCOUNTERS];
    CUDA_TRY(cudaMemcpyAsync(h, ref_counters(c, c->set_last), sizeof(h), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    if (counters) for (int i = 0; i < DCB_NCOUNTERS; i++) counters[i] += h[i];
    return DCB_OK;
}

// Reads per chunk of the chunked paths: at least base, few enough chunks for the kMaxChunks queue counters, a multiple of 1024.
static uint32_t chunk_reads(uint32_t base, uint64_t n) {
    const uint32_t chunk = std::max<uint32_t>(base, (uint32_t)((n + kMaxChunks - 1) / kMaxChunks));
    return (chunk + 1023u) & ~1023u;
}

// The chunk's kernels (chunk_no: its queue counters) and, when out is given, its result records back to the host.
static int run_chunk(dcb_ctx* c, cudaStream_t s, uint32_t first, uint32_t count, int chunk_no, dcb_result* out) {
    int rc;
    if ((rc = launch_range(c, s, first, count, 0, chunk_no, nullptr, false, false))) return rc;
    if (out)
        CUDA_TRY(cudaMemcpyAsync(out + first, (dcb_result*)c->results.p + first, (size_t)count * sizeof(dcb_result),
                                 cudaMemcpyDeviceToHost, s));
    return DCB_OK;
}

// The chunked paths alternate the chunks between st[0] and st[1]: st[1] starts behind what st[0] has queued so far, and
// st[0] ends behind all of st[1].  ran: the kernels ran; the context says so and the counters are added (synchronous).
static int fork_streams(dcb_ctx* c, const cudaStream_t st[2]) {
    CUDA_TRY(cudaEventRecord(c->ev_ready, st[0]));
    CUDA_TRY(cudaStreamWaitEvent(st[1], c->ev_ready, 0));
    return DCB_OK;
}
static int join_streams(dcb_ctx* c, const cudaStream_t st[2], bool ran, uint64_t* counters) {
    CUDA_TRY(cudaEventRecord(c->ev_done, st[1]));
    CUDA_TRY(cudaStreamWaitEvent(st[0], c->ev_done, 0));
    if (!ran) return DCB_OK;
    c->ran = true;
    return read_counters(c, st[0], counters);
}

int dcb_upload(dcb_ctx* c, const dcb_packed* P) {
    if (!c || !P) { dcb_set_error("dcb_upload: null argument"); return DCB_EINVAL; }
    CUDA_TRY(cudaSetDevice(c->device));
    int rc;
    if ((rc = prepare_batch(c, P))) return rc;
    cudaStream_t s = c->stream;
    if (P->n_reads) CUDA_TRY(cudaMemcpyAsync(c->words.p, P->words, (size_t)P->n_reads * P->slot_words * 4, cudaMemcpyHostToDevice, s));
    if ((rc = copy_side_arrays(c, P, s))) return rc;
    CUDA_TRY(cudaStreamSynchronize(s));
    return DCB_OK;
}

// A resident step is its kernels alone, chained by programmatic dependent launch (pdl_wait): step k + 1's exact kernel
// stages its tables while step k's last kernels finish, and a follow-up kernel with nothing queued costs an early exit of
// blocks already resident, not a launch behind a drained grid.  A memset in the stream would end that overlap, so the
// steps alternate between the two counter sets: a step counts in the set the step before it left zeroed, and its general
// kernel zeroes the other one for the step after it.  DCB_PDL=0: plain launches behind a memset of both sets (A/B runs).
int dcb_run_resident(dcb_ctx* c) {
    if (!c || !c->have_batch) { dcb_set_error("dcb_run_resident: no batch uploaded"); return DCB_EINVAL; }
    const char* e = std::getenv("DCB_PDL");
    if (e && std::strcmp(e, "0") && std::strcmp(e, "1")) {
        dcb_set_error("DCB_PDL=%s: accepted values are 1 (the default: the kernels of a step chained by programmatic dependent "
                      "launch) and 0 (plain launches behind a memset of the counters)", e);
        return DCB_EINVAL;
    }
    const bool pdl = !e || e[0] == '1';
    CUDA_TRY(cudaSetDevice(c->device));
    cudaStream_t s = c->stream;
    int rc;
    if (!pdl && (rc = reset_counter_sets(c, s))) return rc;
    const int set = c->set_next;
    if ((rc = launch_range(c, s, 0, c->batch.n_reads, set, 0, pdl ? counter_set(c, 1 - set) : nullptr, true, pdl))) return rc;
    // An empty batch launches nothing, so no general kernel zeroes the other set: the step reports the (zeroed) set it
    // would have counted in, and the next step counts there again.
    c->set_last = set;
    if (c->batch.n_reads) c->set_next = 1 - set;
    c->ran = true;
    return DCB_OK;
}

int dcb_download(dcb_ctx* c, dcb_result* out, uint64_t* counters) {
    if (!c || !c->ran) { dcb_set_error("dcb_download: nothing has been run"); return DCB_EINVAL; }
    CUDA_TRY(cudaSetDevice(c->device));
    cudaStream_t s = c->stream;
    if (out && c->batch.n_reads)
        CUDA_TRY(cudaMemcpyAsync(out, c->results.p, (size_t)c->batch.n_reads * sizeof(dcb_result), cudaMemcpyDeviceToHost, s));
    return read_counters(c, s, counters);
}

// Host buffers in, host buffers out.  The batch is cut into chunks that alternate between two streams, so the upload of
// one chunk, the kernels of another and the download of a third overlap (the copy engines and the SMs run side by
// side); with page-locked buffers (dcb_pack_reads / dcb_pinned_alloc) the step is bound by the host->device copy.
int dcb_decombine_batch(dcb_ctx* c, const dcb_packed* P, dcb_result* out, uint64_t* counters) {
    if (!c || !P) { dcb_set_error("dcb_decombine_batch: null argument"); return DCB_EINVAL; }
    CUDA_TRY(cudaSetDevice(c->device));
    int rc;
    if ((rc = prepare_batch(c, P))) return rc;
    const uint32_t n = (uint32_t)P->n_reads;
    const size_t sw = P->slot_words;
    cudaStream_t st[2] = {c->stream, c->stream2};
    if ((rc = reset_counter_sets(c, st[0]))) return rc;
    if ((rc = copy_side_arrays(c, P, st[0]))) return rc;
    if ((rc = fork_streams(c, st))) return rc;
    const uint32_t chunk = chunk_reads(kChunkReads, n);
    int k = 0;
    for (uint32_t first = 0; first < n; first += chunk, k++) {
        const uint32_t count = std::min<uint32_t>(chunk, n - first);
        cudaStream_t s = st[k & 1];
        CUDA_TRY(cudaMemcpyAsync((uint32_t*)c->words.p + (size_t)first * sw, P->words + (size_t)first * sw, (size_t)count * sw * 4,
                                 cudaMemcpyHostToDevice, s));
        if ((rc = run_chunk(c, s, first, count, k, out))) return rc;
    }
    return join_streams(c, st, true, counters);
}

// ---- ASCII in: pack on the device ----------------------------------------------------------------------------
// Geometry of an ASCII batch: what dcb_pack_reads derives on the host (slot width from the longest read).
static int ascii_geometry(const uint32_t* len, uint64_t n, uint32_t uniform_len, dcb_packed* G) {
    std::memset(G, 0, sizeof(*G));
    uint32_t max_len = uniform_len, min_len = uniform_len;
    if (!uniform_len && n) {
        if (!len) { dcb_set_error("read lengths missing"); return DCB_EINVAL; }
        max_len = 0; min_len = 0xFFFFFFFFu;
        for (uint64_t i = 0; i < n; i++) { max_len = std::max(max_len, len[i]); min_len = std::min(min_len, len[i]); }
    }
    if (max_len > DCB_MAX_READ_LEN) {
        dcb_set_error("read of %u nt exceeds the supported maximum of %d", max_len, DCB_MAX_READ_LEN);
        return DCB_EUNSUPPORTED;
    }
    G->n_reads = n; G->max_len = max_len;
    G->slot_words = std::max<uint32_t>(4u, ((max_len + 63) / 64) * 4);
    G->uniform_len = (n && min_len == max_len) ? max_len : 0;
    G->n_exc = 1;                       // unknown until packed: the kernels take the path that honours the exception list
    return DCB_OK;
}

// Host threads this process may use for packing / gathering: all of them, or its part when several ranks share the host
// (torchrun sets LOCAL_WORLD_SIZE).
static int local_world() {
    const char* e = std::getenv("LOCAL_WORLD_SIZE");
    const int w = e ? std::atoi(e) : 1;
    return w < 1 ? 1 : w;
}
static int host_threads() {
    const unsigned hw = std::thread::hardware_concurrency();
    const int t = (int)(hw ? hw : 4u) / local_world();
    return std::max(1, std::min(32, t));
}

// The scan that continues the exception index over the chunk's groups from where chunk chunk_no - 1 ends (ordered
// across the two streams by events).  Groups whose entries do not fit in the list lose their flag words (see
// dcb_pack_scan_kernel): the kernels of the chunk, which run before ascii_finish fails the call, read no entry past it.
static int scan_chunk(dcb_ctx* c, cudaStream_t s, uint32_t first, uint32_t groups, int chunk_no) {
    if (chunk_no > 0) CUDA_TRY(cudaStreamWaitEvent(s, c->ev_scan[(chunk_no - 1) & 1], 0));
    dcb_pack_scan_kernel<<<1, 1024, 0, s>>>((const uint32_t*)c->group_count.p, first >> 5, groups, c->exc_cap, (uint32_t*)c->exc_index.p,
                                            (uint32_t*)c->flags.p, c->d_exc_total);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaEventRecord(c->ev_scan[chunk_no & 1], s));
    return DCB_OK;
}

// Reads [first, first + count) packed by the host threads (dcb_pack_words) into hw, page-locked: the words, then (reads
// of varying length, len != NULL) the 16-bit lengths behind them.  1: packed, 0: not clean (a symbol beyond A / C / G / T,
// or no AVX2: the device packs the chunk), < 0: error.
static int pack_words_host(const char* ascii, const uint64_t* off, const uint32_t* len, uint32_t uniform_len, int revcomp,
                           uint32_t sw, uint64_t first, uint32_t count, int threads, uint32_t* hw) {
    int clean = 0;
    const int rc = dcb_pack_words(ascii, off, len, first, count, uniform_len, revcomp, sw, hw, threads, &clean);
    if (rc) return rc;
    if (!clean) return 0;
    if (len) {
        uint16_t* hl = reinterpret_cast<uint16_t*>(reinterpret_cast<char*>(hw) + (size_t)count * sw * 4);
        for (uint32_t i = 0; i < count; i++) hl[i] = (uint16_t)len[first + i];
    }
    return 1;
}

// A chunk pack_words_host packed, copied to its slots: a quarter of the text's bytes over the link.
static int copy_host_chunk(dcb_ctx* c, cudaStream_t s, const uint32_t* hw, bool with_lens, uint32_t first, uint32_t count) {
    const uint32_t sw = c->batch.slot_words;
    const size_t wbytes = (size_t)count * sw * 4;
    CUDA_TRY(cudaMemcpyAsync((uint32_t*)c->words.p + (size_t)first * sw, hw, wbytes, cudaMemcpyHostToDevice, s));
    if (with_lens)
        CUDA_TRY(cudaMemcpyAsync((uint16_t*)c->lens.p + first, reinterpret_cast<const char*>(hw) + wbytes, (size_t)count * 2, cudaMemcpyHostToDevice, s));
    return DCB_OK;
}

// A host-packed chunk has no exception list to merge: its groups join the running exception index with a count of zero.
static int index_host_chunk(dcb_ctx* c, cudaStream_t s, uint32_t first, uint32_t count, int chunk_no) {
    const uint32_t groups = (count + 31) / 32;
    CUDA_TRY(cudaMemsetAsync((uint32_t*)c->flags.p + (first >> 5), 0, (size_t)groups * 4, s));
    CUDA_TRY(cudaMemsetAsync((uint32_t*)c->group_count.p + (first >> 5), 0, (size_t)groups * 4, s));
    return scan_chunk(c, s, first, groups, chunk_no);
}

// The chunk packed by the host threads into the page-locked buffer of parity par, copied to its slots and indexed on
// stream s.  1: done, 0: not clean (the caller lets the device pack the chunk), < 0: error.
static int pack_chunk_host(dcb_ctx* c, cudaStream_t s, int par, const char* ascii, const uint64_t* off, const uint32_t* len,
                           uint32_t uniform_len, int revcomp, uint32_t first, uint32_t count, int chunk_no) {
    const uint32_t sw = c->batch.slot_words;
    const size_t wbytes = (size_t)count * sw * 4, lbytes = len ? (((size_t)count * 2 + 255) & ~(size_t)255) : 0;
    if (cudaEventSynchronize(c->ev_hw[par]) != cudaSuccess) { dcb_set_error("cudaEventSynchronize failed"); return DCB_ENOGPU; }
    if (c->hwords_cap[par] < wbytes + lbytes) {
        if (c->hwords[par]) cudaFreeHost(c->hwords[par]);
        c->hwords[par] = nullptr; c->hwords_cap[par] = 0;
        const size_t want = wbytes + lbytes + (wbytes + lbytes) / 8 + 4096;
        if (cudaHostAlloc((void**)&c->hwords[par], want, cudaHostAllocDefault) != cudaSuccess) { (void)cudaGetLastError(); return 0; }
        c->hwords_cap[par] = want;
    }
    int rc = pack_words_host(ascii, off, len, uniform_len, revcomp, sw, first, count, host_threads(), c->hwords[par]);
    if (rc != 1) return rc;
    if ((rc = copy_host_chunk(c, s, c->hwords[par], len != nullptr, first, count))) return rc;
    if ((rc = index_host_chunk(c, s, first, count, chunk_no))) return rc;
    CUDA_TRY(cudaEventRecord(c->ev_hw[par], s));
    return 1;
}

// Pack reads [first, first + count) on stream s (buffers of parity `par`): text bytes and offsets / lengths up, the pack
// kernel, the scan that continues the exception index, the exception entries.  The packed data lands in the context's
// batch buffers at the reads' global positions.
static int pack_chunk(dcb_ctx* c, cudaStream_t s, int par, const char* ascii, const uint64_t* off, const uint32_t* len,
                      uint32_t uniform_len, int revcomp, uint32_t first, uint32_t count, size_t exc_cap, int chunk_no,
                      bool staged = false) {
    if (!count) return DCB_OK;
    const uint32_t L = uniform_len;
    const bool contiguous = off == nullptr;
    const uint64_t lo = contiguous ? (uint64_t)first * L : off[first];
    uint64_t hi = lo;
    if (contiguous) hi = (uint64_t)(first + count) * L;
    else for (uint32_t i = first; i < first + count; i++) hi = std::max<uint64_t>(hi, off[i] + (len ? len[i] : L));
    if (!contiguous) for (uint32_t i = first; i < first + count; i++) if (off[i] < lo) { dcb_set_error("read offsets must not decrease inside a batch"); return DCB_EINVAL; }
    int rc;
    PackSrc src;
    src.stride = L; src.uniform_len = len ? 0u : L;
    src.first = first; src.count = count; src.off = nullptr; src.len = nullptr;
    if (staged) {
        // Pageable text: host threads GATHER the chunk's reads (the sequence lines only, not the headers and qualities
        // between them) into a page-locked buffer, back to back; the copy engine takes it from there at link speed while
        // the threads fill the other buffer.  Layout of the buffer: [local offsets (only when lengths vary)][text].
        CUDA_TRY(cudaEventSynchronize(c->ev_stage[par]));                      // the copy engine is done with this buffer
        const bool vary = len != nullptr;
        uint64_t total = 0;
        if (vary) for (uint32_t i = first; i < first + count; i++) total += len[i];
        else total = (uint64_t)count * L;
        const size_t head = vary ? (((size_t)count * 8 + 255) & ~(size_t)255) : 0;
        if (c->stage_cap[par] < head + total + 64) {
            if (c->stage[par]) cudaFreeHost(c->stage[par]);
            c->stage[par] = nullptr; c->stage_cap[par] = 0;
            const size_t want = head + total + (head + total) / 8 + 4096;
            CUDA_TRY(cudaHostAlloc((void**)&c->stage[par], want, cudaHostAllocDefault));
            c->stage_cap[par] = want;
        }
        uint64_t* loc = reinterpret_cast<uint64_t*>(c->stage[par]);
        char* dst = c->stage[par] + head;
        if (vary) { uint64_t at = 0; for (uint32_t i = 0; i < count; i++) { loc[i] = at; at += len[first + i]; } }
        const int nt = count < 8192 ? 1 : std::min(16, host_threads());
        auto work = [&](uint32_t a, uint32_t b) {
            for (uint32_t i = a; i < b; i++) {
                const uint32_t Li = vary ? len[first + i] : L;
                std::memcpy(dst + (vary ? loc[i] : (uint64_t)i * L), ascii + (contiguous ? (uint64_t)(first + i) * L : off[first + i]), Li);
            }
        };
        if (nt == 1) work(0, count);
        else {
            std::vector<std::thread> th;
            for (int t = 0; t < nt; t++) th.emplace_back(work, (uint32_t)((uint64_t)count * t / nt), (uint32_t)((uint64_t)count * (t + 1) / nt));
            for (auto& x : th) x.join();
        }
        if ((rc = c->text[par].ensure(total + 64))) return rc;
        CUDA_TRY(cudaMemcpyAsync(c->text[par].p, dst, total, cudaMemcpyHostToDevice, s));
        src.text = (const unsigned char*)c->text[par].p;
        src.text_lo = vary ? 0 : (uint64_t)first * L;                          // read i of the chunk at i * L (uniform) or loc[i]
        if (vary) {
            if ((rc = c->roff[par].ensure((size_t)count * 8 + 16))) return rc;
            CUDA_TRY(cudaMemcpyAsync(c->roff[par].p, loc, (size_t)count * 8, cudaMemcpyHostToDevice, s));
            src.off = (const uint64_t*)c->roff[par].p;
        }
        CUDA_TRY(cudaEventRecord(c->ev_stage[par], s));
    } else {
        if ((rc = c->text[par].ensure(hi - lo + 64))) return rc;
        CUDA_TRY(cudaMemcpyAsync(c->text[par].p, ascii + lo, hi - lo, cudaMemcpyHostToDevice, s));
        CUDA_TRY(cudaEventRecord(c->ev_text[par], s));
        c->text_pending[par] = true;
        src.text = (const unsigned char*)c->text[par].p; src.text_lo = lo;
        if (!contiguous) {
            if ((rc = c->roff[par].ensure((size_t)count * 8 + 16))) return rc;
            CUDA_TRY(cudaMemcpyAsync(c->roff[par].p, off + first, (size_t)count * 8, cudaMemcpyHostToDevice, s));
            src.off = (const uint64_t*)c->roff[par].p;
        }
    }
    if (len) {
        if ((rc = c->rlen[par].ensure((size_t)count * 4 + 16))) return rc;
        CUDA_TRY(cudaMemcpyAsync(c->rlen[par].p, len + first, (size_t)count * 4, cudaMemcpyHostToDevice, s));
        src.len = (const uint32_t*)c->rlen[par].p;
    }
    const uint32_t groups = (count + 31) / 32, blocks = (groups + 7) / 8;
    const uint32_t sw = c->batch.slot_words;
    dcb_pack_kernel<<<blocks, 256, 0, s>>>(src, revcomp, sw, (uint32_t*)c->words.p, (uint16_t*)c->lens.p, (uint32_t*)c->flags.p,
                                           (uint32_t*)c->group_count.p);
    CUDA_TRY(cudaGetLastError());
    if ((rc = scan_chunk(c, s, first, groups, chunk_no))) return rc;
    dcb_pack_exc_kernel<<<blocks, 256, 0, s>>>(src, revcomp, sw, (const uint32_t*)c->flags.p, (const uint32_t*)c->exc_index.p, (uint32_t)exc_cap,
                                               (uint32_t*)c->exc_read.p, (uint16_t*)c->exc_pos.p, (uint8_t*)c->exc_kind.p);
    CUDA_TRY(cudaGetLastError());
    return DCB_OK;
}

static size_t exc_capacity(uint64_t n) { return (size_t)std::min<uint64_t>(0xFFFFFFF0ull, 2 * n + (1u << 20)); }

static int ascii_begin(dcb_ctx* c, const char* ascii, const uint64_t* off, const uint32_t* len, uint64_t n, uint32_t uniform_len,
                       size_t* exc_cap) {
    if (!c || (n && !ascii)) { dcb_set_error("null argument"); return DCB_EINVAL; }
    if (!off && !uniform_len && n) { dcb_set_error("contiguous reads (off == NULL) need uniform_len"); return DCB_EINVAL; }
    CUDA_TRY(cudaSetDevice(c->device));
    dcb_packed G;
    int rc;
    if ((rc = ascii_geometry(uniform_len ? nullptr : len, n, uniform_len, &G))) return rc;
    *exc_cap = exc_capacity(n);
    c->exc_cap = (uint32_t)*exc_cap;
    if ((rc = prepare_batch(c, &G, *exc_cap))) return rc;
    if ((rc = c->group_count.ensure(((n + 31) / 32 + 2) * 4))) return rc;
    CUDA_TRY(cudaMemsetAsync(c->d_exc_total, 0, 16, c->stream));
    return DCB_OK;
}

// The exception list of a device-packed batch is complete: its length, against the capacity it was given.
static int ascii_finish(dcb_ctx* c, size_t exc_cap, uint32_t* n_exc) {
    uint32_t total = 0;
    CUDA_TRY(cudaMemcpy(&total, c->d_exc_total, 4, cudaMemcpyDeviceToHost));
    if (total > exc_cap) {
        dcb_set_error("device packing: %u non-ACGT symbols exceed the list capacity %zu (pack on the host with dcb_pack_reads)", total, exc_cap);
        return DCB_EUNSUPPORTED;
    }
    c->batch.n_exc = total;
    if (n_exc) *n_exc = total;
    return DCB_OK;
}

// Page-locked text, this process alone on its host: the chunks are shared from BOTH ENDS.  The calling thread gives the
// device the chunks from the front (the text crosses the link, dcb_pack_kernel packs it), never more than two text copies
// queued; meanwhile one worker packs chunks from the back with the host threads (dcb_pack_words) into a page-locked region.
// Each packed chunk is copied to its slots at once (a quarter of its text's bytes over the link, between the device's text
// copies); when the two meet, the host's chunks take their place in the exception index and run their kernels, in index
// order (the index runs on from chunk to chunk).  Neither side waits for the other until then, so the link never idles while a
// chunk is being packed and the shares settle at whatever the host's memory system allows.  A chunk in which the worker
// meets a symbol beyond A / C / G / T ends the host's share: the device packs that chunk and the worker claims no more.
// The region holds at most DCB_HOST_STAGE_MB (default 1024) of packed reads; the worker stops claiming when it is full.
static int ascii_two_ended(dcb_ctx* c, const char* ascii, const uint64_t* off, const uint32_t* lens, uint64_t n, uint32_t uniform_len,
                           int revcomp, dcb_result* out, uint32_t chunk, size_t exc_cap) {
    cudaStream_t st[2] = {c->stream, c->stream2};
    const int K = (int)((n + chunk - 1) / chunk);
    const uint32_t sw = c->batch.slot_words;
    const size_t slot_bytes = (((size_t)chunk * sw * 4 + (lens ? (size_t)chunk * 2 : 0)) + 255) & ~(size_t)255;
    size_t budget = (size_t)1024 << 20;
    if (const char* e = std::getenv("DCB_HOST_STAGE_MB")) budget = (size_t)std::max(0, std::atoi(e)) << 20;
    const int max_host = (int)std::min<size_t>((size_t)(K - 1), budget / slot_bytes);     // chunk 0 is the device's
    if (max_host > 0 && c->hstage_cap < (size_t)max_host * slot_bytes) {
        if (c->hstage) cudaFreeHost(c->hstage);
        c->hstage = nullptr; c->hstage_cap = 0;
        if (cudaHostAlloc((void**)&c->hstage, (size_t)max_host * slot_bytes, cudaHostAllocDefault) == cudaSuccess) c->hstage_cap = (size_t)max_host * slot_bytes;
        else (void)cudaGetLastError();
    }
    const int host_cap = c->hstage ? std::min<int>(max_host, (int)(c->hstage_cap / slot_bytes)) : 0;
    auto slot_of = [&](int k) { return reinterpret_cast<uint32_t*>(c->hstage + (size_t)(K - 1 - k) * slot_bytes); };
    auto first_of = [&](int k) { return (uint64_t)k * chunk; };
    auto count_of = [&](int k) { return (uint32_t)std::min<uint64_t>(chunk, n - (uint64_t)k * chunk); };

    std::mutex m;
    int dev_next = 0, host_lo = K;           // device owns [0, dev_next), host owns [host_lo, K); under m
    bool host_open = host_cap > 0;
    std::vector<char> dirty(K, 0);           // host chunks the worker could not pack (device packs them)
    int worker_rc = DCB_OK;
    if (!c->stream3 && cudaStreamCreateWithFlags(&c->stream3, cudaStreamNonBlocking) != cudaSuccess) { dcb_set_error("cudaStreamCreate failed"); return DCB_ENOGPU; }
    while ((int)c->ev_hcopy.size() < K) {
        cudaEvent_t e;
        CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        c->ev_hcopy.push_back(e);
    }
    CUDA_TRY(cudaStreamWaitEvent(c->stream3, c->ev_ready, 0));
    std::thread worker([&] {
        const int nt = std::max(1, host_threads() - 1);
        if (cudaSetDevice(c->device) != cudaSuccess) { std::lock_guard<std::mutex> g(m); worker_rc = DCB_ENOGPU; host_open = false; return; }
        for (;;) {
            int k;
            {
                std::lock_guard<std::mutex> g(m);
                if (!host_open || host_lo - 1 < dev_next || K - host_lo >= host_cap) { host_open = false; return; }
                k = --host_lo;
            }
            const uint32_t count = count_of(k);
            uint32_t* hw = slot_of(k);
            const int rc = pack_words_host(ascii, off, lens, uniform_len, revcomp, sw, first_of(k), count, nt, hw);
            if (rc != 1) {
                std::lock_guard<std::mutex> g(m);
                if (rc < 0) worker_rc = rc;
                dirty[k] = 1; host_open = false;
                return;
            }
            // the packed words go to their slots right away, between the device's text copies: only the chunk's place in
            // the exception index and its kernels have to wait for the chunks in front of it
            int crc = copy_host_chunk(c, c->stream3, hw, lens != nullptr, (uint32_t)first_of(k), count);
            if (!crc && cudaEventRecord(c->ev_hcopy[k], c->stream3) != cudaSuccess) { dcb_set_error("cudaEventRecord failed"); crc = DCB_ENOGPU; }
            if (crc) {
                std::lock_guard<std::mutex> g(m);
                worker_rc = crc; host_open = false;
                return;
            }
        }
    });
    struct Joiner {          // an early return: the worker claims nothing more and is waited for
        std::thread& t; std::mutex& m; bool& open;
        ~Joiner() { if (t.joinable()) { { std::lock_guard<std::mutex> g(m); open = false; } t.join(); } }
    } joiner{worker, m, host_open};

    int rc = DCB_OK;
    auto device_chunk = [&](int k) -> int {
        cudaStream_t s = st[k & 1];
        const uint32_t first = (uint32_t)first_of(k), count = count_of(k);
        int r;
        if ((r = pack_chunk(c, s, k & 1, ascii, off, lens, uniform_len, revcomp, first, count, exc_cap, k, false))) return r;
        c->device_chunks++;
        return run_chunk(c, s, first, count, k, out);
    };
    c->text_pending[0] = c->text_pending[1] = false;
    int k = 0;
    for (;; k++) {
        // at most two text copies queued: the one the copy engine works on and the next
        if (c->text_pending[k & 1]) {
            for (;;) {
                const cudaError_t q = cudaEventQuery(c->ev_text[k & 1]);
                if (q == cudaSuccess) break;
                if (q != cudaErrorNotReady) { dcb_set_error("cudaEventQuery failed: %s", cudaGetErrorString(q)); return DCB_ENOGPU; }
                std::this_thread::sleep_for(std::chrono::microseconds(20));
            }
        }
        {
            std::lock_guard<std::mutex> g(m);
            if (k >= host_lo) break;
            dev_next = k + 1;
        }
        if ((rc = device_chunk(k))) return rc;
    }
    worker.join();
    if (worker_rc) return worker_rc;
    for (; k < K; k++) {                    // the host's chunks, in index order
        if (dirty[k]) { if ((rc = device_chunk(k))) return rc; continue; }
        cudaStream_t s = st[k & 1];
        const uint32_t first = (uint32_t)first_of(k), count = count_of(k);
        CUDA_TRY(cudaStreamWaitEvent(s, c->ev_hcopy[k], 0));
        if ((rc = index_host_chunk(c, s, first, count, k))) return rc;
        c->host_chunks++;
        if ((rc = run_chunk(c, s, first, count, k, out))) return rc;
    }
    return DCB_OK;
}

int dcb_decombine_ascii(dcb_ctx* c, const char* ascii, const uint64_t* off, const uint32_t* len, uint64_t n, uint32_t uniform_len,
                        int revcomp, dcb_result* out, uint64_t* counters) {
    // Who packs a chunk: the device (the text goes over the link, 4 bytes per packed byte) or the host threads.  Text in
    // pageable memory would have to be gathered into page-locked staging by the host threads anyway: they pack it instead,
    // until a chunk holds a symbol beyond A / C / G / T.  Page-locked text: shared from both ends (ascii_two_ended) -- also
    // with several ranks on one host, each with its share of the host threads (LOCAL_WORLD_SIZE): measured on 2 ranks
    // 407 -> 528 M reads/s, on 8 ranks 655 -> 686 M (there the host's memory system bounds the copies of all eight links
    // and the packer takes 11 of 39 chunks).  DCB_HOST_SHARE=0: the device packs every chunk (measurements, tests).
    const char* hs = std::getenv("DCB_HOST_SHARE");
    if (hs && std::strcmp(hs, "0") && std::strcmp(hs, "1")) {
        dcb_set_error("DCB_HOST_SHARE=%s: accepted values are 1 (the default: chunks shared between the host threads and the "
                      "device) and 0 (the device packs every chunk)", hs);
        return DCB_EINVAL;
    }
    const bool host_share = !hs || hs[0] == '1';
    size_t exc_cap = 0;
    int rc;
    if ((rc = ascii_begin(c, ascii, off, len, n, uniform_len, &exc_cap))) return rc;
    const uint32_t* lens = uniform_len ? nullptr : len;
    cudaStream_t st[2] = {c->stream, c->stream2};
    if ((rc = reset_counter_sets(c, st[0]))) return rc;
    if ((rc = fork_streams(c, st))) return rc;
    // text in pageable memory (a memory-mapped file): smaller chunks through page-locked staging buffers
    bool staged = false;
    if (n) {
        cudaPointerAttributes attr;
        if (cudaPointerGetAttributes(&attr, ascii) != cudaSuccess) { (void)cudaGetLastError(); staged = true; }
        else staged = attr.type == cudaMemoryTypeUnregistered;
    }
    c->host_chunks = c->device_chunks = 0;
    bool shared = false;
    if (host_share && !staged && n) {
        // smaller chunks: the shares are settled chunk by chunk, and the two sides meet inside one
        uint32_t fine = kChunkReads / 4;
        if (const char* e = std::getenv("DCB_CHUNK_READS")) fine = (uint32_t)std::max(1024, std::atoi(e));
        fine = chunk_reads(fine, n);
        if ((n + fine - 1) / fine >= 4) {
            if ((rc = ascii_two_ended(c, ascii, off, lens, n, uniform_len, revcomp, out, fine, exc_cap))) {
                cudaStreamSynchronize(st[0]); cudaStreamSynchronize(st[1]);
                if (c->stream3) cudaStreamSynchronize(c->stream3);
                return rc;
            }
            shared = true;
        }
    }
    const uint32_t chunk = chunk_reads(staged ? kChunkReads / 2 : kChunkReads, n);
    bool host_ok = host_share && staged;
    int k = 0;
    for (uint64_t first = 0; first < n && !shared; first += chunk, k++) {
        const uint32_t count = (uint32_t)std::min<uint64_t>(chunk, n - first);
        cudaStream_t s = st[k & 1];
        if (host_ok) {
            if ((rc = pack_chunk_host(c, s, k & 1, ascii, off, lens, uniform_len, revcomp, (uint32_t)first, count, k)) < 0) return rc;
            host_ok = rc == 1;                          // not clean: the device packs this chunk and the rest
        }
        if (host_ok) c->host_chunks++;
        else {
            if ((rc = pack_chunk(c, s, k & 1, ascii, off, lens, uniform_len, revcomp, (uint32_t)first, count, exc_cap, k, staged))) return rc;
            c->device_chunks++;
        }
        if ((rc = run_chunk(c, s, (uint32_t)first, count, k, out))) return rc;
    }
    if ((rc = join_streams(c, st, true, counters))) return rc;
    return ascii_finish(c, exc_cap, nullptr);
}

// The device packer alone, its output copied back into a host dcb_packed (tests: bit-identical to dcb_pack_reads;
// tools: the pack kernels' device time through dcb_pack_device_ms).
int dcb_pack_device(dcb_ctx* c, const char* ascii, const uint64_t* off, const uint32_t* len, uint64_t n, uint32_t uniform_len,
                    int revcomp, dcb_packed** out) {
    if (!out) { dcb_set_error("dcb_pack_device: null argument"); return DCB_EINVAL; }
    size_t exc_cap = 0;
    int rc;
    if ((rc = ascii_begin(c, ascii, off, len, n, uniform_len, &exc_cap))) return rc;
    const uint32_t* lens = uniform_len ? nullptr : len;
    cudaStream_t st[2] = {c->stream, c->stream2};
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0)); CUDA_TRY(cudaEventCreate(&e1));
    if ((rc = fork_streams(c, st))) return rc;
    const uint32_t chunk = kChunkReads;
    int k = 0;
    CUDA_TRY(cudaEventRecord(e0, st[0]));
    for (uint64_t first = 0; first < n; first += chunk, k++)
        if ((rc = pack_chunk(c, st[k & 1], k & 1, ascii, off, lens, uniform_len, revcomp, (uint32_t)first,
                             (uint32_t)std::min<uint64_t>(chunk, n - first), exc_cap, k))) return rc;
    if ((rc = join_streams(c, st, false, nullptr))) return rc;
    CUDA_TRY(cudaEventRecord(e1, st[0]));
    CUDA_TRY(cudaStreamSynchronize(st[0]));
    float ms = 0.f;
    CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
    c->pack_ms = ms;
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    uint32_t n_exc = 0;
    if ((rc = ascii_finish(c, exc_cap, &n_exc))) return rc;
    // a host dcb_packed of the same shape (no reads packed on the host: n = 0 buffers would be too small, so pack a
    // batch of empty reads of the right count is not possible either) -- allocate through the host packer's owner
    dcb_packed* P = nullptr;
    if ((rc = dcb_packed_alloc(n, c->batch.slot_words, n_exc, &P))) return rc;
    P->uniform_len = c->batch.uniform_len; P->max_len = 0;
    if (n) {
        CUDA_TRY(cudaMemcpy(P->words, c->words.p, (size_t)n * c->batch.slot_words * 4, cudaMemcpyDeviceToHost));
        CUDA_TRY(cudaMemcpy(P->lens, c->lens.p, (size_t)n * 2, cudaMemcpyDeviceToHost));
        CUDA_TRY(cudaMemcpy(P->flags, c->flags.p, ((size_t)n + 31) / 32 * 4, cudaMemcpyDeviceToHost));
        for (uint64_t i = 0; i < n; i++) P->max_len = std::max<uint32_t>(P->max_len, P->lens[i]);
    }
    if (n_exc) {
        CUDA_TRY(cudaMemcpy(P->exc_read, c->exc_read.p, (size_t)n_exc * 4, cudaMemcpyDeviceToHost));
        CUDA_TRY(cudaMemcpy(P->exc_pos, c->exc_pos.p, (size_t)n_exc * 2, cudaMemcpyDeviceToHost));
        CUDA_TRY(cudaMemcpy(P->exc_kind, c->exc_kind.p, (size_t)n_exc, cudaMemcpyDeviceToHost));
    }
    *out = P;
    return DCB_OK;
}
int dcb_pack_device_ms(dcb_ctx* c, double* ms) {
    if (!c || !ms) return DCB_EINVAL;
    *ms = c->pack_ms;
    return DCB_OK;
}

void* dcb_pinned_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 16, cudaHostAllocDefault) != cudaSuccess) {
        dcb_set_error("dcb_pinned_alloc(%zu): %s", bytes, cudaGetErrorString(cudaGetLastError()));
        return nullptr;
    }
    return p;
}
void dcb_pinned_free(void* p) { if (p) cudaFreeHost(p); }

int dcb_timing_enable(dcb_ctx* c, int on) {
    if (!c) return DCB_EINVAL;
    if (on && !c->d_stamps) {   // zeroed before the first timed launch: the stamps are taken with atomicMax
        CUDA_TRY(cudaSetDevice(c->device));
        CUDA_TRY(cudaMalloc((void**)&c->d_stamps, kStamps * sizeof(TierStamp)));
        CUDA_TRY(cudaMemset(c->d_stamps, 0, kStamps * sizeof(TierStamp)));
        CUDA_TRY(cudaDeviceSynchronize());
    }
    c->timing = on != 0;
    return DCB_OK;
}
int dcb_timing_reset(dcb_ctx* c) {
    if (!c) return DCB_EINVAL;
    int rc = timing_collect(c);
    for (int i = 0; i < DCB_NTIMERS; i++) { c->ms[i] = 0; c->launches[i] = 0; }
    return rc;
}
int dcb_timing_get(dcb_ctx* c, double ms[DCB_NTIMERS], uint64_t launches[DCB_NTIMERS]) {
    if (!c) return DCB_EINVAL;
    int rc = timing_collect(c);
    for (int i = 0; i < DCB_NTIMERS; i++) { if (ms) ms[i] = c->ms[i]; if (launches) launches[i] = c->launches[i]; }
    return rc;
}
const char* dcb_exact_kernel_name(const dcb_ctx* c) {
    if (!c || !c->have_batch) return "";
    return c->q_fn ? "dcb_exact_kernel_flat" : c->spec_fn ? "dcb_exact_kernel_spec" : "dcb_exact_kernel";
}
static int sum_queue_counts(dcb_ctx* c, int which, uint64_t* total) {
    uint32_t q[kMaxChunks];
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    CUDA_TRY(cudaMemcpy(q, counter_set(c, c->set_last) + which * kMaxChunks, sizeof(q), cudaMemcpyDeviceToHost));
    *total = 0;
    for (int i = 0; i < kMaxChunks; i++) *total += q[i];
    return DCB_OK;
}
int dcb_last_deferred(dcb_ctx* c, uint64_t* n) {
    if (!c || !n || !c->ran) return DCB_EINVAL;
    if (c->params.force_general == 1) { *n = c->batch.n_reads; return DCB_OK; }
    return sum_queue_counts(c, 0, n);
}
int dcb_last_general(dcb_ctx* c, uint64_t* n) {
    if (!c || !n || !c->ran) return DCB_EINVAL;
    if (c->params.force_general == 1) { *n = c->batch.n_reads; return DCB_OK; }
    return sum_queue_counts(c, c->half_fn ? 1 : 0, n);
}
int dcb_last_pack_shares(dcb_ctx* c, uint32_t* host_chunks, uint32_t* device_chunks) {
    if (!c || !host_chunks || !device_chunks) { dcb_set_error("dcb_last_pack_shares: null argument"); return DCB_EINVAL; }
    *host_chunks = c->host_chunks; *device_chunks = c->device_chunks;
    return DCB_OK;
}

const char* dcb_halftag_kernel_name(const dcb_ctx* c) {
    return (c && c->have_batch && c->half_fn) ? "dcb_halftag_kernel" : "";
}

}  // extern "C"
