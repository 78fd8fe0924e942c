// collapse.cu -- the distance primitives of the collapse step on the GPU (sm_100a).
//
//   dcb_umi_pairs  all unordered pairs of UMIs within Levenshtein distance max_edits.  Replaces
//                  prsnn.symdel(umi_list, max_edits=bcthreshold, output_type="coo_matrix") + sparse.triu +
//                  sum_duplicates  (/root/reference/src/decombinator/collapse.py:735-742): output is the sorted
//                  list of (row, col), row < col, i.e. the COO entries in the order make_clusters walks them.
//   dcb_lev_leq    batch of are_seqs_equivalent(seq1, seq2, frac) verdicts (collapse.py:355-360):
//                  polyleven.levenshtein(a, b) <= len(shorter) * frac, compared in double like the reference.
//
// Both are integer-pipe bound (no tensor cores: nothing is a dense contraction).  The pair search has two forms:
//   * deletion neighbourhoods (what symdel does), for max_edits <= 2 and more than a few thousand UMIs: every UMI
//     emits its variants with up to max_edits symbols deleted (79 for a 12-symbol UMI), the (variant, UMI) entries
//     are radix-sorted by variant, and two UMIs within max_edits edits necessarily share a variant -- so only the
//     pairs inside a run of equal variants are verified (Hamming first, then the bit-parallel Levenshtein), appended
//     with a warp-aggregated atomic, sorted and made unique.  2 M random 12-mers: 158 M entries, ~8 G verifications,
//     instead of the 2 x 10^12 of an all-pairs sweep;
//   * a tiled all-pairs sweep for small lists (and max_edits > 2) -- tile of 256 UMIs staged in shared memory and
//     broadcast to 256 threads that each keep one UMI's match masks in registers -- with a pigeonhole prefilter in
//     front of the verifier.
// The output of both is the device radix sort of the 64-bit (row << 32 | col) keys.
#include "dcb_internal.h"
#include "lev_core.cuh"

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_select.cuh>
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#define CUDA_TRY(expr)                                                                          \
    do {                                                                                        \
        cudaError_t e__ = (expr);                                                               \
        if (e__ != cudaSuccess) {                                                               \
            dcb_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
            return DCB_ENOGPU;                                                                  \
        }                                                                                       \
    } while (0)

static constexpr int kPairTile = 256;

// grid.x enumerates the tile pairs (bi <= bj) of the upper triangle
__global__ void __launch_bounds__(kPairTile)
dcb_umi_pairs_kernel(const uint64_t* __restrict__ codes, uint32_t n, int k, uint32_t n_tiles,
                     unsigned long long* __restrict__ keys, unsigned long long cap, unsigned long long* __restrict__ count,
                     uint32_t part, uint32_t n_parts) {
    __shared__ uint64_t s_j[kPairTile];
    if (blockIdx.x % n_parts != part) return;            // a multi-GPU search: every GPU takes its share of the tile pairs
    // decode the linear block index into (bi, bj), bi <= bj: row bi of the triangle starts at bi*n_tiles - bi*(bi-1)/2
    unsigned long long lin = blockIdx.x;
    uint32_t bi = 0;
    {
        // largest bi with start(bi) <= lin, by a float estimate corrected with integer steps
        const double nt = (double)n_tiles;
        double est = nt + 0.5 - sqrt((nt + 0.5) * (nt + 0.5) - 2.0 * (double)lin);
        long long b = (long long)est;
        if (b < 0) b = 0;
        if (b >= (long long)n_tiles) b = n_tiles - 1;
        auto start = [&](long long x) { return (unsigned long long)x * n_tiles - (unsigned long long)(x * (x - 1) / 2); };
        while (b > 0 && start(b) > lin) b--;
        while (b + 1 < (long long)n_tiles && start(b + 1) <= lin) b++;
        bi = (uint32_t)b;
        lin -= start(b);
    }
    const uint32_t bj = bi + (uint32_t)lin;
    const uint32_t i = bi * kPairTile + threadIdx.x;
    const uint32_t j0 = bj * kPairTile;
    s_j[threadIdx.x] = (j0 + threadIdx.x < n) ? codes[j0 + threadIdx.x] : 0ull;
    __syncthreads();
    const bool live = i < n;
    const uint64_t ci = live ? codes[i] : 0ull;
    UmiPattern pat;
    umi_pattern(ci, pat);
    const uint32_t jn = min((uint32_t)kPairTile, n - j0);
    const int lane = threadIdx.x & 31;
    for (uint32_t t = 0; t < jn; t++) {
        const uint32_t j = j0 + t;
        const uint64_t cj = s_j[t];
        bool hit = live && j > i && umi_may_be_within(ci, cj, k);
        if (hit) hit = umi_distance(pat, cj) <= k;
        const unsigned m = __ballot_sync(0xFFFFFFFFu, hit);
        if (m) {
            const int leader = __ffs(m) - 1;
            unsigned long long base = 0;
            if (lane == leader) base = atomicAdd(count, (unsigned long long)__popc(m));
            base = __shfl_sync(0xFFFFFFFFu, base, leader);
            if (hit) {
                const unsigned long long slot = base + __popc(m & ((1u << lane) - 1u));
                if (slot < cap) keys[slot] = ((unsigned long long)i << 32) | j;
            }
        }
    }
}

// ---- deletion neighbourhoods ------------------------------------------------------------------------------------
// variants of a UMI of L symbols with up to d <= 2 deletions: 1 + L (+ L (L - 1) / 2)
__host__ __device__ __forceinline__ uint32_t umi_n_variants(int L, int d) {
    return 1u + (d >= 1 ? (uint32_t)L : 0u) + (d >= 2 ? (uint32_t)(L * (L - 1) / 2) : 0u);
}
__device__ __forceinline__ uint64_t umi_delete(uint64_t c, int p) {        // symbol p removed, length - 1
    const uint64_t body = c & ((1ull << 58) - 1ull);
    const uint64_t low = body & ((1ull << (3 * p)) - 1ull);
    const uint64_t high = (body >> (3 * (p + 1))) << (3 * p);
    return (low | high) | ((uint64_t)(umi_len(c) - 1) << 58);
}
// entry t of UMI i: variant t in the order (none), (p), (p < q)
__global__ void __launch_bounds__(256)
dcb_umi_variants_kernel(const uint64_t* __restrict__ codes, const uint64_t* __restrict__ first, uint32_t n, int d,
                        uint64_t* __restrict__ keys, uint32_t* __restrict__ ids) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint64_t c = codes[i];
    const int L = umi_len(c);
    uint64_t at = first[i];
    keys[at] = c; ids[at] = i; at++;
    if (d >= 1)
        for (int p = 0; p < L; p++) {
            const uint64_t c1 = umi_delete(c, p);
            keys[at] = c1; ids[at] = i; at++;
            if (d >= 2)
                for (int q = p; q < L - 1; q++) {      // second deletion at or behind p in the shortened code: original p < q + 1
                    keys[at] = umi_delete(c1, q); ids[at] = i; at++;
                }
        }
}
// Do two UMIs of EQUAL length share a variant with one deletion each (a - p == b - q)?  Then they agree on a prefix of
// p symbols and a suffix behind q, and between the two one is the other shifted by a symbol.  The longest common prefix
// and suffix give the smallest window that has to match under the shift.
__device__ __forceinline__ bool umi_share_one_deletion(uint64_t a, uint64_t b) {
    const int L = umi_len(a);
    const uint64_t body = (1ull << (3 * L)) - 1ull;
    const uint64_t x = (a ^ b) & body;
    if (!x) return true;
    const int pre = (__ffsll((long long)x) - 1) / 3;                 // symbols before the first difference
    const int suf = (__clzll((long long)x) - (64 - 3 * L)) / 3;      // symbols behind the last difference
    const int q = L - 1 - suf;                                       // last differing symbol
    if (q <= pre) return true;                                       // one substitution: delete it in both
    // a - pre == b - q  <=>  a[pre+1 .. q] == b[pre .. q-1];   or the mirror image
    const uint64_t win = ((1ull << (3 * (q - pre))) - 1ull) << (3 * pre);
    return ((((a >> 3) ^ b) & win) == 0ull) || ((((b >> 3) ^ a) & win) == 0ull);
}
// Block B owns entries [256 B, 256 B + 256) of the sorted (variant, UMI) list; thread t owns one entry and tests it
// against the entries BEHIND it in its run of equal variants.  The partners are staged tile by tile in shared memory
// (variant, UMI, code: the code gathered once per entry instead of once per pair), so the inner loop reads shared
// memory only.  A pair within max_edits edits is emitted from the run of a two-deletion variant only when the two UMIs
// share no one-deletion variant (they are then emitted from that run): without this rule a pair one substitution apart
// would be emitted 12 times for 12-symbol UMIs and the output would be 15 times the number of distinct pairs.
__global__ void __launch_bounds__(256)
dcb_umi_runs_kernel(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ ids, uint64_t n_entries,
                    const uint64_t* __restrict__ codes, int k, unsigned long long* __restrict__ out, unsigned long long cap,
                    unsigned long long* __restrict__ count, uint32_t part, uint32_t n_parts) {
    __shared__ uint64_t s_key[256], s_code[256];
    __shared__ uint32_t s_id[256];
    const int tid = threadIdx.x, lane = tid & 31;
    const uint64_t e = (uint64_t)blockIdx.x * 256 + tid;
    bool live = e < n_entries;
    const uint64_t key = live ? keys[e] : ~0ull;
    const uint32_t ia = live ? ids[e] : 0u;
    const uint64_t ca = live ? codes[ia] : 0ull;
    // Deleting either symbol of a repeat gives the same variant, so a UMI can be listed several times under one
    // variant.  The entries were generated in UMI order and the radix sort is stable: such copies are neighbours, and
    // every copy but the first is skipped, as owner and as partner.
    live = live && !(e > 0 && keys[e - 1] == key && ids[e - 1] == ia);
    // a multi-GPU search: the runs are dealt out by a hash of their variant (the verification is where the time goes)
    live = live && (n_parts == 1 || (uint32_t)((key * 0x9E3779B97F4A7C15ull) >> 40) % n_parts == part);
    const bool two_del = live && umi_len(key) + 2 == umi_len(ca);
    UmiPattern pat;
    bool have_pat = false;
    for (uint64_t tile = blockIdx.x; tile * 256 < n_entries; tile++) {
        const uint64_t base = tile * 256;
        __syncthreads();
        {
            const uint64_t f = base + tid;
            const bool in = f < n_entries;
            const uint64_t kf = in ? keys[f] : ~0ull - 1ull;
            const uint32_t id = in ? ids[f] : 0u;
            const bool copy = in && f > 0 && keys[f - 1] == kf && ids[f - 1] == id;
            s_key[tid] = kf;
            s_id[tid] = copy ? 0xFFFFFFFFu : id;             // a repeated listing of the UMI in front of it: no partner
            s_code[tid] = in ? codes[id] : 0ull;
        }
        __syncthreads();
        const bool need = live && (tile == blockIdx.x || s_key[0] == key);      // sorted: my run reaches this tile or it does not
        if (!__syncthreads_or(need)) break;
        int j = tile == blockIdx.x ? tid + 1 : 0;
        bool more = need && j < 256 && s_key[j] == key;
        while (__any_sync(0xFFFFFFFFu, more)) {
            bool hit = false;
            uint32_t ib = 0;
            if (more) {
                ib = s_id[j];
                const uint64_t cb = s_code[j];
                if (ib != ia && ib != 0xFFFFFFFFu) {
                    const bool same_len = umi_len(ca) == umi_len(cb);
                    if (same_len) {          // Hamming distance <= k settles it at once
                        const uint64_t x = (ca ^ cb) & ((1ull << 58) - 1ull);
                        hit = __popcll((x | (x >> 1) | (x >> 2)) & 0x0249249249249249ull) <= k;
                    }
                    if (!hit && umi_may_be_within(ca, cb, k)) {
                        if (!have_pat) { umi_pattern(ca, pat); have_pat = true; }
                        hit = umi_distance(pat, cb) <= k;
                    }
                    if (hit && two_del && same_len && umi_share_one_deletion(ca, cb)) hit = false;   // emitted from that run
                }
                j++;
                more = j < 256 && s_key[j] == key;
            }
            const unsigned m = __ballot_sync(0xFFFFFFFFu, hit);
            if (m) {
                const int leader = __ffs(m) - 1;
                unsigned long long at = 0;
                if (lane == leader) at = atomicAdd(count, (unsigned long long)__popc(m));
                at = __shfl_sync(0xFFFFFFFFu, at, leader);
                if (hit) {
                    const unsigned long long slot = at + __popc(m & ((1u << lane) - 1u));
                    if (slot < cap) out[slot] = ia < ib ? (((unsigned long long)ia << 32) | ib) : (((unsigned long long)ib << 32) | ia);
                }
            }
        }
    }
}

// DCB_UMI_TRACE=1: phase times of the pair search on stderr (tuning aid; synchronises the stream at every mark)
struct PhaseTrace {
    bool on; cudaStream_t s; cudaEvent_t last = nullptr;
    PhaseTrace(cudaStream_t st) : on(std::getenv("DCB_UMI_TRACE") != nullptr), s(st) { if (on) { cudaEventCreate(&last); cudaEventRecord(last, s); } }
    ~PhaseTrace() { if (last) cudaEventDestroy(last); }
    void mark(const char* what, double count = 0) {
        if (!on) return;
        cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, s); cudaEventSynchronize(e);
        float ms = 0.f; cudaEventElapsedTime(&ms, last, e);
        std::fprintf(stderr, "[umi_pairs] %-28s %9.3f ms  %.4g\n", what, ms, count);
        cudaEventDestroy(last); last = e;
    }
};

// device memory that is released on every way out of a function
struct DevMem {
    void* p = nullptr;
    ~DevMem() { if (p) cudaFree(p); }
    cudaError_t alloc(size_t bytes) { if (p) { cudaFree(p); p = nullptr; } return cudaMalloc(&p, bytes ? bytes : 16); }
    template <class T> T* as() { return static_cast<T*>(p); }
    void* release() { void* q = p; p = nullptr; return q; }
};
struct Events {
    cudaEvent_t a = nullptr, b = nullptr;
    ~Events() { if (a) cudaEventDestroy(a); if (b) cudaEventDestroy(b); }
};

// one thread per pair; the shorter sequence is the pattern.  NP: code bits per symbol (3: codes 0..7; 8: any byte)
template <int W, int NP>
__device__ __forceinline__ int lev_pair(const uint8_t* pa, int la, const uint8_t* pb, int lb) {
    SeqPattern<W, NP> pat;
    seq_pattern<W, NP>(pa, la, pat);
    return seq_distance<W, NP>(pat, pb, lb);
}

template <int NP>
__global__ void __launch_bounds__(128)
dcb_lev_leq_kernel(const uint8_t* __restrict__ sym, const uint64_t* __restrict__ off, const uint32_t* __restrict__ len,
                   const uint32_t* __restrict__ a, const uint32_t* __restrict__ b, unsigned long long n_pairs, uint32_t n_seqs,
                   double frac, uint8_t* __restrict__ verdict, uint32_t* __restrict__ flag) {
    const unsigned long long t = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_pairs) return;
    uint32_t ia = a[t], ib = b[t];
    if (ia >= n_seqs || ib >= n_seqs) { flag[0] = 1u; flag[1] = (uint32_t)t; verdict[t] = 0; return; }
    if (NP < 8) {   // symbol codes are NP bits wide
        uint32_t any = 0;
        for (uint32_t k = 0; k < len[ia]; k++) any |= sym[off[ia] + k];
        for (uint32_t k = 0; k < len[ib]; k++) any |= sym[off[ib] + k];
        if (any >> NP) { flag[2] = 1u; flag[3] = (uint32_t)t; verdict[t] = 0; return; }
    }
    int la = (int)len[ia], lb = (int)len[ib];
    if (la > lb) { const uint32_t x = ia; ia = ib; ib = x; const int y = la; la = lb; lb = y; }
    const uint8_t* pa = sym + off[ia];
    const uint8_t* pb = sym + off[ib];
    int d;
    if (la <= 64) d = lev_pair<1, NP>(pa, la, pb, lb);
    else if (la <= 128) d = lev_pair<2, NP>(pa, la, pb, lb);
    else if (la <= 192) d = lev_pair<3, NP>(pa, la, pb, lb);
    else if (la <= 256) d = lev_pair<4, NP>(pa, la, pb, lb);
    else d = lev_pair<8, NP>(pa, la, pb, lb);
    // threshold = len(min(seq1, seq2, key=len)) * lev_threshold_fraction ; return distance <= threshold  (collapse.py:359-360)
    verdict[t] = ((double)d <= (double)la * frac) ? 1 : 0;
}

// ---- barcode extraction (SURVEY 8(f) row 3) ------------------------------------------------------------------------
// One thread per decombined row: the barcode region (R2[:bclength], field 8 of an .n12 row) and its quality string.
// What collapse.py does per row before any grouping (get_barcode_positions, collapse.py:367-479): an 'N' anywhere rejects
// the row (unless -N); spacer 1 is searched in its window bc[lo:hi] and must be found exactly once (regex.findall:
// leftmost, non-overlapping).  Then, per layout of the ligation oligo:
//   two spacers (M13, I8): window bc[0 : 10 + len(spacer1)]; spacer 2 is searched in bc[len(spacer1):] and must be found
//     exactly once; N1 lies between the spacers, N2 is the six bases behind spacer 2;
//   N1, spacer, N2 (I8_single): window bc[0:18]; N1 is bc[0 : spacer position], N2 the six bases behind the spacer;
//     for both: N1 of <= 3 or >= 9 bases and an N2 that runs past the end reject the row, and set_barcode (:281-326)
//     makes N1 + N2, a short N1 padded with 'S' (quality '?'), a long one cut to five bases + 'L';
//   fixed barcode (NEBIO: window bc[18:28], barcode bc[0:17]; TAKARA: window bc[0:19], barcode bc[0:12]): the spacer only
//     has to be there, its position is not used.
// check_umi_quality (:340-352): more than `max_below` barcode qualities under `min_q`, or a mean under `avg_q`, rejects the row.
// Only the EXACT spacer search is done here.  The reference escalates to fuzzy regular expressions ({1s<=2}, then
// {2i+2d+1s<=2}) when an exact search finds nothing: such rows (a few percent) come back as DCB_BC_HOST and the host
// runs the reference's own search on them; so do rows with symbols outside ACGTN, a quality string of another length, a
// region longer than 250, and fixed-barcode regions shorter than the barcode (the reference would cut the barcode short).
__device__ __forceinline__ int bc_find(const unsigned char* s, int from, int to, const char* pat, int plen) {   // first match in [from, to)
    for (int p = from; p + plen <= to; p++) {
        int k = 0;
        while (k < plen && s[p + k] == (unsigned char)pat[k]) k++;
        if (k == plen) return p;
    }
    return -1;
}
__device__ __forceinline__ int bc_count(const unsigned char* s, int from, int to, const char* pat, int plen, int& first) {
    int n = 0;
    first = -1;
    for (int p = bc_find(s, from, to, pat, plen); p >= 0; p = bc_find(s, p + plen, to, pat, plen)) { if (!n) first = p; n++; }
    return n;
}
enum { BC_TWO_SPACERS = 0, BC_N1_SPACER_N2 = 1, BC_FIXED = 2 };   // BcParams::layout
struct BcParams { char sp1[32], sp2[32]; int layout, lo, hi, bclen, len1, len2, allow_ns, min_q, max_below; double avg_q; };

__global__ void __launch_bounds__(128)
dcb_barcodes_kernel(const unsigned char* __restrict__ bc, const unsigned char* __restrict__ qual, const uint64_t* __restrict__ bc_off,
                    const uint32_t* __restrict__ bc_len, const uint64_t* __restrict__ q_off, const uint32_t* __restrict__ q_len,
                    uint64_t n, BcParams P, uint8_t* __restrict__ status, uint8_t* __restrict__ n1len, uint64_t* __restrict__ code) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const unsigned char* s = bc + bc_off[i];
    const unsigned char* q = qual + q_off[i];
    const int L = (int)bc_len[i];
    status[i] = DCB_BC_HOST; n1len[i] = 0; code[i] = 0;
    if (L > 250 || (int)q_len[i] != L) return;
    bool has_n = false, odd = false;
    for (int p = 0; p < L; p++) {
        const unsigned char c = s[p];
        has_n |= c == 'N';
        odd |= !(c == 'A' || c == 'C' || c == 'G' || c == 'T' || c == 'N');
    }
    if (has_n && !P.allow_ns) { status[i] = DCB_BC_FAIL_N; return; }                        // collapse.py:388-392
    if (odd || (P.layout == BC_FIXED && L < P.bclen)) return;
    int w0, w1;
    const int hi = L < P.hi ? L : P.hi;
    const int c1 = bc_count(s, P.lo, hi, P.sp1, P.len1, w0);                                // :405-413
    if (c1 == 0) return;                                                                    // the fuzzy searches decide
    if (c1 != 1) { status[i] = DCB_BC_FAIL_NOSPACER; return; }
    // the barcode symbols (A C G T N S L = 0..6) and their qualities
    uint64_t cd = (uint64_t)P.bclen << 58;
    int qsum = 0, qn = 0, below = 0, k = 0;
    auto sym = [](unsigned char c) -> uint64_t { return c == 'A' ? 0 : c == 'C' ? 1 : c == 'G' ? 2 : c == 'T' ? 3 : 4; };
    auto addq = [&](int v) { qsum += v; qn++; below += v < P.min_q; };
    if (P.layout == BC_FIXED) {                                                             // set_barcode: bc[0:bclen], q[0:bclen]
        for (; k < P.bclen; k++) { cd |= sym(s[k]) << (3 * k); addq((int)q[k] - 33); }
    } else {
        int b1s = 0, b1e = w0, b2s = w0 + P.len1;                                           // I8_single: N1, spacer, N2
        if (P.layout == BC_TWO_SPACERS) {
            const int c2 = bc_count(s, P.len1, L, P.sp2, P.len2, w1);                       // :417-422
            if (c2 == 0) return;
            if (c2 != 1) { status[i] = DCB_BC_FAIL_NOT2; return; }
            b1s = w0 + P.len1; b1e = w1; b2s = w1 + P.len2;
        }
        const int b2e = b2s + 6, n1 = b1e - b1s;
        if (n1 <= 3) { status[i] = DCB_BC_FAIL_N1SHORT; return; }                           // :241-254
        if (n1 >= 9) { status[i] = DCB_BC_FAIL_N1LONG; return; }
        if (b2e > L) { status[i] = DCB_BC_FAIL_N2END; return; }
        n1len[i] = (uint8_t)n1;
        // 12 symbols; a long N1 has no pad quality (11 values)
        const int take1 = n1 > 6 ? 5 : n1;
        for (int p = 0; p < take1; p++, k++) { cd |= sym(s[b1s + p]) << (3 * k); addq((int)q[b1s + p] - 33); }
        if (n1 < 6) for (int p = n1; p < 6; p++, k++) { cd |= 5ull << (3 * k); addq('?' - 33); }   // 'S', quality '?'
        if (n1 > 6) { cd |= 6ull << (3 * k); k++; }                                               // 'L'; "?" * (6 - n1) is empty
        for (int p = 0; p < 6; p++, k++) { cd |= sym(s[b2s + p]) << (3 * k); addq((int)q[b2s + p] - 33); }
    }
    code[i] = cd;
    const bool bad_q = below > P.max_below || (double)qsum / (double)qn < P.avg_q;            // :350-352
    status[i] = bad_q ? DCB_BC_FAIL_QUALITY : DCB_BC_OK;
}

struct GrowBuf {            // grow-only device buffer kept between calls (dcb_lev_leq is called once per grouping round)
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        const size_t want = bytes + bytes / 4 + 4096;
        const cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};
struct dcb_dist {
    int device = 0;
    cudaStream_t stream = nullptr;
    unsigned long long* d_keys = nullptr;      // sorted pair keys of the last dcb_umi_pairs
    unsigned long long n_keys = 0;
    double last_ms = 0.0;
    GrowBuf sym, off, len, a, b, ver, flag;   // dcb_lev_leq
    const char* last_method = "";
};

extern "C" {

dcb_dist* dcb_dist_create(int device) {
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0) {
        (void)cudaGetLastError();
        dcb_set_error("dcb_dist_create: no CUDA device available (there is no CPU fallback)");
        return nullptr;
    }
    if (device < 0 || device >= n_dev || cudaSetDevice(device) != cudaSuccess) {
        dcb_set_error("dcb_dist_create: device %d not usable", device);
        return nullptr;
    }
    dcb_dist* d = new dcb_dist();
    d->device = device;
    if (cudaStreamCreateWithFlags(&d->stream, cudaStreamNonBlocking) != cudaSuccess) {
        dcb_set_error("dcb_dist_create: cudaStreamCreate failed");
        delete d;
        return nullptr;
    }
    return d;
}

void dcb_dist_destroy(dcb_dist* d) {
    if (!d) return;
    cudaSetDevice(d->device);
    if (d->stream) { cudaStreamSynchronize(d->stream); cudaStreamDestroy(d->stream); }
    cudaFree(d->d_keys);
    d->sym.release(); d->off.release(); d->len.release(); d->a.release(); d->b.release(); d->ver.release(); d->flag.release();
    delete d;
}

int dcb_umi_pairs(dcb_dist* d, const uint64_t* codes, uint32_t n, int max_edits, uint64_t* keys, uint64_t cap,
                  uint64_t* n_pairs) {
    return dcb_umi_pairs_part(d, codes, n, max_edits, 0, 1, keys, cap, n_pairs);
}

int dcb_umi_pairs_part(dcb_dist* d, const uint64_t* codes, uint32_t n, int max_edits, uint32_t part, uint32_t n_parts,
                       uint64_t* keys, uint64_t cap, uint64_t* n_pairs) {
    if (!d || !n_pairs) { dcb_set_error("dcb_umi_pairs: null argument"); return DCB_EINVAL; }
    if (n_parts == 0 || part >= n_parts) { dcb_set_error("dcb_umi_pairs_part: part %u of %u", part, n_parts); return DCB_EINVAL; }
    CUDA_TRY(cudaSetDevice(d->device));
    cudaStream_t s = d->stream;
    if (codes) {   // compute (and cache) the sorted pair list
        if (max_edits < 0 || max_edits > DCB_UMI_MAX_LEN) { dcb_set_error("dcb_umi_pairs: max_edits out of range"); return DCB_EINVAL; }
        for (uint32_t i = 0; i < n; i++)
            if ((codes[i] >> 58) > DCB_UMI_MAX_LEN) { dcb_set_error("dcb_umi_pairs: UMI %u longer than %d symbols", i, DCB_UMI_MAX_LEN); return DCB_EUNSUPPORTED; }
        cudaFree(d->d_keys); d->d_keys = nullptr; d->n_keys = 0;
        *n_pairs = 0;
        if (n < 2) return DCB_OK;
        DevMem d_codes, d_count, d_raw;
        Events ev;
        CUDA_TRY(d_codes.alloc((size_t)n * 8));
        CUDA_TRY(d_count.alloc(8));
        CUDA_TRY(cudaMemcpyAsync(d_codes.p, codes, (size_t)n * 8, cudaMemcpyHostToDevice, s));
        CUDA_TRY(cudaEventCreate(&ev.a)); CUDA_TRY(cudaEventCreate(&ev.b));
        unsigned long long found = 0;
        // which form: deletion neighbourhoods for long lists (DCB_UMI_SYMDEL_MIN overrides the switch-over, for tests)
        uint32_t symdel_min = 4096;
        if (const char* e = std::getenv("DCB_UMI_SYMDEL_MIN")) symdel_min = (uint32_t)std::strtoul(e, nullptr, 10);
        const bool symdel = max_edits >= 1 && max_edits <= 2 && n >= symdel_min;
        d->last_method = symdel ? "deletion neighbourhoods" : "all pairs";
        if (symdel) {
            std::vector<uint64_t> first((size_t)n + 1);
            uint64_t total = 0;
            for (uint32_t i = 0; i < n; i++) { first[i] = total; total += umi_n_variants((int)(codes[i] >> 58), max_edits); }
            first[n] = total;
            DevMem d_first, k_in, k_out, v_in, v_out, d_tmp;
            CUDA_TRY(d_first.alloc(((size_t)n + 1) * 8));
            CUDA_TRY(k_in.alloc(total * 8)); CUDA_TRY(k_out.alloc(total * 8));
            CUDA_TRY(v_in.alloc(total * 4)); CUDA_TRY(v_out.alloc(total * 4));
            CUDA_TRY(cudaMemcpyAsync(d_first.p, first.data(), ((size_t)n + 1) * 8, cudaMemcpyHostToDevice, s));
            CUDA_TRY(cudaEventRecord(ev.a, s));
            PhaseTrace tr(s);
            dcb_umi_variants_kernel<<<(n + 255) / 256, 256, 0, s>>>(d_codes.as<uint64_t>(), d_first.as<uint64_t>(), n, max_edits,
                                                                    k_in.as<uint64_t>(), v_in.as<uint32_t>());
            CUDA_TRY(cudaGetLastError());
            tr.mark("variants", (double)total);
            size_t tmp_bytes = 0;
            CUDA_TRY(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, k_in.as<uint64_t>(), k_out.as<uint64_t>(), v_in.as<uint32_t>(),
                                                     v_out.as<uint32_t>(), (size_t)total, 0, 64, s));
            CUDA_TRY(d_tmp.alloc(tmp_bytes));
            CUDA_TRY(cub::DeviceRadixSort::SortPairs(d_tmp.p, tmp_bytes, k_in.as<uint64_t>(), k_out.as<uint64_t>(), v_in.as<uint32_t>(),
                                                     v_out.as<uint32_t>(), (size_t)total, 0, 64, s));
            tr.mark("sort entries", (double)total);
            unsigned long long capacity = std::max<unsigned long long>(1ull << 22, 96ull * n);
            for (int attempt = 0; attempt < 2; attempt++) {
                CUDA_TRY(d_raw.alloc(capacity * 8));
                CUDA_TRY(cudaMemsetAsync(d_count.p, 0, 8, s));
                dcb_umi_runs_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(k_out.as<uint64_t>(), v_out.as<uint32_t>(), total,
                                                                                   d_codes.as<uint64_t>(), max_edits,
                                                                                   d_raw.as<unsigned long long>(), capacity,
                                                                                   d_count.as<unsigned long long>(), part, n_parts);
                CUDA_TRY(cudaGetLastError());
                CUDA_TRY(cudaMemcpyAsync(&found, d_count.p, 8, cudaMemcpyDeviceToHost, s));
                CUDA_TRY(cudaStreamSynchronize(s));
                tr.mark("verify runs", (double)found);
                if (found <= capacity) break;
                capacity = found;                  // the list did not fit: size it exactly and walk the runs again
            }
            // a pair turns up once per variant its two UMIs share: sort, then keep one of each
            if (found) {
                DevMem d_sorted, d_uniq, d_nsel, d_tmp2;
                CUDA_TRY(d_sorted.alloc(found * 8));
                size_t tb = 0;
                CUDA_TRY(cub::DeviceRadixSort::SortKeys(nullptr, tb, d_raw.as<unsigned long long>(), d_sorted.as<unsigned long long>(), (size_t)found, 0, 64, s));
                CUDA_TRY(d_tmp2.alloc(tb));
                CUDA_TRY(cub::DeviceRadixSort::SortKeys(d_tmp2.p, tb, d_raw.as<unsigned long long>(), d_sorted.as<unsigned long long>(), (size_t)found, 0, 64, s));
                CUDA_TRY(d_uniq.alloc(found * 8));
                CUDA_TRY(d_nsel.alloc(8));
                size_t tb2 = 0;
                CUDA_TRY(cub::DeviceSelect::Unique(nullptr, tb2, d_sorted.as<unsigned long long>(), d_uniq.as<unsigned long long>(), d_nsel.as<unsigned long long>(), (size_t)found, s));
                if (tb2 > tb) CUDA_TRY(d_tmp2.alloc(tb2));
                CUDA_TRY(cub::DeviceSelect::Unique(d_tmp2.p, tb2, d_sorted.as<unsigned long long>(), d_uniq.as<unsigned long long>(), d_nsel.as<unsigned long long>(), (size_t)found, s));
                tr.mark("sort + unique pairs", (double)found);
                CUDA_TRY(cudaEventRecord(ev.b, s));
                unsigned long long nu = 0;
                CUDA_TRY(cudaMemcpyAsync(&nu, d_nsel.p, 8, cudaMemcpyDeviceToHost, s));
                CUDA_TRY(cudaStreamSynchronize(s));
                d->d_keys = (unsigned long long*)d_uniq.release();
                found = nu;
            } else {
                CUDA_TRY(cudaEventRecord(ev.b, s));
                CUDA_TRY(cudaStreamSynchronize(s));
            }
        } else {
            const uint32_t n_tiles = (n + kPairTile - 1) / kPairTile;
            const unsigned long long n_blocks = (unsigned long long)n_tiles * (n_tiles + 1) / 2;
            if (n_blocks > 0x7FFFFFFFull) { dcb_set_error("dcb_umi_pairs: too many UMIs for an all-pairs sweep (%u)", n); return DCB_EUNSUPPORTED; }
            unsigned long long capacity = std::max<unsigned long long>(1ull << 20, 8ull * n);
            for (int attempt = 0; attempt < 2; attempt++) {
                CUDA_TRY(d_raw.alloc(capacity * 8));
                CUDA_TRY(cudaMemsetAsync(d_count.p, 0, 8, s));
                CUDA_TRY(cudaEventRecord(ev.a, s));
                dcb_umi_pairs_kernel<<<(unsigned)n_blocks, kPairTile, 0, s>>>(d_codes.as<uint64_t>(), n, max_edits, n_tiles,
                                                                              d_raw.as<unsigned long long>(), capacity,
                                                                              d_count.as<unsigned long long>(), part, n_parts);
                CUDA_TRY(cudaGetLastError());
                CUDA_TRY(cudaEventRecord(ev.b, s));
                CUDA_TRY(cudaMemcpyAsync(&found, d_count.p, 8, cudaMemcpyDeviceToHost, s));
                CUDA_TRY(cudaStreamSynchronize(s));
                if (found <= capacity) break;
                capacity = found;      // the list did not fit: size it exactly and sweep again
            }
            if (found) {
                DevMem d_sorted, d_tmp;
                CUDA_TRY(d_sorted.alloc(found * 8));
                size_t tmp_bytes = 0;
                CUDA_TRY(cub::DeviceRadixSort::SortKeys(nullptr, tmp_bytes, d_raw.as<unsigned long long>(), d_sorted.as<unsigned long long>(), (size_t)found, 0, 64, s));
                CUDA_TRY(d_tmp.alloc(tmp_bytes));
                CUDA_TRY(cub::DeviceRadixSort::SortKeys(d_tmp.p, tmp_bytes, d_raw.as<unsigned long long>(), d_sorted.as<unsigned long long>(), (size_t)found, 0, 64, s));
                CUDA_TRY(cudaStreamSynchronize(s));
                d->d_keys = (unsigned long long*)d_sorted.release();
            }
        }
        float ms = 0.f;
        cudaEventElapsedTime(&ms, ev.a, ev.b);
        d->last_ms = ms;
        d->n_keys = found;
    }
    *n_pairs = d->n_keys;
    if (keys) {
        if (cap < d->n_keys) { dcb_set_error("dcb_umi_pairs: output holds %llu pairs, %llu needed", (unsigned long long)cap, d->n_keys); return DCB_ENOMEM; }
        if (d->n_keys) {
            CUDA_TRY(cudaMemcpyAsync(keys, d->d_keys, d->n_keys * 8, cudaMemcpyDeviceToHost, s));
            CUDA_TRY(cudaStreamSynchronize(s));
        }
    }
    return DCB_OK;
}

static int lev_leq_impl(dcb_dist* d, const uint8_t* symbols, const uint64_t* off, const uint32_t* len, uint32_t n_seqs,
                        const uint32_t* a, const uint32_t* b, uint64_t n_pairs, double frac, uint8_t* verdict, bool bytes);

int dcb_lev_leq(dcb_dist* d, const uint8_t* symbols, const uint64_t* off, const uint32_t* len, uint32_t n_seqs,
                const uint32_t* a, const uint32_t* b, uint64_t n_pairs, double frac, uint8_t* verdict) {
    return lev_leq_impl(d, symbols, off, len, n_seqs, a, b, n_pairs, frac, verdict, false);
}
int dcb_lev_leq_bytes(dcb_dist* d, const uint8_t* symbols, const uint64_t* off, const uint32_t* len, uint32_t n_seqs,
                      const uint32_t* a, const uint32_t* b, uint64_t n_pairs, double frac, uint8_t* verdict) {
    return lev_leq_impl(d, symbols, off, len, n_seqs, a, b, n_pairs, frac, verdict, true);
}

static int lev_leq_impl(dcb_dist* d, const uint8_t* symbols, const uint64_t* off, const uint32_t* len, uint32_t n_seqs,
                        const uint32_t* a, const uint32_t* b, uint64_t n_pairs, double frac, uint8_t* verdict, bool bytes) {
    if (!d || (n_pairs && (!symbols || !off || !len || !a || !b || !verdict))) { dcb_set_error("dcb_lev_leq: null argument"); return DCB_EINVAL; }
    if (n_pairs == 0) return DCB_OK;
    CUDA_TRY(cudaSetDevice(d->device));
    cudaStream_t s = d->stream;
    uint64_t total = 0;
    for (uint32_t i = 0; i < n_seqs; i++) {
        if (len[i] > 512) { dcb_set_error("dcb_lev_leq: sequence %u has %u symbols (limit 512)", i, len[i]); return DCB_EUNSUPPORTED; }
        total = std::max<uint64_t>(total, off[i] + len[i]);
    }
    // buffers are kept between calls (the grouping of read_in_data calls this once per round); symbol codes and pair
    // indices are checked by the kernel itself (a flag comes back), not by host loops over every symbol and pair
    CUDA_TRY(d->sym.ensure(total + 16)); CUDA_TRY(d->off.ensure((size_t)n_seqs * 8)); CUDA_TRY(d->len.ensure((size_t)n_seqs * 4));
    CUDA_TRY(d->a.ensure(n_pairs * 4)); CUDA_TRY(d->b.ensure(n_pairs * 4)); CUDA_TRY(d->ver.ensure(n_pairs)); CUDA_TRY(d->flag.ensure(16));
    CUDA_TRY(cudaMemsetAsync(d->flag.p, 0, 16, s));
    CUDA_TRY(cudaMemcpyAsync(d->sym.p, symbols, total, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(d->off.p, off, (size_t)n_seqs * 8, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(d->len.p, len, (size_t)n_seqs * 4, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(d->a.p, a, n_pairs * 4, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(d->b.p, b, n_pairs * 4, cudaMemcpyHostToDevice, s));
    const unsigned long long blocks = (n_pairs + 127) / 128;
    Events ev;
    CUDA_TRY(cudaEventCreate(&ev.a));
    CUDA_TRY(cudaEventCreate(&ev.b));
    CUDA_TRY(cudaEventRecord(ev.a, s));
    if (bytes)
        dcb_lev_leq_kernel<8><<<(unsigned)blocks, 128, 0, s>>>((const uint8_t*)d->sym.p, (const uint64_t*)d->off.p, (const uint32_t*)d->len.p,
                                                               (const uint32_t*)d->a.p, (const uint32_t*)d->b.p, n_pairs, n_seqs, frac,
                                                               (uint8_t*)d->ver.p, (uint32_t*)d->flag.p);
    else
        dcb_lev_leq_kernel<3><<<(unsigned)blocks, 128, 0, s>>>((const uint8_t*)d->sym.p, (const uint64_t*)d->off.p, (const uint32_t*)d->len.p,
                                                               (const uint32_t*)d->a.p, (const uint32_t*)d->b.p, n_pairs, n_seqs, frac,
                                                               (uint8_t*)d->ver.p, (uint32_t*)d->flag.p);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaEventRecord(ev.b, s));
    uint32_t flag[4] = {0, 0, 0, 0};
    CUDA_TRY(cudaMemcpyAsync(verdict, d->ver.p, n_pairs, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(flag, d->flag.p, 16, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ev.a, ev.b) == cudaSuccess) d->last_ms = ms;   // kernel time of this call (dcb_dist_last_ms)
    if (flag[0]) { dcb_set_error("dcb_lev_leq: pair %u names a sequence out of range", flag[1]); return DCB_EINVAL; }
    if (flag[2]) { dcb_set_error("dcb_lev_leq: a symbol code above 7 in a sequence of pair %u (codes are 0..7)", flag[3]); return DCB_EINVAL; }
    return DCB_OK;
}

int dcb_barcodes(dcb_dist* d, const char* bc_text, const uint64_t* bc_off, const uint32_t* bc_len, const char* q_text,
                 const uint64_t* q_off, const uint32_t* q_len, uint64_t n, const dcb_bc_params* prm, uint8_t* status,
                 uint8_t* n1len, uint64_t* code) {
    if (!d || !prm || (n && (!bc_text || !bc_off || !bc_len || !q_text || !q_off || !q_len || !status || !n1len || !code))) {
        dcb_set_error("dcb_barcodes: null argument");
        return DCB_EINVAL;
    }
    if (n == 0) return DCB_OK;
    BcParams P;
    std::memset(&P, 0, sizeof(P));
    // spacers, window of spacer 1 and barcode length per design (collapse.py:172-189, 367-479)
    const char *sp1, *sp2 = "";
    switch (prm->oligo) {
    case DCB_OLIGO_M13:       sp1 = "GTCGTGACTGGGAAAACCCTGG"; sp2 = "GTCGTGAT"; P.layout = BC_TWO_SPACERS; break;
    case DCB_OLIGO_I8:        sp1 = "GTCGTGAT"; sp2 = "GTCGTGAT"; P.layout = BC_TWO_SPACERS; break;
    case DCB_OLIGO_I8_SINGLE: sp1 = "ATCACGAC"; P.layout = BC_N1_SPACER_N2; break;
    case DCB_OLIGO_NEBIO:     sp1 = "TACGGG"; P.layout = BC_FIXED; P.lo = 18; P.hi = 28; P.bclen = 17; break;
    case DCB_OLIGO_TAKARA:    sp1 = "GTACGGG"; P.layout = BC_FIXED; P.lo = 0; P.hi = 19; P.bclen = 12; break;
    default: dcb_set_error("dcb_barcodes: oligo %d has no device path (DCB_OLIGO_* are 0..4)", prm->oligo); return DCB_EUNSUPPORTED;
    }
    P.len1 = (int)std::strlen(sp1); P.len2 = (int)std::strlen(sp2);
    if (P.layout != BC_FIXED) { P.lo = 0; P.hi = 10 + P.len1; P.bclen = 12; }
    std::memcpy(P.sp1, sp1, P.len1); std::memcpy(P.sp2, sp2, P.len2);
    P.allow_ns = prm->allow_ns; P.min_q = prm->min_q; P.max_below = prm->max_below; P.avg_q = prm->avg_q;
    CUDA_TRY(cudaSetDevice(d->device));
    cudaStream_t s = d->stream;
    uint64_t bc_bytes = 0, q_bytes = 0;
    for (uint64_t i = 0; i < n; i++) { bc_bytes = std::max<uint64_t>(bc_bytes, bc_off[i] + bc_len[i]); q_bytes = std::max<uint64_t>(q_bytes, q_off[i] + q_len[i]); }
    DevMem dbc, dq, dbo, dbl, dqo, dql, dst, dn1, dcd;
    CUDA_TRY(dbc.alloc(bc_bytes + 16)); CUDA_TRY(dq.alloc(q_bytes + 16));
    CUDA_TRY(dbo.alloc(n * 8)); CUDA_TRY(dbl.alloc(n * 4)); CUDA_TRY(dqo.alloc(n * 8)); CUDA_TRY(dql.alloc(n * 4));
    CUDA_TRY(dst.alloc(n)); CUDA_TRY(dn1.alloc(n)); CUDA_TRY(dcd.alloc(n * 8));
    CUDA_TRY(cudaMemcpyAsync(dbc.p, bc_text, bc_bytes, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(dq.p, q_text, q_bytes, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(dbo.p, bc_off, n * 8, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(dbl.p, bc_len, n * 4, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(dqo.p, q_off, n * 8, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(dql.p, q_len, n * 4, cudaMemcpyHostToDevice, s));
    Events ev;
    CUDA_TRY(cudaEventCreate(&ev.a)); CUDA_TRY(cudaEventCreate(&ev.b));
    CUDA_TRY(cudaEventRecord(ev.a, s));
    dcb_barcodes_kernel<<<(unsigned)((n + 127) / 128), 128, 0, s>>>(dbc.as<unsigned char>(), dq.as<unsigned char>(), dbo.as<uint64_t>(),
                                                                   dbl.as<uint32_t>(), dqo.as<uint64_t>(), dql.as<uint32_t>(), n, P,
                                                                   dst.as<uint8_t>(), dn1.as<uint8_t>(), dcd.as<uint64_t>());
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaEventRecord(ev.b, s));
    CUDA_TRY(cudaMemcpyAsync(status, dst.p, n, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(n1len, dn1.p, n, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(code, dcd.p, n * 8, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ev.a, ev.b) == cudaSuccess) d->last_ms = ms;
    return DCB_OK;
}

const char* dcb_dist_last_method(const dcb_dist* d) { return d ? d->last_method : ""; }

}  // extern "C"

int dcb_dist_device(const dcb_dist* d) { return d->device; }
void* dcb_dist_stream(const dcb_dist* d) { return (void*)d->stream; }
void dcb_dist_set_last_ms(dcb_dist* d, double ms) { d->last_ms = ms; }

extern "C" {

int dcb_dist_last_ms(dcb_dist* d, double* ms) {
    if (!d || !ms) return DCB_EINVAL;
    *ms = d->last_ms;
    return DCB_OK;
}

}  // extern "C"
