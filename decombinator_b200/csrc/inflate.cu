// inflate.cu -- gzip input inflated on the GPU (sm_100a): the decoder of inflate_core.cuh run as one thread per
// chunk or per member.
//
// Members with known bounds (BGZF): one decoder per member in byte mode, straight to the member's place in the
// segment's output; CRC-32 and ISIZE checked per member on the device.
//
// One deflate stream (or members without sizes): the compressed bytes are cut into nominal chunks of C bytes.
//   find     one block per chunk tests every bit offset after the chunk's nominal start with inf_dyn_ok and keeps the
//            first that passes (chunk 0 starts behind the first member header);
//   decode   every chunk decodes from its candidate in marker mode and stops where it lands on a later candidate;
//   chain    chunk 0 starts at the true start; from there the host follows "landed on".  A chunk decoded from a true
//            block boundary lands only on true block boundaries, so every kept start is one and a false candidate
//            never reaches the output (the chunk before it decodes past it and absorbs the dropped chunk);
//   windows  one block walks the chain: the window of chunk k + 1 is the last 32 KB of chunk k resolved;
//   resolve  one parallel pass replaces every marker and writes the segment's bytes contiguously;
//   CRC      CRC-32 of 32 KB pieces split at member ends, combined on the host and checked against each trailer.
// The chunk list is processed in segments: device memory holds the compressed file, one segment's symbol buffers and
// one segment's text; the window, the chain position and the running CRC carry from one segment to the next.  The
// decode of segment s + 1 runs while segment s is copied to the caller.
#include "dcb_internal.h"
#include "inflate_core.cuh"

#include <cuda_runtime.h>

#include <algorithm>
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

namespace {

constexpr uint64_t kChunkBytes = 64 << 10;         // nominal chunk (DESIGN §4.8: why this size)
constexpr uint64_t kSegmentBytes = 1ull << 30;     // compressed bytes per segment
constexpr uint64_t kSymPerByte = 8;                // first-attempt output capacity per compressed byte of a chunk
constexpr uint64_t kLimitChunks = 16;              // a chunk gives up after this many nominal chunks of input,
constexpr uint64_t kLimitMin = 4 << 20;            // and at least this many bytes (deflate blocks are up to ~100 KB)
constexpr uint32_t kMaxMemberEnds = 64;            // member ends recorded per chunk
constexpr uint64_t kPiece = 32768;                 // CRC piece
constexpr int kDecodeThreads = 32;                 // decoders per block (their tables interleaved in shared memory)
constexpr int kFindThreads = 128;

struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
    ~DevBuf() { if (p) cudaFree(p); }
    cudaError_t alloc(size_t n) {
        if (p) { cudaFree(p); p = nullptr; bytes = 0; }
        cudaError_t e = cudaMalloc(&p, n ? n : 16);
        if (e == cudaSuccess) bytes = n;
        return e;
    }
    cudaError_t reserve(size_t n) { return n <= bytes && p ? cudaSuccess : alloc(n + n / 4); }
    template <class T> T* as() { return static_cast<T*>(p); }
};

// One decoder's work and its report.
struct Job {
    uint64_t start, limit, out_off, cap;
};
struct Report {
    int32_t status;
    uint32_t landed, n_members, pad;
    uint64_t produced, end_bit;
};

template <typename T>
__global__ void __launch_bounds__(kDecodeThreads)
dcb_inflate_decode_kernel(const uint8_t* __restrict__ in, uint64_t n, const Job* __restrict__ jobs, uint32_t n_jobs,
                          const uint64_t* __restrict__ cand, uint32_t ncand, int gzip, T* __restrict__ out, Report* __restrict__ rep,
                          uint64_t* __restrict__ mend_pos, uint32_t* __restrict__ mend_crc, uint32_t* __restrict__ mend_isize,
                          const uint64_t* __restrict__ expect_end, unsigned int* __restrict__ n_bad) {
    __shared__ uint16_t u16[INF_TAB_U16 * kDecodeThreads];
    __shared__ uint8_t u8[INF_TAB_U8 * kDecodeThreads];
    const uint32_t i = blockIdx.x * kDecodeThreads + threadIdx.x;
    if (i >= n_jobs) return;
    const Job jb = jobs[i];
    InfJob J;
    J.in = in; J.n = n; J.start = jb.start; J.limit = jb.limit; J.cand = cand; J.ncand = ncand; J.gzip = gzip;
    J.marker = sizeof(T) == 2;
    J.mend_pos = mend_pos ? mend_pos + (uint64_t)i * kMaxMemberEnds : nullptr;
    J.mend_crc = mend_crc ? mend_crc + (uint64_t)i * kMaxMemberEnds : nullptr;
    J.mend_isize = mend_isize ? mend_isize + (uint64_t)i * kMaxMemberEnds : nullptr;
    J.mend_cap = mend_pos ? kMaxMemberEnds : 0;
    J.blocks = nullptr; J.blocks_cap = 0;
    const InfResult R = inf_decode<T, kDecodeThreads>(J, inf_tab<kDecodeThreads>(u16, u8, threadIdx.x), out + jb.out_off, jb.cap);
    if (rep) {
        Report r;
        r.status = R.status; r.landed = R.landed; r.n_members = R.n_members; r.pad = 0; r.produced = R.produced; r.end_bit = R.end_bit;
        rep[i] = r;
    }
    // members with known bounds: the decode must end where the member's deflate data ends, with ISIZE bytes
    if (expect_end && (R.status != INF_END || R.produced != jb.cap || (R.end_bit + 7) / 8 != expect_end[i])) atomicAdd(n_bad, 1u);
}

// first bit offset in [k * C * 8, (k + 1) * C * 8) holding a dynamic block header with complete codes; ~0 when none
__global__ void __launch_bounds__(kFindThreads)
dcb_inflate_find_kernel(const uint8_t* __restrict__ in, uint64_t n, uint64_t chunk_bytes, uint64_t first, uint64_t* __restrict__ starts) {
    __shared__ uint16_t u16[INF_VTAB_U16 * kFindThreads];
    __shared__ uint8_t u8[INF_VTAB_U8 * kFindThreads];
    __shared__ unsigned long long best;
    const uint64_t k = blockIdx.x;
    if (k == 0) {
        if (threadIdx.x == 0) starts[0] = first;
        return;
    }
    const uint64_t lo = k * chunk_bytes * 8, hi = min((k + 1) * chunk_bytes, n) * 8;
    if (threadIdx.x == 0) best = ~0ull;
    __syncthreads();
    for (uint64_t base = lo; base < hi; base += kFindThreads) {
        const uint64_t bit = base + threadIdx.x;
        if (bit < hi && inf_dyn_ok<kFindThreads>(in, n, bit, u16, u8, threadIdx.x)) atomicMin(&best, (unsigned long long)bit);
        __syncthreads();
        if (best != ~0ull) break;
        __syncthreads();
    }
    if (threadIdx.x == 0) starts[k] = best;
}

// windows[j + 1] = last 32 KB of (windows[j] ++ chain chunk j resolved through windows[j]), j = 0 .. m - 1
__global__ void __launch_bounds__(1024)
dcb_inflate_window_kernel(const uint16_t* const* __restrict__ sym, const uint64_t* __restrict__ len, uint32_t m, uint8_t* __restrict__ windows) {
    for (uint32_t j = 0; j < m; j++) {
        const uint8_t* w = windows + (uint64_t)j * INF_WINDOW;
        uint8_t* nw = windows + (uint64_t)(j + 1) * INF_WINDOW;
        const uint64_t L = len[j];
        const uint16_t* s = sym[j];
        for (uint32_t i = threadIdx.x; i < INF_WINDOW; i += blockDim.x) {
            const uint64_t g = L + i;             // index into windows[j] ++ chunk j
            nw[i] = g < INF_WINDOW ? w[g] : inf_resolve(s[g - INF_WINDOW], w);
        }
        __syncthreads();
    }
}

// out[off[j] + i] = chain chunk j's symbol i resolved; blockIdx.y = j
__global__ void __launch_bounds__(256)
dcb_inflate_resolve_kernel(const uint16_t* const* __restrict__ sym, const uint64_t* __restrict__ len, const uint64_t* __restrict__ off,
                           const uint8_t* __restrict__ windows, uint8_t* __restrict__ out) {
    const uint32_t j = blockIdx.y;
    const uint16_t* s = sym[j];
    const uint8_t* w = windows + (uint64_t)j * INF_WINDOW;
    uint8_t* o = out + off[j];
    const uint64_t L = len[j];
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < L; i += (uint64_t)gridDim.x * blockDim.x) o[i] = inf_resolve(s[i], w);
}

// crc[i] = crc32 of out[off[i], + len[i]); with expect: count the pieces whose CRC differs
__global__ void __launch_bounds__(256)
dcb_inflate_crc_kernel(const uint8_t* __restrict__ out, const uint64_t* __restrict__ off, const uint32_t* __restrict__ len, uint64_t n,
                       uint32_t* __restrict__ crc, const uint32_t* __restrict__ expect, unsigned int* __restrict__ n_bad) {
    __shared__ uint32_t table[256];
    table[threadIdx.x] = inf_crc_entry(threadIdx.x);
    __syncthreads();
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t c = inf_crc32(0, out + off[i], len[i], table);
    if (crc) crc[i] = c;
    if (expect && c != expect[i]) atomicAdd(n_bad, 1u);
}

}  // namespace

struct dcb_inflate {
    int device = 0;
    cudaStream_t s = nullptr, copy = nullptr;
    uint64_t n = 0, chunk = kChunkBytes, seg_bytes = kSegmentBytes, first = 0;
    const unsigned char* host = nullptr;       // the caller's compressed bytes (trailers of BGZF members are read here)
    DevBuf d_in, d_cand, d_jobs, d_rep, d_mpos, d_mcrc, d_misize, d_sym, d_big, d_out, d_win, d_chain, d_pieces, d_crc, d_misc;
    bool members = false, started = false, done = false, has_pending = false, launched = false;
    uint64_t pending = 0;
    // stream mode
    std::vector<uint64_t> cand;
    uint64_t next_chunk = 0, chain_next = 0, seg_a = 0, seg_b = 0;
    bool chain_done = false;
    uint32_t crc_cur = 0;
    uint64_t len_cur = 0;
    std::vector<Job> jobs;
    std::vector<uint64_t> job_chunk;
    // members mode
    std::vector<uint64_t> m_start, m_end;
    std::vector<uint32_t> m_isize;
    uint64_t next_member = 0, seg_m0 = 0, seg_m1 = 0;

    ~dcb_inflate() {
        if (s) cudaStreamDestroy(s);
        if (copy) cudaStreamDestroy(copy);
    }
};

namespace {

int gzip_header_end(const unsigned char* p, uint64_t n, uint64_t* bit) {
    InfBits b;
    b.init(p, n, 0);
    if (n < 18 || inf_gzip_header(b) != 0) {
        dcb_set_error("dcb_inflate: not a gzip member header at the start of the file");
        return DCB_EIO;
    }
    *bit = b.pos();
    return DCB_OK;
}

// Stream mode: launch the decode of the next segment's chunks from the chain's position on.
int launch_stream_decode(dcb_inflate* h) {
    const uint64_t nc = h->cand.size();
    const uint64_t per_seg = std::min<uint64_t>(65535, std::max<uint64_t>(1, h->seg_bytes / h->chunk));   // grid.y of the resolve pass
    h->seg_a = std::max(h->next_chunk, h->chain_next);
    h->seg_b = std::min(nc, h->seg_a + per_seg);
    h->next_chunk = h->seg_b;
    const uint64_t cap = h->chunk * kSymPerByte;
    h->jobs.clear();
    h->job_chunk.clear();
    for (uint64_t k = h->seg_a; k < h->seg_b; k++) {
        Job j;
        j.start = h->cand[k];
        j.limit = h->cand[k] + std::max(kLimitChunks * h->chunk, kLimitMin) * 8;
        j.out_off = (k - h->seg_a) * cap;
        j.cap = cap;
        h->jobs.push_back(j);
        h->job_chunk.push_back(k);
    }
    const uint64_t nj = h->jobs.size();
    CUDA_TRY(h->d_jobs.reserve(nj * sizeof(Job)));
    CUDA_TRY(h->d_rep.reserve(nj * sizeof(Report)));
    CUDA_TRY(h->d_mpos.reserve(nj * kMaxMemberEnds * 8));
    CUDA_TRY(h->d_mcrc.reserve(nj * kMaxMemberEnds * 4));
    CUDA_TRY(h->d_misize.reserve(nj * kMaxMemberEnds * 4));
    CUDA_TRY(h->d_sym.reserve(nj * cap * 2));
    CUDA_TRY(cudaMemcpyAsync(h->d_jobs.p, h->jobs.data(), nj * sizeof(Job), cudaMemcpyHostToDevice, h->s));
    dcb_inflate_decode_kernel<uint16_t><<<(unsigned)((nj + kDecodeThreads - 1) / kDecodeThreads), kDecodeThreads, 0, h->s>>>(
        h->d_in.as<uint8_t>(), h->n, h->d_jobs.as<Job>(), (uint32_t)nj, h->d_cand.as<uint64_t>(), (uint32_t)nc, 1, h->d_sym.as<uint16_t>(),
        h->d_rep.as<Report>(), h->d_mpos.as<uint64_t>(), h->d_mcrc.as<uint32_t>(), h->d_misize.as<uint32_t>(), nullptr, nullptr);
    CUDA_TRY(cudaGetLastError());
    h->launched = true;
    return DCB_OK;
}

const char* status_text(int st) {
    switch (st) {
        case INF_LIMIT: return "a chunk on the chain reached its bit limit (no block start found for a long stretch)";
        case INF_E_CODE: return "invalid code";
        case INF_E_DIST: return "distance too far back";
        case INF_E_OVERRUN: return "input ended inside a block";
        case INF_E_STORED: return "stored block LEN / NLEN mismatch";
        case INF_E_TABLE: return "invalid block header";
        case INF_E_HEADER: return "invalid member header";
        case INF_E_MEMBERS: return "too many member ends in one chunk";
        default: return "chain broken";
    }
}

// Stream mode: the chain through the decoded segment, windows, resolve, CRC.  Leaves the text in d_out (h->pending).
int finish_stream_segment(dcb_inflate* h) {
    h->launched = false;
    const uint64_t nj = h->jobs.size();
    std::vector<Report> rep(nj);
    std::vector<uint64_t> mpos(nj * kMaxMemberEnds);
    std::vector<uint32_t> mcrc(nj * kMaxMemberEnds), misize(nj * kMaxMemberEnds);
    CUDA_TRY(cudaMemcpyAsync(rep.data(), h->d_rep.p, nj * sizeof(Report), cudaMemcpyDeviceToHost, h->s));
    CUDA_TRY(cudaMemcpyAsync(mpos.data(), h->d_mpos.p, nj * kMaxMemberEnds * 8, cudaMemcpyDeviceToHost, h->s));
    CUDA_TRY(cudaMemcpyAsync(mcrc.data(), h->d_mcrc.p, nj * kMaxMemberEnds * 4, cudaMemcpyDeviceToHost, h->s));
    CUDA_TRY(cudaMemcpyAsync(misize.data(), h->d_misize.p, nj * kMaxMemberEnds * 4, cudaMemcpyDeviceToHost, h->s));
    CUDA_TRY(cudaStreamSynchronize(h->s));
    // the chain inside this segment
    std::vector<uint64_t> chain;           // job indices
    while (!h->chain_done && h->chain_next < h->seg_b) {
        const uint64_t j = h->chain_next - h->seg_a;
        const Report& r = rep[j];
        chain.push_back(j);
        if (r.status == INF_END) {
            h->chain_done = true;
        } else if (r.status == INF_LANDED && r.landed > h->chain_next) {
            h->chain_next = r.landed;
        } else {
            dcb_set_error("dcb_inflate: chunk %llu at bit %llu: %s", (unsigned long long)h->chain_next, (unsigned long long)h->cand[h->chain_next],
                          status_text(r.status));
            return DCB_EIO;
        }
    }
    // chunks that outgrew their buffer: decode once more with their exact size
    const uint64_t cap = h->chunk * kSymPerByte;
    std::vector<Job> big;
    std::vector<uint64_t> big_of;
    uint64_t big_total = 0;
    for (uint64_t j : chain)
        if (rep[j].produced > cap) {
            Job b = h->jobs[j];
            b.out_off = big_total;
            b.cap = rep[j].produced;
            big_total += b.cap;
            big.push_back(b);
            big_of.push_back(j);
        }
    if (!big.empty()) {
        CUDA_TRY(h->d_big.reserve(big_total * 2));
        CUDA_TRY(h->d_jobs.reserve(big.size() * sizeof(Job)));
        CUDA_TRY(cudaMemcpyAsync(h->d_jobs.p, big.data(), big.size() * sizeof(Job), cudaMemcpyHostToDevice, h->s));
        dcb_inflate_decode_kernel<uint16_t><<<(unsigned)((big.size() + kDecodeThreads - 1) / kDecodeThreads), kDecodeThreads, 0, h->s>>>(
            h->d_in.as<uint8_t>(), h->n, h->d_jobs.as<Job>(), (uint32_t)big.size(), h->d_cand.as<uint64_t>(), (uint32_t)h->cand.size(), 1,
            h->d_big.as<uint16_t>(), nullptr, h->d_mpos.as<uint64_t>(), h->d_mcrc.as<uint32_t>(), h->d_misize.as<uint32_t>(), nullptr, nullptr);
        CUDA_TRY(cudaGetLastError());
    }
    const uint32_t m = (uint32_t)chain.size();
    std::vector<const uint16_t*> sym(m);
    std::vector<uint64_t> len(m), off(m + 1, 0);
    for (uint32_t c = 0, b = 0; c < m; c++) {
        const uint64_t j = chain[c];
        if (b < big_of.size() && big_of[b] == j) sym[c] = h->d_big.as<uint16_t>() + big[b++].out_off;
        else sym[c] = h->d_sym.as<uint16_t>() + h->jobs[j].out_off;
        len[c] = rep[j].produced;
        off[c + 1] = off[c] + len[c];
    }
    const uint64_t total = off[m];
    // chain arrays: sym pointers, lengths, offsets
    CUDA_TRY(h->d_chain.reserve((size_t)m * 24 + 64));
    uint8_t* dc = h->d_chain.as<uint8_t>();
    if (m) {
        CUDA_TRY(cudaMemcpyAsync(dc, sym.data(), m * 8, cudaMemcpyHostToDevice, h->s));
        CUDA_TRY(cudaMemcpyAsync(dc + m * 8, len.data(), m * 8, cudaMemcpyHostToDevice, h->s));
        CUDA_TRY(cudaMemcpyAsync(dc + m * 16, off.data(), m * 8, cudaMemcpyHostToDevice, h->s));
    }
    // windows[0] carries over from the previous segment; windows[m] carries on to the next
    const size_t wbytes = (size_t)(m + 1) * INF_WINDOW;
    if (h->d_win.bytes < wbytes) {
        DevBuf nw;
        CUDA_TRY(nw.alloc(wbytes + wbytes / 4));
        if (h->d_win.p) CUDA_TRY(cudaMemcpyAsync(nw.p, h->d_win.p, INF_WINDOW, cudaMemcpyDeviceToDevice, h->s));
        else CUDA_TRY(cudaMemsetAsync(nw.p, 0, INF_WINDOW, h->s));
        std::swap(h->d_win.p, nw.p);
        std::swap(h->d_win.bytes, nw.bytes);
        CUDA_TRY(cudaStreamSynchronize(h->s));
    }
    CUDA_TRY(h->d_out.reserve(total + 16));
    if (m) {
        dcb_inflate_window_kernel<<<1, 1024, 0, h->s>>>((const uint16_t* const*)dc, (const uint64_t*)(dc + m * 8), m, h->d_win.as<uint8_t>());
        CUDA_TRY(cudaGetLastError());
        dcb_inflate_resolve_kernel<<<dim3(64, m), 256, 0, h->s>>>((const uint16_t* const*)dc, (const uint64_t*)(dc + m * 8),
                                                                   (const uint64_t*)(dc + m * 16), h->d_win.as<uint8_t>(), h->d_out.as<uint8_t>());
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(cudaMemcpyAsync(h->d_win.p, h->d_win.as<uint8_t>() + (size_t)m * INF_WINDOW, INF_WINDOW, cudaMemcpyDeviceToDevice, h->s));
    }
    // CRC pieces: 32 KB, split at member ends
    struct End { uint64_t at; uint32_t crc, isize; };
    std::vector<End> ends;
    for (uint32_t c = 0; c < m; c++) {
        const uint64_t j = chain[c];
        for (uint32_t e = 0; e < rep[j].n_members; e++)
            ends.push_back({off[c] + mpos[j * kMaxMemberEnds + e], mcrc[j * kMaxMemberEnds + e], misize[j * kMaxMemberEnds + e]});
    }
    std::vector<uint64_t> poff;
    std::vector<uint32_t> plen;
    std::vector<int64_t> pend;             // index into ends of the member a piece closes, or -1
    {
        uint64_t at = 0;
        size_t e = 0;
        while (at < total || e < ends.size()) {
            while (e < ends.size() && ends[e].at == at) {
                poff.push_back(at); plen.push_back(0); pend.push_back((int64_t)e);
                e++;
            }
            if (at >= total) break;
            uint64_t to = std::min(total, at + kPiece);
            if (e < ends.size() && ends[e].at < to) to = ends[e].at;
            poff.push_back(at); plen.push_back((uint32_t)(to - at)); pend.push_back(-1);
            at = to;
        }
    }
    const uint64_t np = poff.size();
    std::vector<uint32_t> pcrc(np);
    if (np) {
        CUDA_TRY(h->d_pieces.reserve(np * 12 + 16));
        CUDA_TRY(h->d_crc.reserve(np * 4));
        uint8_t* dp = h->d_pieces.as<uint8_t>();
        CUDA_TRY(cudaMemcpyAsync(dp, poff.data(), np * 8, cudaMemcpyHostToDevice, h->s));
        CUDA_TRY(cudaMemcpyAsync(dp + np * 8, plen.data(), np * 4, cudaMemcpyHostToDevice, h->s));
        dcb_inflate_crc_kernel<<<(unsigned)((np + 255) / 256), 256, 0, h->s>>>(h->d_out.as<uint8_t>(), (const uint64_t*)dp, (const uint32_t*)(dp + np * 8),
                                                                            np, h->d_crc.as<uint32_t>(), nullptr, nullptr);
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(cudaMemcpyAsync(pcrc.data(), h->d_crc.p, np * 4, cudaMemcpyDeviceToHost, h->s));
    }
    CUDA_TRY(cudaStreamSynchronize(h->s));
    const uint32_t full_shift = inf_crc_shift(kPiece);
    for (uint64_t i = 0; i < np; i++) {
        if (plen[i]) {
            h->crc_cur = inf_crc_combine(h->crc_cur, pcrc[i], plen[i] == kPiece ? full_shift : inf_crc_shift(plen[i]));
            h->len_cur += plen[i];
        }
        if (pend[i] >= 0) {
            const End& e = ends[(size_t)pend[i]];
            if (e.crc != h->crc_cur || e.isize != (uint32_t)h->len_cur) {
                dcb_set_error("dcb_inflate: member ending at output byte %llu: %s mismatch", (unsigned long long)(h->len_cur),
                              e.crc != h->crc_cur ? "CRC-32" : "ISIZE");
                return DCB_EIO;
            }
            h->crc_cur = 0;
            h->len_cur = 0;
        }
    }
    h->pending = total;
    h->has_pending = true;
    if (h->chain_done) h->done = true;
    else if (h->chain_next >= h->cand.size()) {
        dcb_set_error("dcb_inflate: the chain ran past the last chunk");
        return DCB_EIO;
    }
    return DCB_OK;
}

// Members mode: the next segment of members decoded straight to d_out, checked on the device.
int members_segment(dcb_inflate* h) {
    const uint64_t nm = h->m_start.size();
    uint64_t a = h->next_member, b = a, in_bytes = 0, total = 0;
    while (b < nm && (b == a || in_bytes + (h->m_end[b] - h->m_start[b]) <= h->seg_bytes)) {
        in_bytes += h->m_end[b] - h->m_start[b];
        total += h->m_isize[b];
        b++;
    }
    h->next_member = b;
    const uint64_t nj = b - a;
    std::vector<Job> jobs(nj);
    std::vector<uint64_t> expect_end(nj), poff(nj);
    std::vector<uint32_t> plen(nj), pcrc(nj);
    uint64_t at = 0;
    for (uint64_t i = 0; i < nj; i++) {
        const uint64_t k = a + i;
        jobs[i].start = h->m_start[k] * 8;
        jobs[i].limit = ~0ull;
        jobs[i].out_off = at;
        jobs[i].cap = h->m_isize[k];
        expect_end[i] = h->m_end[k];
        poff[i] = at;
        plen[i] = h->m_isize[k];
        std::memcpy(&pcrc[i], h->host + h->m_end[k], 4);
        at += h->m_isize[k];
    }
    CUDA_TRY(h->d_jobs.reserve(nj * sizeof(Job)));
    CUDA_TRY(h->d_pieces.reserve(nj * 20 + 16));
    CUDA_TRY(h->d_out.reserve(total + 16));
    CUDA_TRY(h->d_misc.reserve(16));
    uint8_t* dp = h->d_pieces.as<uint8_t>();
    CUDA_TRY(cudaMemcpyAsync(h->d_jobs.p, jobs.data(), nj * sizeof(Job), cudaMemcpyHostToDevice, h->s));
    CUDA_TRY(cudaMemcpyAsync(dp, expect_end.data(), nj * 8, cudaMemcpyHostToDevice, h->s));
    CUDA_TRY(cudaMemcpyAsync(dp + nj * 8, poff.data(), nj * 8, cudaMemcpyHostToDevice, h->s));
    CUDA_TRY(cudaMemcpyAsync(dp + nj * 16, plen.data(), nj * 4, cudaMemcpyHostToDevice, h->s));
    CUDA_TRY(h->d_crc.reserve(nj * 4));
    CUDA_TRY(cudaMemcpyAsync(h->d_crc.p, pcrc.data(), nj * 4, cudaMemcpyHostToDevice, h->s));
    CUDA_TRY(cudaMemsetAsync(h->d_misc.p, 0, 8, h->s));
    unsigned int* bad = h->d_misc.as<unsigned int>();
    if (nj) {
        dcb_inflate_decode_kernel<uint8_t><<<(unsigned)((nj + kDecodeThreads - 1) / kDecodeThreads), kDecodeThreads, 0, h->s>>>(
            h->d_in.as<uint8_t>(), h->n, h->d_jobs.as<Job>(), (uint32_t)nj, nullptr, 0, 0, h->d_out.as<uint8_t>(), nullptr, nullptr, nullptr,
            nullptr, (const uint64_t*)dp, bad);
        CUDA_TRY(cudaGetLastError());
        dcb_inflate_crc_kernel<<<(unsigned)((nj + 255) / 256), 256, 0, h->s>>>(h->d_out.as<uint8_t>(), (const uint64_t*)(dp + nj * 8),
                                                                            (const uint32_t*)(dp + nj * 16), nj, nullptr, h->d_crc.as<uint32_t>(), bad + 1);
        CUDA_TRY(cudaGetLastError());
    }
    unsigned int nbad[2] = {0, 0};
    CUDA_TRY(cudaMemcpyAsync(nbad, bad, 8, cudaMemcpyDeviceToHost, h->s));
    CUDA_TRY(cudaStreamSynchronize(h->s));
    if (nbad[0] || nbad[1]) {
        dcb_set_error("dcb_inflate: %u member(s) do not decode to their size and end, %u fail their CRC-32", nbad[0], nbad[1]);
        return DCB_EIO;
    }
    h->pending = total;
    h->has_pending = true;
    if (h->next_member >= nm) h->done = true;
    h->launched = false;
    return DCB_OK;
}

}  // namespace

extern "C" {

int dcb_inflate_create(int device, const unsigned char* gz, uint64_t n_bytes, uint64_t chunk_bytes, uint64_t segment_bytes, dcb_inflate** out) {
    if (!out || (n_bytes && !gz)) {
        dcb_set_error("dcb_inflate_create: null argument");
        return DCB_EINVAL;
    }
    *out = nullptr;
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0) {
        (void)cudaGetLastError();
        dcb_set_error("dcb_inflate_create: no CUDA device available (there is no CPU fallback)");
        return DCB_ENOGPU;
    }
    if (device < 0 || device >= n_dev) {
        dcb_set_error("dcb_inflate_create: device %d of %d", device, n_dev);
        return DCB_EINVAL;
    }
    if (chunk_bytes && chunk_bytes < 1024) {
        dcb_set_error("dcb_inflate_create: chunks of at least 1 KiB");
        return DCB_EINVAL;
    }
    CUDA_TRY(cudaSetDevice(device));
    auto* h = new dcb_inflate();
    h->device = device;
    h->n = n_bytes;
    h->host = gz;
    if (chunk_bytes) h->chunk = chunk_bytes;
    if (segment_bytes) h->seg_bytes = segment_bytes;
    cudaError_t e = cudaStreamCreateWithFlags(&h->s, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->copy, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = h->d_in.alloc(n_bytes + 16);
    if (e == cudaSuccess && n_bytes) e = cudaMemcpyAsync(h->d_in.p, gz, n_bytes, cudaMemcpyHostToDevice, h->s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->s);
    if (e != cudaSuccess) {
        dcb_set_error("dcb_inflate_create: %s", cudaGetErrorString(e));
        delete h;
        return DCB_ENOGPU;
    }
    *out = h;
    return DCB_OK;
}

void dcb_inflate_destroy(dcb_inflate* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    if (h->s) cudaStreamSynchronize(h->s);
    delete h;
}

int dcb_inflate_find_starts(dcb_inflate* h, uint64_t* starts, uint64_t cap, uint64_t* n_chunks) {
    if (!h || !n_chunks || (cap && !starts)) {
        dcb_set_error("dcb_inflate_find_starts: null argument");
        return DCB_EINVAL;
    }
    const uint64_t nc = h->n ? (h->n + h->chunk - 1) / h->chunk : 0;
    *n_chunks = nc;
    if (!starts) return DCB_OK;
    if (cap < nc) {
        dcb_set_error("dcb_inflate_find_starts: room for %llu of %llu starts", (unsigned long long)cap, (unsigned long long)nc);
        return DCB_EINVAL;
    }
    uint64_t first = 0;
    int rc = gzip_header_end(h->host, h->n, &first);
    if (rc) return rc;
    CUDA_TRY(cudaSetDevice(h->device));
    DevBuf d;
    CUDA_TRY(d.alloc(nc * 8));
    dcb_inflate_find_kernel<<<(unsigned)nc, kFindThreads, 0, h->s>>>(h->d_in.as<uint8_t>(), h->n, h->chunk, first, d.as<uint64_t>());
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(starts, d.p, nc * 8, cudaMemcpyDeviceToHost, h->s));
    CUDA_TRY(cudaStreamSynchronize(h->s));
    return DCB_OK;
}

int dcb_inflate_begin(dcb_inflate* h, const uint64_t* starts, uint64_t n) {
    if (!h || !starts || n == 0) {
        dcb_set_error("dcb_inflate_begin: null argument");
        return DCB_EINVAL;
    }
    if (h->started) {
        dcb_set_error("dcb_inflate_begin: already started");
        return DCB_EINVAL;
    }
    uint64_t first = 0;
    int rc = gzip_header_end(h->host, h->n, &first);
    if (rc) return rc;
    if (starts[0] != first) {
        dcb_set_error("dcb_inflate_begin: the first start must be the first block of the stream (bit %llu)", (unsigned long long)first);
        return DCB_EINVAL;
    }
    h->cand.clear();
    for (uint64_t i = 0; i < n; i++) {
        if (starts[i] == ~0ull) continue;
        if (starts[i] >= h->n * 8 || (!h->cand.empty() && starts[i] <= h->cand.back())) {
            dcb_set_error("dcb_inflate_begin: start %llu is out of order or beyond the input", (unsigned long long)i);
            return DCB_EINVAL;
        }
        h->cand.push_back(starts[i]);
    }
    CUDA_TRY(cudaSetDevice(h->device));
    CUDA_TRY(h->d_cand.alloc(h->cand.size() * 8));
    CUDA_TRY(cudaMemcpyAsync(h->d_cand.p, h->cand.data(), h->cand.size() * 8, cudaMemcpyHostToDevice, h->s));
    CUDA_TRY(cudaStreamSynchronize(h->s));
    h->started = true;
    return DCB_OK;
}

int dcb_inflate_begin_members(dcb_inflate* h, const uint64_t* start, const uint64_t* end, const uint32_t* isize, uint64_t n) {
    if (!h || (n && (!start || !end || !isize))) {
        dcb_set_error("dcb_inflate_begin_members: null argument");
        return DCB_EINVAL;
    }
    if (h->started) {
        dcb_set_error("dcb_inflate_begin_members: already started");
        return DCB_EINVAL;
    }
    for (uint64_t i = 0; i < n; i++)
        if (start[i] > end[i] || end[i] + 8 > h->n) {
            dcb_set_error("dcb_inflate_begin_members: member %llu lies outside the input", (unsigned long long)i);
            return DCB_EINVAL;
        }
    h->m_start.assign(start, start + n);
    h->m_end.assign(end, end + n);
    h->m_isize.assign(isize, isize + n);
    h->members = true;
    h->started = true;
    if (n == 0) h->done = true;
    return DCB_OK;
}

int dcb_inflate_read(dcb_inflate* h, unsigned char* out, uint64_t cap, uint64_t* produced, uint64_t* more) {
    if (!h || !produced || !more || (cap && !out)) {
        dcb_set_error("dcb_inflate_read: null argument");
        return DCB_EINVAL;
    }
    if (!h->started) {
        dcb_set_error("dcb_inflate_read: call dcb_inflate_begin or dcb_inflate_begin_members first");
        return DCB_EINVAL;
    }
    *produced = 0;
    *more = 0;
    CUDA_TRY(cudaSetDevice(h->device));
    for (;;) {
        if (!h->has_pending) {
            if (h->done && !h->launched) return DCB_OK;
            int rc;
            if (h->members) rc = members_segment(h);
            else {
                rc = h->launched ? DCB_OK : launch_stream_decode(h);
                if (rc == DCB_OK) rc = finish_stream_segment(h);
            }
            if (rc) return rc;
            continue;
        }
        if (h->pending > cap - *produced) {
            *more = h->pending;
            return DCB_OK;
        }
        // the next segment decodes while this one is copied out
        if (!h->members && !h->done && !h->launched) {
            int rc = launch_stream_decode(h);
            if (rc) return rc;
        }
        if (h->pending) {
            CUDA_TRY(cudaMemcpyAsync(out + *produced, h->d_out.p, h->pending, cudaMemcpyDeviceToHost, h->copy));
            CUDA_TRY(cudaStreamSynchronize(h->copy));
        }
        *produced += h->pending;
        h->pending = 0;
        h->has_pending = false;
        if (h->launched) {
            int rc = finish_stream_segment(h);
            if (rc) return rc;
        }
    }
}

}  // extern "C"
