// pack_device.cuh -- device side of the ingest: ASCII reads -> 2-bit packed read slots ON THE GPU, and the host-buffer
// entry point that starts from ASCII (dcb_decombine_ascii).  Textually included by decombine.cu (one translation unit:
// it drives the same context and kernels).
//
// Replaces, like csrc/pack.cpp on the host, the string handling in front of dcr() in the reference's main loop:
// `vdj = record1[1]` (decombine.py:965-977) and revcomp(vdj) (decombine.py:182-184, 1000) = Bio.Seq.reverse_complement.
// Output is bit-identical to dcb_pack_reads: slot words, lengths, flag bits, and the exception list sorted by
// (read, position) with kind 1 = 'N', 2 = any other symbol, 3 = 'U' read on the reverse strand (its complement 'A' is a
// real base in that frame).  tests/test_gpu_pack.py compares the two.
//
// Layout of the work: one warp per group of 32 consecutive reads (= one flag word, one entry of the exception index).
// A read is packed by the whole warp: lane l takes bases [8 l, 8 l + 8) of every 256-base pass -- one unaligned 8-byte
// window of the text, two aligned 64-bit loads -- classifies them through a 256-entry table in shared memory, and the
// 16 bits of two neighbouring lanes make one slot word (coalesced 64-byte stores).  Exceptions are rare, so they are
// only COUNTED in this pass (per group); a one-block scan turns the counts into the exception index (with the running
// total of the previous chunk carried in, so the list of a batch packed chunk by chunk on two streams is contiguous),
// and a second pass over the flagged reads alone writes the entries in order.
#ifndef DCB_PACK_DEVICE_CUH
#define DCB_PACK_DEVICE_CUH

// table entry: bits 0-1 base code, bit 2 valid, bit 3 the symbol is 'N' (kind 1), bit 4 kind 3
#define DCB_PK_VALID 4u
#define DCB_PK_N 8u
#define DCB_PK_K3 16u
__device__ __forceinline__ uint32_t pack_table_entry(int c, int revcomp) {
    // Bio.Seq's complement leaves everything but the IUPAC letters alone; only upper-case A/C/G/T (after the
    // complement) can match a tag or a germline region
    if (c == 'N') return DCB_PK_N;
    if (!revcomp) return c == 'A' ? (DCB_PK_VALID | 0u) : c == 'C' ? (DCB_PK_VALID | 1u) : c == 'G' ? (DCB_PK_VALID | 2u) : c == 'T' ? (DCB_PK_VALID | 3u) : 0u;
    return c == 'A' ? (DCB_PK_VALID | 3u) : c == 'C' ? (DCB_PK_VALID | 2u) : c == 'G' ? (DCB_PK_VALID | 1u) : c == 'T' ? (DCB_PK_VALID | 0u)
         : c == 'U' ? (DCB_PK_VALID | DCB_PK_K3 | 0u) : 0u;
}

struct PackSrc {
    const unsigned char* text;   // device copy of the text bytes [text_lo, ...) of this chunk (8 spare bytes behind)
    const uint64_t* off;         // per read of the chunk: offset into the host text (null: read i at i * stride)
    const uint32_t* len;         // per read (null: uniform_len)
    uint64_t text_lo;            // host offset of text[0]
    uint64_t stride;
    uint32_t uniform_len;
    uint32_t first;              // global index of the chunk's first read (a multiple of 32)
    uint32_t count;
};

// Eight oriented bases from position i0 of a read of L bases at text + o: the bytes of the unaligned 8-byte window as one
// 64-bit value, byte j = oriented base i0 + j (reverse strand: the window is read backwards from the read's end).
// Bytes outside the read are whatever lies there; the caller masks by position.
__device__ __forceinline__ uint64_t pack_window(const unsigned char* text, uint64_t o, uint32_t L, uint32_t i0, int revcomp) {
    const long long a = revcomp ? (long long)o + (long long)L - 8 - (long long)i0 : (long long)o + (long long)i0;
    // a may be negative by up to 7 at the start of the text (reverse strand, last window): clamp the aligned loads
    const long long al = a >= 0 ? (a & ~7ll) : -8ll;
    const int sh = (int)(a - al) * 8;
    const unsigned long long lo = al >= 0 ? __ldg(reinterpret_cast<const unsigned long long*>(text + al)) : 0ull;
    const unsigned long long hi = sh ? __ldg(reinterpret_cast<const unsigned long long*>(text + al + 8)) : 0ull;
    unsigned long long x = sh ? (lo >> sh) | (hi << (64 - sh)) : lo;
    if (revcomp) {
        const uint32_t xl = (uint32_t)x, xh = (uint32_t)(x >> 32);
        x = ((unsigned long long)__byte_perm(xl, 0u, 0x0123) << 32) | (unsigned long long)__byte_perm(xh, 0u, 0x0123);
    }
    return x;
}

// Classify the 8 bases of a window: 16 packed bits + masks (bit j <-> base i0 + j) of the exceptions by kind.
__device__ __forceinline__ void pack_classify(uint64_t x, uint32_t L, uint32_t i0, const uint8_t* tab, uint32_t& bits,
                                              uint32_t& m_exc, uint32_t& m_n, uint32_t& m_k3) {
    bits = 0; m_exc = 0; m_n = 0; m_k3 = 0;
#pragma unroll
    for (int j = 0; j < 8; j++) {
        const uint32_t e = tab[(uint32_t)(x >> (8 * j)) & 255u];
        const bool in = i0 + j < L;
        if (in) {
            bits |= (e & 3u) << (2 * j);                       // invalid symbols pack as base 0
            if (!(e & DCB_PK_VALID) || (e & DCB_PK_K3)) m_exc |= 1u << j;
            if (e & DCB_PK_N) m_n |= 1u << j;
            if (e & DCB_PK_K3) m_k3 |= 1u << j;
        }
    }
}

// pass 1: words, lengths, flag words, exception count per group
__global__ void __launch_bounds__(256)
dcb_pack_kernel(PackSrc src, int revcomp, uint32_t slot_words, uint32_t* __restrict__ words, uint16_t* __restrict__ lens,
                uint32_t* __restrict__ flags, uint32_t* __restrict__ group_count) {
    __shared__ uint8_t tab[256];
    tab[threadIdx.x] = (uint8_t)pack_table_entry((int)threadIdx.x, revcomp);
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const uint32_t n_groups = (src.count + 31) / 32;
    const uint32_t g = blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5);
    if (g >= n_groups) return;
    uint32_t flag_word = 0, n_exc = 0;
    for (uint32_t rr = 0; rr < 32; rr++) {
        const uint32_t rl = 32 * g + rr;                        // read of the chunk
        if (rl >= src.count) break;
        const uint32_t L = src.len ? __ldg(src.len + rl) : src.uniform_len;
        const uint64_t o = (src.off ? __ldg(src.off + rl) : (uint64_t)(src.first + rl) * src.stride) - src.text_lo;
        uint32_t* w = words + (size_t)(src.first + rl) * slot_words;
        uint32_t read_exc = 0;
        for (uint32_t base = 0; base < 16 * slot_words; base += 256) {
            const uint32_t i0 = base + 8 * lane;
            uint32_t bits = 0, m_exc = 0, m_n, m_k3;
            if (i0 < L) pack_classify(pack_window(src.text, o, L, i0, revcomp), L, i0, tab, bits, m_exc, m_n, m_k3);
            const uint32_t other = __shfl_down_sync(0xFFFFFFFFu, bits, 1);
            const uint32_t wi = i0 >> 4;
            if (!(lane & 1) && wi < slot_words) w[wi] = bits | (other << 16);
            read_exc += __popc(m_exc);
        }
        read_exc = __reduce_add_sync(0xFFFFFFFFu, read_exc);
        if (read_exc) flag_word |= 1u << rr;
        n_exc += read_exc;
        if (lane == 0) lens[src.first + rl] = (uint16_t)L;
    }
    if (lane == 0) {
        flags[(src.first >> 5) + g] = flag_word;
        group_count[(src.first >> 5) + g] = n_exc;
    }
}

// exclusive scan of the chunk's group counts into the exception index, continuing from *carry (the entries written by
// the chunks before); one block.  index[first_group + n_groups] = the new total, which is also left in *carry.
// The list holds cap entries: the index values are clamped to cap, and a group whose run does not end inside the list
// loses its flag word, so that pass 2 writes none of its entries and no decombine kernel looks for them.  *carry keeps the
// true total (the host compares it with cap and fails the call).
__global__ void __launch_bounds__(1024)
dcb_pack_scan_kernel(const uint32_t* __restrict__ group_count, uint32_t first_group, uint32_t n_groups, uint32_t cap,
                     uint32_t* __restrict__ index, uint32_t* __restrict__ flags, uint32_t* __restrict__ carry) {
    __shared__ uint32_t warp_sum[32];
    __shared__ uint32_t running;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    if (tid == 0) running = *carry;
    __syncthreads();
    for (uint32_t base = 0; base < n_groups; base += 1024) {
        const uint32_t k = base + tid;
        const uint32_t v = k < n_groups ? group_count[first_group + k] : 0u;
        uint32_t incl = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, d);
            if (lane >= d) incl += t;
        }
        if (lane == 31) warp_sum[wid] = incl;
        __syncthreads();
        if (wid == 0) {
            uint32_t s = warp_sum[lane];
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, s, d);
                if (lane >= d) s += t;
            }
            warp_sum[lane] = s;                                // inclusive over the warps
        }
        __syncthreads();
        const uint32_t before = running + (wid ? warp_sum[wid - 1] : 0u) + incl - v;
        if (k < n_groups) {
            const uint32_t at = min(before, cap);
            index[first_group + k] = at;
            if (v > cap - at) flags[first_group + k] = 0u;        // the run crosses or lies beyond the end of the list
        }
        __syncthreads();
        if (tid == 1023) running = before + v;
        __syncthreads();
    }
    if (tid == 0) { index[first_group + n_groups] = min(running, cap); *carry = running; }
}

// pass 2: the entries of the flagged reads, in (read, position) order, at index[group] onwards
__global__ void __launch_bounds__(256)
dcb_pack_exc_kernel(PackSrc src, int revcomp, uint32_t slot_words, const uint32_t* __restrict__ flags,
                    const uint32_t* __restrict__ index, uint32_t cap, uint32_t* __restrict__ exc_read,
                    uint16_t* __restrict__ exc_pos, uint8_t* __restrict__ exc_kind) {
    __shared__ uint8_t tab[256];
    tab[threadIdx.x] = (uint8_t)pack_table_entry((int)threadIdx.x, revcomp);
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const uint32_t n_groups = (src.count + 31) / 32;
    const uint32_t g = blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5);
    if (g >= n_groups) return;
    uint32_t fw = flags[(src.first >> 5) + g];
    uint32_t at = index[(src.first >> 5) + g];
    for (; fw; fw &= fw - 1u) {
        const uint32_t rl = 32 * g + (uint32_t)__ffs(fw) - 1u;
        const uint32_t L = src.len ? __ldg(src.len + rl) : src.uniform_len;
        const uint64_t o = (src.off ? __ldg(src.off + rl) : (uint64_t)(src.first + rl) * src.stride) - src.text_lo;
        for (uint32_t base = 0; base < 16 * slot_words; base += 256) {
            const uint32_t i0 = base + 8 * lane;
            uint32_t bits, m_exc = 0, m_n = 0, m_k3 = 0;
            if (i0 < L) pack_classify(pack_window(src.text, o, L, i0, revcomp), L, i0, tab, bits, m_exc, m_n, m_k3);
            const uint32_t mine = __popc(m_exc);
            uint32_t incl = mine;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, d);
                if (lane >= d) incl += t;
            }
            uint32_t k = at + incl - mine;
            for (uint32_t m = m_exc; m; m &= m - 1u, k++) {
                const int j = __ffs(m) - 1;
                if (k < cap) {
                    exc_read[k] = src.first + rl;
                    exc_pos[k] = (uint16_t)(i0 + j);
                    exc_kind[k] = (uint8_t)(((m_k3 >> j) & 1u) ? 3u : ((m_n >> j) & 1u) ? 1u : 2u);
                }
            }
            at += __shfl_sync(0xFFFFFFFFu, incl, 31);
        }
    }
}

#endif  // DCB_PACK_DEVICE_CUH
