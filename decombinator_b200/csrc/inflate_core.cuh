// inflate_core.cuh -- an RFC 1951 (deflate) decoder with RFC 1952 (gzip) member framing, written once for host and
// device.
//
// inf_decode() inflates from a block header at any bit offset of a compressed buffer:
//   * byte mode (T = uint8_t): the window is known (a member's start); it writes bytes;
//   * marker mode (T = uint16_t, speculative): the 32 KB before the start are unknown.  It writes 16-bit symbols:
//     0..255 are bytes, 256 + w is "the byte at offset w of the 32 KB window that ends where this chunk starts".
//     Once the chunk crosses into a new gzip member the window is empty again and no further marker can appear.
// Output past `cap` is counted, not written (a match needs no data to know its length), so a chunk that outgrows
// its buffer reports its exact size for a second attempt.  It stops at the end of the last member (or, raw, of the
// final block), on landing at a block header listed in a sorted array of candidate starts, once past a bit limit,
// or on bad data -- each a status of its own.  No read or write outside the given buffers on any input: bit reads
// past the end see zeros and end in INF_E_OVERRUN, and every table index is range-checked first.
//
// inf_dyn_ok() is the start finder's test of a bit offset: a dynamic block header whose code-length code and
// literal/length and distance codes are all complete and whose end-of-block code has a length.
//
// The decode tables are strided (element i of a thread's table at i * S): the kernels keep S threads' tables
// interleaved in shared memory so that lanes reading the same element hit different banks.  Host code uses S = 1.
#ifndef DCB_INFLATE_CORE_CUH
#define DCB_INFLATE_CORE_CUH

#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
#define INF_HD __host__ __device__ __forceinline__
#else
#define INF_HD inline
#endif

enum {
    INF_END = 0,          // end of the last gzip member (zero padding after it allowed) / of the final block (raw)
    INF_LANDED = 1,       // stopped at a block header that is one of the candidate starts
    INF_LIMIT = 2,        // the bit limit was passed before either of the above
    INF_E_CODE = -1,      // a code the tables do not hold, or a length / distance symbol out of range
    INF_E_DIST = -2,      // a distance reaching before the data (a member's start, or the 32 KB window)
    INF_E_OVERRUN = -3,   // the input ended inside a block or a trailer
    INF_E_STORED = -4,    // a stored block whose LEN is not the complement of NLEN
    INF_E_TABLE = -5,     // a dynamic block header that does not describe valid codes, or BTYPE 11
    INF_E_HEADER = -6,    // a gzip member header that cannot be parsed (or garbage after a member)
    INF_E_MEMBERS = -7,   // more member ends inside one chunk than the caller has room for
};

#define INF_WINDOW 32768u
#define INF_TAB_U16 352      // lit count 16 + lit symbol 288 + dist count 16 + dist symbol 32
#define INF_TAB_U8 320       // code lengths of one dynamic header
#define INF_VTAB_U16 72      // validator: code-length count 16 + symbol 20 + lit count 16 + dist count 16 + 4 spare
#define INF_VTAB_U8 20       // validator: code-length code lengths

// ------------------------------------------------------------------------------------------------- bits
struct InfBits {
    const uint8_t* p;
    uint64_t n;        // bytes of p
    uint64_t next;     // next byte to load into buf (may pass n: zeros are loaded then)
    uint64_t buf;
    int cnt;           // valid bits in buf

    INF_HD void refill() {
        if (next + 16 <= n) {              // eight bytes in one load (two aligned words on the device)
            uint64_t v;
#if defined(__CUDA_ARCH__)
            const uint64_t* w = (const uint64_t*)((uintptr_t)(p + next) & ~(uintptr_t)7);
            const int sh = (int)((uintptr_t)(p + next) & 7) * 8;
            v = sh ? (w[0] >> sh) | (w[1] << (64 - sh)) : w[0];
#else
            memcpy(&v, p + next, 8);
#endif
            const int take = (64 - cnt) >> 3;
            buf |= v << cnt;
            cnt += take * 8;
            next += (uint64_t)take;
            if (cnt < 64) buf &= (1ull << cnt) - 1;
            return;
        }
        while (cnt <= 56) {
            const uint64_t b = next < n ? p[next] : 0;
            buf |= b << cnt;
            cnt += 8;
            next++;
        }
    }
    INF_HD void init(const uint8_t* p_, uint64_t n_, uint64_t bit) {
        p = p_; n = n_; next = bit >> 3; buf = 0; cnt = 0;
        refill();
        drop((int)(bit & 7));
    }
    INF_HD uint64_t pos() const { return next * 8 - (uint64_t)cnt; }
    INF_HD bool over() const { return pos() > n * 8; }
    INF_HD void drop(int k) { buf >>= k; cnt -= k; }
    INF_HD uint32_t get(int k) {          // k <= 32
        if (cnt < k) refill();
        const uint32_t v = (uint32_t)(buf & ((1ull << k) - 1));
        drop(k);
        return v;
    }
    INF_HD void align() { drop(cnt & 7); }
};

// ------------------------------------------------------------------------------------------------- constants
INF_HD int inf_clorder(int i) {
    return "\x10\x11\x12\x00\x08\x07\x09\x06\x0a\x05\x0b\x04\x0c\x03\x0d\x02\x0e\x01\x0f"[i];
}
// length symbol 0..28 (code 257..285): base and extra bits
INF_HD int inf_lextra(int s) { return s < 8 || s == 28 ? 0 : (s - 4) >> 2; }
INF_HD int inf_lbase(int s) { return s < 8 ? s + 3 : s == 28 ? 258 : ((4 + (s & 3)) << ((s - 4) >> 2)) + 3; }
// distance symbol 0..29
INF_HD int inf_dextra(int s) { return s < 4 ? 0 : (s - 2) >> 1; }
INF_HD int inf_dbase(int s) { return s < 4 ? s + 1 : ((2 + (s & 1)) << ((s - 2) >> 1)) + 1; }

// ------------------------------------------------------------------------------------------------- Huffman codes
// Canonical code from code lengths (RFC 1951 3.2.2): count[len] codes of each length, symbols in code order.
// -> 0 complete, > 0 incomplete, < 0 over-subscribed.  No codes at all: 0 with count[0] == n.
template <int S>
INF_HD int inf_build(uint16_t* count, uint16_t* symbol, const uint8_t* length, int n) {
    for (int len = 0; len < 16; len++) count[len * S] = 0;
    for (int s = 0; s < n; s++) count[length[s * S] * S]++;
    if (count[0] == n) return 0;
    int left = 1;
    for (int len = 1; len < 16; len++) {
        left <<= 1;
        left -= count[len * S];
        if (left < 0) return left;
    }
    // offsets of each length's first symbol, kept in symbol[] order by a running pass per length
    int off = 0;
    for (int len = 1; len < 16; len++)
        for (int s = 0; s < n; s++)
            if (length[s * S] == len) symbol[(off++) * S] = (uint16_t)s;
    return left;
}

template <int S>
INF_HD int inf_sym(InfBits& b, const uint16_t* count, const uint16_t* symbol) {
    if (b.cnt < 16) b.refill();
    uint32_t bits = (uint32_t)b.buf;
    int code = 0, first = 0, index = 0;
    for (int len = 1; len < 16; len++) {
        code |= bits & 1;
        bits >>= 1;
        const int c = count[len * S];
        if (code - c < first) {
            b.drop(len);
            return symbol[(index + (code - first)) * S];
        }
        index += c;
        first += c;
        first <<= 1;
        code <<= 1;
    }
    return -1;
}

template <int S>
struct InfTab {
    uint16_t *lc, *ls, *dc, *ds;   // literal/length count, symbols; distance count, symbols
    uint8_t* lens;                 // INF_TAB_U8 code lengths
};
// u16: INF_TAB_U16 * S elements, u8: INF_TAB_U8 * S; the thread's tables start at element `lane`.
template <int S>
INF_HD InfTab<S> inf_tab(uint16_t* u16, uint8_t* u8, int lane) {
    InfTab<S> t;
    t.lc = u16 + lane; t.ls = t.lc + 16 * S; t.dc = t.ls + 288 * S; t.ds = t.dc + 16 * S;
    t.lens = u8 + lane;
    return t;
}

template <int S>
INF_HD void inf_fixed(InfTab<S>& t) {
    for (int s = 0; s < 288; s++) t.lens[s * S] = s < 144 ? 8 : s < 256 ? 9 : s < 280 ? 7 : 8;
    inf_build<S>(t.lc, t.ls, t.lens, 288);
    for (int s = 0; s < 30; s++) t.lens[s * S] = 5;
    inf_build<S>(t.dc, t.ds, t.lens, 30);
}

// A dynamic block's header after BTYPE.  strict: every code complete (the start finder's rule); else what zlib takes
// (an incomplete literal/length or distance code only as a single code of length 1).
template <int S>
INF_HD int inf_dynamic(InfBits& b, InfTab<S>& t, bool strict) {
    const int nlen = (int)b.get(5) + 257, ndist = (int)b.get(5) + 1, ncode = (int)b.get(4) + 4;
    if (nlen > 286 || ndist > 30) return INF_E_TABLE;
    for (int i = 0; i < 19; i++) t.lens[inf_clorder(i) * S] = i < ncode ? (uint8_t)b.get(3) : 0;
    if (inf_build<S>(t.lc, t.ls, t.lens, 19) != 0 || t.lc[0] == 19) return INF_E_TABLE;
    int idx = 0;
    while (idx < nlen + ndist) {
        const int sym = inf_sym<S>(b, t.lc, t.ls);
        if (sym < 0) return INF_E_TABLE;
        if (sym < 16) {
            t.lens[(idx++) * S] = (uint8_t)sym;
        } else {
            int len = 0, rep;
            if (sym == 16) {
                if (idx == 0) return INF_E_TABLE;
                len = t.lens[(idx - 1) * S];
                rep = 3 + (int)b.get(2);
            } else if (sym == 17) {
                rep = 3 + (int)b.get(3);
            } else {
                rep = 11 + (int)b.get(7);
            }
            if (idx + rep > nlen + ndist) return INF_E_TABLE;
            while (rep--) t.lens[(idx++) * S] = (uint8_t)len;
        }
        if (b.over()) return INF_E_OVERRUN;
    }
    if (t.lens[256 * S] == 0) return INF_E_TABLE;
    int err = inf_build<S>(t.lc, t.ls, t.lens, nlen);
    if (err < 0 || (err > 0 && (strict || nlen != t.lc[0] + t.lc[S]))) return INF_E_TABLE;
    err = inf_build<S>(t.dc, t.ds, t.lens + nlen * S, ndist);
    if (err < 0 || (err > 0 && (strict || ndist != t.dc[0] + t.dc[S]))) return INF_E_TABLE;
    if (strict && t.dc[0] == ndist) return INF_E_TABLE;
    return 0;
}

// ------------------------------------------------------------------------------------------------- start finder test
template <int S>
INF_HD int inf_kraft_left(const uint16_t* count) {
    int left = 1;
    for (int len = 1; len < 16; len++) {
        left = (left << 1) - count[len * S];
        if (left < 0) return left;
    }
    return left;
}

// Is there a dynamic block header at `bit` whose three codes are complete?  Works on counts alone (no symbol tables
// for the literal/length and distance codes).  u16: INF_VTAB_U16 * S elements, u8: INF_VTAB_U8 * S; lane offsets.
template <int S>
INF_HD bool inf_dyn_ok(const uint8_t* in, uint64_t n, uint64_t bit, uint16_t* u16, uint8_t* u8, int lane) {
    if (bit + 17 > n * 8) return false;
    InfBits b;
    b.init(in, n, bit);
    b.get(1);
    if (b.get(2) != 2) return false;
    const int nlen = (int)b.get(5) + 257, ndist = (int)b.get(5) + 1, ncode = (int)b.get(4) + 4;
    if (nlen > 286 || ndist > 30) return false;
    uint16_t *cc = u16 + lane, *cs = cc + 16 * S, *lcnt = cs + 20 * S, *dcnt = lcnt + 16 * S;
    uint8_t* cl = u8 + lane;
    for (int i = 0; i < 19; i++) cl[inf_clorder(i) * S] = i < ncode ? (uint8_t)b.get(3) : 0;
    if (inf_build<S>(cc, cs, cl, 19) != 0 || cc[0] == 19) return false;
    for (int len = 0; len < 16; len++) lcnt[len * S] = dcnt[len * S] = 0;
    int idx = 0, prev = -1, eob = 0;
    while (idx < nlen + ndist) {
        const int sym = inf_sym<S>(b, cc, cs);
        int len, rep;
        if (sym < 0) return false;
        if (sym < 16) {
            len = sym; rep = 1;
        } else if (sym == 16) {
            if (prev < 0) return false;
            len = prev; rep = 3 + (int)b.get(2);
        } else {
            len = 0; rep = sym == 17 ? 3 + (int)b.get(3) : 11 + (int)b.get(7);
        }
        if (idx + rep > nlen + ndist || b.over()) return false;
        for (; rep; rep--, idx++) {
            if (idx == 256) eob = len;
            if (idx < nlen) lcnt[len * S]++;
            else dcnt[len * S]++;
        }
        prev = len;
    }
    return eob != 0 && inf_kraft_left<S>(lcnt) == 0 && dcnt[0] != ndist && inf_kraft_left<S>(dcnt) == 0;
}

// ------------------------------------------------------------------------------------------------- decoder
struct InfJob {
    const uint8_t* in;      // the whole compressed buffer
    uint64_t n;             // its bytes
    uint64_t start;         // bit offset of a block header
    uint64_t limit;         // INF_LIMIT once the bit position passes this
    const uint64_t* cand;   // sorted candidate starts (bit offsets); landing on one > start stops the decode
    uint32_t ncand;
    int gzip;               // 1: a final block ends a gzip member (trailer, then maybe another member); 0: raw deflate
    int marker;             // 1: the window before `start` is unknown (marker mode; T must be uint16_t)
    uint64_t* mend_pos;     // member ends inside the chunk: output offset, trailer CRC-32 and ISIZE (gzip only)
    uint32_t* mend_crc;
    uint32_t* mend_isize;
    uint32_t mend_cap;
    uint64_t* blocks;       // optional (tests): bit offset << 2 | BTYPE of every block header decoded
    uint32_t blocks_cap;
};

struct InfResult {
    int status;
    uint32_t landed;        // INF_LANDED: index into cand
    uint64_t produced;      // output symbols (also those past cap)
    uint64_t end_bit;       // bit position where the decode stopped
    uint32_t n_members;     // member ends recorded
    uint32_t n_blocks;
};

// Parses a gzip member header at the (byte-aligned) bit position of b.  -> 0 or INF_E_HEADER.
INF_HD int inf_gzip_header(InfBits& b) {
    if (b.get(8) != 0x1f || b.get(8) != 0x8b || b.get(8) != 8) return INF_E_HEADER;
    const uint32_t flg = b.get(8);
    if (flg & 0xe0) return INF_E_HEADER;
    b.get(16); b.get(16); b.get(16);                      // MTIME, XFL, OS
    if (flg & 4) {
        uint32_t xlen = b.get(16);
        while (xlen-- && !b.over()) b.get(8);
    }
    if (flg & 8) while (!b.over() && b.get(8) != 0) {}
    if (flg & 16) while (!b.over() && b.get(8) != 0) {}
    if (flg & 2) b.get(16);
    return b.over() ? INF_E_HEADER : 0;
}

template <typename T, int S>
INF_HD InfResult inf_decode(const InfJob& J, InfTab<S> t, T* out, uint64_t cap) {
    InfResult R;
    R.status = INF_E_OVERRUN; R.landed = 0; R.produced = 0; R.end_bit = 0; R.n_members = 0; R.n_blocks = 0;
    InfBits b;
    b.init(J.in, J.n, J.start);
    uint64_t pos = 0, mstart = 0;
    bool spec = J.marker != 0;          // distances may reach into the unknown window before the start
    const uint64_t nbits = J.n * 8;
    for (;;) {
        const uint64_t bp = b.pos();
        if (bp > nbits) { R.status = INF_E_OVERRUN; break; }
        if (bp > J.start && J.ncand) {
            uint32_t lo = 0, hi = J.ncand;
            while (lo < hi) {
                const uint32_t mid = (lo + hi) >> 1;
                if (J.cand[mid] < bp) lo = mid + 1; else hi = mid;
            }
            if (lo < J.ncand && J.cand[lo] == bp) { R.status = INF_LANDED; R.landed = lo; break; }
        }
        if (bp > J.limit) { R.status = INF_LIMIT; break; }
        const int last = (int)b.get(1), type = (int)b.get(2);
        if (J.blocks && R.n_blocks < J.blocks_cap) J.blocks[R.n_blocks] = bp << 2 | (uint64_t)type;
        R.n_blocks++;
        int st = 0;
        if (type == 0) {
            b.align();
            const uint32_t len = b.get(16), nlen = b.get(16);
            if (b.over()) { st = INF_E_OVERRUN; }
            else if (len != (~nlen & 0xffffu)) { st = INF_E_STORED; }
            else if (b.pos() / 8 + len > J.n) { st = INF_E_OVERRUN; }
            else {
                for (uint32_t i = 0; i < len; i++) {
                    const uint32_t v = b.get(8);
                    if (pos < cap) out[pos] = (T)v;
                    pos++;
                }
            }
        } else if (type == 3) {
            st = INF_E_TABLE;
        } else {
            if (type == 1) inf_fixed<S>(t);
            else st = inf_dynamic<S>(b, t, false);
            while (st == 0) {
                if (b.pos() > J.limit) { st = INF_LIMIT; break; }
                int sym = inf_sym<S>(b, t.lc, t.ls);
                if (sym < 0) { st = INF_E_CODE; break; }
                if (sym < 256) {
                    if (pos < cap) out[pos] = (T)sym;
                    pos++;
                } else if (sym == 256) {
                    break;
                } else {
                    sym -= 257;
                    if (sym >= 29) { st = INF_E_CODE; break; }
                    const uint32_t len = (uint32_t)inf_lbase(sym) + b.get(inf_lextra(sym));
                    const int ds = inf_sym<S>(b, t.dc, t.ds);
                    if (ds < 0 || ds >= 30) { st = INF_E_CODE; break; }
                    const uint64_t dist = (uint64_t)inf_dbase(ds) + b.get(inf_dextra(ds));
                    if (dist > pos - mstart && !spec) { st = INF_E_DIST; break; }
                    if (dist > pos + INF_WINDOW) { st = INF_E_DIST; break; }
                    for (uint32_t i = 0; i < len; i++, pos++) {
                        if (pos >= cap) { pos += len - i; break; }
                        uint32_t v;
                        if (dist > pos) v = 256u + (uint32_t)(INF_WINDOW + pos - dist);   // marker (spec only)
                        else v = out[pos - dist];
                        out[pos] = (T)v;
                    }
                }
                if (b.over()) { st = INF_E_OVERRUN; break; }
            }
        }
        if (st) { R.status = st; break; }
        if (!last) continue;
        if (!J.gzip) { R.status = INF_END; break; }
        // end of a member: trailer, zero padding, then the end of the input or the next member's header
        b.align();
        const uint32_t crc = b.get(16) | b.get(16) << 16;
        const uint32_t isize = b.get(16) | b.get(16) << 16;
        if (b.over()) { R.status = INF_E_OVERRUN; break; }
        if (R.n_members >= J.mend_cap) { R.status = INF_E_MEMBERS; break; }
        J.mend_pos[R.n_members] = pos; J.mend_crc[R.n_members] = crc; J.mend_isize[R.n_members] = isize;
        R.n_members++;
        while (b.pos() < nbits) {
            if (b.cnt < 8) b.refill();
            if ((b.buf & 0xff) != 0) break;
            b.drop(8);
        }
        if (b.pos() >= nbits) { R.status = INF_END; break; }
        if (inf_gzip_header(b)) { R.status = INF_E_HEADER; break; }
        mstart = pos;
        spec = false;
    }
    R.produced = pos;
    R.end_bit = b.pos();
    return R;
}

// Symbol of marker mode -> byte, given the chunk's resolved window (INF_WINDOW bytes ending at the chunk's start).
INF_HD uint8_t inf_resolve(uint16_t v, const uint8_t* window) { return v < 256 ? (uint8_t)v : window[v - 256]; }

// ------------------------------------------------------------------------------------------------- chain
// Follows "landed on" from chunk 0: chain[0..m) are the chunks kept.  -> m, or 0 when a chunk on the chain ended in
// anything but INF_LANDED / INF_END (its status in *bad, its index in *bad_chunk).  status / landed per chunk.
static inline uint32_t inf_chain(const int* status, const uint32_t* landed, uint32_t n, uint32_t* chain, int* bad,
                                 uint32_t* bad_chunk) {
    uint32_t m = 0, k = 0;
    *bad = 0;
    for (;;) {
        if (k >= n) { *bad = INF_E_CODE; *bad_chunk = k; return 0; }
        chain[m++] = k;
        if (status[k] == INF_END) return m;
        if (status[k] != INF_LANDED || landed[k] <= k) { *bad = status[k] == INF_LANDED ? INF_E_CODE : status[k]; *bad_chunk = k; return 0; }
        k = landed[k];
    }
}

// ------------------------------------------------------------------------------------------------- CRC-32
INF_HD uint32_t inf_crc_entry(uint32_t i) {
    uint32_t c = i;
    for (int k = 0; k < 8; k++) c = c & 1 ? 0xedb88320u ^ (c >> 1) : c >> 1;
    return c;
}
// zlib's crc32(crc, p, n) with a 256-entry table
INF_HD uint32_t inf_crc32(uint32_t crc, const uint8_t* p, uint64_t n, const uint32_t* table) {
    crc = ~crc;
    for (uint64_t i = 0; i < n; i++) crc = table[(crc ^ p[i]) & 0xff] ^ (crc >> 8);
    return ~crc;
}
// a(x) * b(x) modulo the CRC-32 polynomial, reflected (zlib's multmodp)
INF_HD uint32_t inf_multmodp(uint32_t a, uint32_t b) {
    uint32_t m = 1u << 31, p = 0;
    for (;;) {
        if (a & m) {
            p ^= b;
            if ((a & (m - 1)) == 0) break;
        }
        m >>= 1;
        b = b & 1 ? (b >> 1) ^ 0xedb88320u : b >> 1;
    }
    return p;
}
// x^(8 * len) modulo the polynomial: what appending len bytes does to a CRC
INF_HD uint32_t inf_crc_shift(uint64_t len) {
    uint32_t p = 1u << 31, t = 1u << 30;          // x^0, x^1
    for (int k = 0; k < 3; k++) t = inf_multmodp(t, t);
    while (len) {
        if (len & 1) p = inf_multmodp(t, p);
        len >>= 1;
        t = inf_multmodp(t, t);
    }
    return p;
}
// crc32(A + B) from crc32(A), crc32(B) and len(B) (zlib's crc32_combine); `shift` = inf_crc_shift(len(B))
INF_HD uint32_t inf_crc_combine(uint32_t crc_a, uint32_t crc_b, uint32_t shift) { return inf_multmodp(shift, crc_a) ^ crc_b; }

#endif
