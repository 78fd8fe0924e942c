// translate_core.cuh -- one row of the translate stage, written once for host and device.
//
// Replaces get_cdr3 (decombinator_b200/translate.py; reference translate.py:257-357) for one DCR: rebuild the
// nucleotide sequence from the germline regions (V minus vdel, the insert, J minus jdel), translate it with the
// standard table (Bio.Seq.translate semantics), and run the frame, stop, conserved-C and J-motif checks.  Every quirk
// of the host code is kept: Python slice rules for the deletions and the junction slices, Python indexing for the
// conserved residue (position 0 reads the LAST residue), the in-frame test (len(seq) - 1) % 3 == 0, findall on the
// motif window.  The kernels (translate.cu) size a row's .tsv line with tr_row() and write it with tr_write(); tests/sim
// compiles this header for the host and compares it with get_cdr3 field for field.
#ifndef DCB_TRANSLATE_CORE_CUH
#define DCB_TRANSLATE_CORE_CUH

#include <stdint.h>

#if defined(__CUDACC__)
#define TR_HD __host__ __device__ __forceinline__
#else
#define TR_HD inline
#endif

#define DCB_TR_MAX_SEQ 1024        // longest rebuilt nucleotide sequence the device path takes (DESIGN §7)
#define DCB_TR_MAGIC 0x54524331u   // "TRC1"

// Row flags: the row is outside the device path's envelope (the whole call then takes the host path).
// (the DCB_TR_* values of include/dcb.h)
enum {
    TR_F_SYMBOL = 1,     // insert byte outside IUPAC / U (either case): the host may raise ValueError
    TR_F_GENE = 2,       // v or j out of range: the host raises IndexError
    TR_F_CINDEX = 4,     // conserved-C index beyond the protein: the host raises IndexError
    TR_F_QUOTE = 8,      // decombinator_id holds a byte to_csv would quote (or a control / non-ASCII byte)
    TR_F_LONG = 16,      // rebuilt sequence longer than DCB_TR_MAX_SEQ
};

// Per gene record of the table blob.  Strings live in the blob's pool (offsets from the pool's start).
struct TrGene {
    uint32_t region_off, call_off, cdr1_off, cdr2_off;
    uint16_t region_len, call_len, cdr1_len, cdr2_len;
    int32_t pos;          // v: conserved-C position; j: motif window start (negative)
    uint8_t res[4];       // v: residue in res[0] (0: never matches); j: motif, '.' = any residue
};

// Blob: TrHeader, TrGene[n_v], TrGene[n_j], codon table (4096 bytes), pool.  16-byte aligned sections.
struct TrHeader {
    uint32_t magic, n_v, n_j, genes_off, codon_off, pool_off, bytes, pad;
};

struct TrTables {
    const TrGene* v;
    const TrGene* j;
    const uint8_t* codon;   // [m1 << 8 | m2 << 4 | m3] for 4-bit IUPAC masks (A=1 C=2 G=4 T=8)
    const uint8_t* pool;
    uint32_t n_v, n_j;
};

TR_HD TrTables tr_tables(const uint8_t* blob) {
    const TrHeader* h = (const TrHeader*)blob;
    TrTables t;
    t.v = (const TrGene*)(blob + h->genes_off);
    t.j = t.v + h->n_v;
    t.codon = blob + h->codon_off;
    t.pool = blob + h->pool_off;
    t.n_v = h->n_v;
    t.n_j = h->n_j;
    return t;
}

// 4-bit IUPAC mask of a nucleotide symbol after upper-casing ('U' counts as 'T'); 0 for anything else.
TR_HD uint32_t tr_mask(uint32_t c) {
    if (c >= 'a' && c <= 'z') c -= 32;
    switch (c) {
    case 'A': return 1; case 'C': return 2; case 'G': return 4; case 'T': case 'U': return 8;
    case 'R': return 5; case 'Y': return 10; case 'S': return 6; case 'W': return 9; case 'K': return 12; case 'M': return 3;
    case 'B': return 14; case 'D': return 13; case 'H': return 11; case 'V': return 7; case 'N': return 15;
    default: return 0;
    }
}

// Python's s[a:b] on a sequence of length n -> [*s, *e) (e >= s)
TR_HD void tr_slice(int n, int a, int b, int& s, int& e) {
    if (a < 0) { a += n; if (a < 0) a = 0; } else if (a > n) a = n;
    if (b < 0) { b += n; if (b < 0) b = 0; } else if (b > n) b = n;
    s = a;
    e = b < a ? a : b;
}

// One row: the rebuilt sequence is V[0:vl] + insert + J[js:js + jl]
struct TrRow {
    const uint8_t* vseq;
    const uint8_t* jseq;
    const uint8_t* ins;
    int vl, il, js, jl, len, naa;
    int flags;
    bool in_frame, stop, c_ok, f_ok, productive;
    int start, end;        // start_cdr3 / end_cdr3 as the host computes them (Python values, start may be -1)
};

TR_HD uint32_t tr_base(const TrRow& r, int p) {
    if (p < r.vl) return r.vseq[p];
    p -= r.vl;
    if (p < r.il) return r.ins[p];
    return r.jseq[r.js + p - r.il];
}

TR_HD uint32_t tr_codon(const TrTables& t, const TrRow& r, int k) {
    const uint32_t m = (tr_mask(tr_base(r, 3 * k)) << 8) | (tr_mask(tr_base(r, 3 * k + 1)) << 4) | tr_mask(tr_base(r, 3 * k + 2));
    return t.codon[m];
}

// Everything get_cdr3 decides for a row.  On return r.flags != 0 means the host must take the row.
TR_HD void tr_row(const TrTables& t, uint32_t v, uint32_t j, uint32_t vdel, uint32_t jdel, const uint8_t* ins, int il, TrRow& r) {
    r.flags = 0;
    r.in_frame = r.stop = r.c_ok = r.f_ok = r.productive = false;
    r.start = r.end = 0;
    r.len = r.naa = 0;
    if (v >= t.n_v || j >= t.n_j) { r.flags = TR_F_GENE; return; }
    const TrGene& gv = t.v[v];
    const TrGene& gj = t.j[j];
    r.vseq = t.pool + gv.region_off;
    r.jseq = t.pool + gj.region_off;
    r.ins = ins;
    r.il = il;
    const int lv = gv.region_len, lj = gj.region_len;
    r.vl = vdel == 0 ? lv : (vdel >= (uint32_t)lv ? 0 : lv - (int)vdel);        // region[:-vdel]
    r.js = jdel >= (uint32_t)lj ? lj : (int)jdel;                                 // region[jdel:]
    r.jl = lj - r.js;
    for (int p = 0; p < il; p++)
        if (tr_mask(ins[p]) == 0) r.flags |= TR_F_SYMBOL;
    if (il > DCB_TR_MAX_SEQ || r.vl + il + r.jl > DCB_TR_MAX_SEQ) r.flags |= TR_F_LONG;
    if (r.flags) return;
    r.len = r.vl + il + r.jl;
    r.naa = r.len / 3;
    const int n = r.naa;
    r.in_frame = r.len % 3 == 1;
    for (int k = 0; k < n && !r.stop; k++) r.stop = tr_codon(t, r, k) == '*';
    // conserved C: aa[pos - 1] under Python indexing
    int idx = gv.pos - 1;
    if (idx < 0) idx += n;
    if (idx < 0 || idx >= n) { r.flags = TR_F_CINDEX; return; }
    r.c_ok = gv.res[0] != 0 && tr_codon(t, r, idx) == gv.res[0];
    r.start = r.c_ok ? gv.pos - 1 : 0;
    // J motif: findall(motif, downstream[jp:jp + 4]) with downstream = aa[start:]
    int ds, de;
    tr_slice(n, r.start, n, ds, de);
    const int dlen = de - ds;
    int ws, we;
    tr_slice(dlen, gj.pos, gj.pos + 4, ws, we);
    if (we - ws == 4) {
        bool ok = true;
        for (int q = 0; q < 4 && ok; q++) ok = gj.res[q] == '.' || tr_codon(t, r, ds + ws + q) == gj.res[q];
        r.f_ok = ok;
    }
    if (r.f_ok) r.end = dlen + gj.pos + r.start + 1;
    r.productive = r.in_frame && !r.stop && r.c_ok && r.f_ok;
}

// ------------------------------------------------------------------------------------------------
// The .tsv line (DataFrame.to_csv(sep="\t", index=False) of the host's row): 24 fields, '\n' at the end.
// ------------------------------------------------------------------------------------------------
TR_HD int tr_int_len(int64_t x) {
    uint64_t u = x < 0 ? (uint64_t)0 - (uint64_t)x : (uint64_t)x;
    int n = x < 0 ? 2 : 1;
    while (u >= 10) { u /= 10; n++; }
    return n;
}

TR_HD char* tr_put_int(char* o, int64_t x) {
    uint64_t u = x < 0 ? (uint64_t)0 - (uint64_t)x : (uint64_t)x;
    if (x < 0) *o++ = '-';
    char tmp[20];
    int n = 0;
    do { tmp[n++] = (char)('0' + u % 10); u /= 10; } while (u);
    while (n) *o++ = tmp[--n];
    return o;
}

TR_HD char* tr_put(char* o, const uint8_t* s, int n) {
    for (int i = 0; i < n; i++) o[i] = (char)s[i];
    return o + n;
}

struct TrLine {
    int64_t seq_id, freq, cluster;
    bool nbc;                     // -nbc: duplicate_count 1, empty av_UMI_cluster_size
    const uint8_t* id;            // decombinator_id
    int id_len;
};

// Length of the row's line; r must be a row without flags.
TR_HD uint64_t tr_line_len(const TrTables& t, const TrRow& r, const TrLine& L, uint32_t v, uint32_t j) {
    const TrGene& gv = t.v[v];
    const TrGene& gj = t.j[j];
    uint64_t n = 23 + 1;                                            // 23 tabs + '\n'
    n += tr_int_len(L.seq_id) + gv.call_len + gj.call_len;
    n += L.nbc ? 1 : tr_int_len(L.freq);
    n += r.len + L.id_len + 1 + 1 + r.naa + 1 + 1 + 1 + 1;          // sequence .. conserved_f (one-letter flags)
    n += L.nbc ? 0 : tr_int_len(L.cluster);
    if (r.productive) {
        int s, e;
        tr_slice(r.naa, r.start, r.end, s, e);
        n += e - s;
        tr_slice(r.len, 3 * r.start, 3 * r.end, s, e);
        n += e - s;
        n += gv.cdr1_len + gv.cdr2_len;
    }
    return n;
}

TR_HD char* tr_put_aa(const TrTables& t, const TrRow& r, char* o, int s, int e) {
    for (int k = s; k < e; k++) *o++ = (char)tr_codon(t, r, k);
    return o;
}

TR_HD char* tr_put_nt(const TrRow& r, char* o, int s, int e) {
    for (int p = s; p < e; p++) *o++ = (char)tr_base(r, p);
    return o;
}

// Writes the line at o; returns the end.
TR_HD char* tr_write(const TrTables& t, const TrRow& r, const TrLine& L, uint32_t v, uint32_t j, char* o) {
    const TrGene& gv = t.v[v];
    const TrGene& gj = t.j[j];
    int as = 0, ae = 0, ns = 0, ne = 0;
    if (r.productive) {
        tr_slice(r.naa, r.start, r.end, as, ae);
        tr_slice(r.len, 3 * r.start, 3 * r.end, ns, ne);
    }
    o = tr_put_int(o, L.seq_id); *o++ = '\t';                                  // sequence_id
    o = tr_put(o, t.pool + gv.call_off, gv.call_len); *o++ = '\t';             // v_call
    *o++ = '\t';                                                               // d_call
    o = tr_put(o, t.pool + gj.call_off, gj.call_len); *o++ = '\t';             // j_call
    o = tr_put_aa(t, r, o, as, ae); *o++ = '\t';                               // junction_aa
    o = tr_put_int(o, L.nbc ? 1 : L.freq); *o++ = '\t';                        // duplicate_count
    o = tr_put_nt(r, o, 0, r.len); *o++ = '\t';                                // sequence
    o = tr_put_nt(r, o, ns, ne); *o++ = '\t';                                  // junction
    o = tr_put(o, L.id, L.id_len); *o++ = '\t';                                // decombinator_id
    *o++ = 'F'; *o++ = '\t';                                                   // rev_comp
    *o++ = r.productive ? 'T' : 'F'; *o++ = '\t';                              // productive
    o = tr_put_aa(t, r, o, 0, r.naa); *o++ = '\t';                             // sequence_aa
    if (r.productive) o = tr_put(o, t.pool + gv.cdr1_off, gv.cdr1_len);
    *o++ = '\t';                                                               // cdr1_aa
    if (r.productive) o = tr_put(o, t.pool + gv.cdr2_off, gv.cdr2_len);
    *o++ = '\t';                                                               // cdr2_aa
    *o++ = r.in_frame ? 'T' : 'F'; *o++ = '\t';
    *o++ = r.stop ? 'T' : 'F'; *o++ = '\t';
    *o++ = r.c_ok ? 'T' : 'F'; *o++ = '\t';
    *o++ = r.f_ok ? 'T' : 'F'; *o++ = '\t';
    for (int k = 0; k < 5; k++) *o++ = '\t';                                   // five empty alignment / cigar fields
    if (!L.nbc) o = tr_put_int(o, L.cluster);                                  // av_UMI_cluster_size
    *o++ = '\n';
    return o;
}

// decombinator_id bytes the .tsv can hold verbatim: printable ASCII other than '"' (to_csv quotes '"', '\t', '\r', '\n')
TR_HD bool tr_plain(const uint8_t* s, int n) {
    for (int i = 0; i < n; i++)
        if (s[i] < 0x20 || s[i] >= 0x7F || s[i] == '"') return false;
    return true;
}

#endif  // DCB_TRANSLATE_CORE_CUH
