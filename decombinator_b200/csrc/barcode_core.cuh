// barcode_core.cuh -- barcode extraction of one decombined row, written once for host and device.
//
// What collapse.py does per row before any grouping (get_barcode_positions, collapse.py:367-479): an 'N' anywhere rejects
// the row (unless -N); spacer 1 is searched in its window bc[lo:hi] and must be found exactly once.  Then, per layout of
// the ligation oligo:
//   two spacers (M13, I8): window bc[0 : 10 + len(spacer1)]; spacer 2 is searched in bc[len(spacer1):] and must be found
//     exactly once; N1 lies between the spacers, N2 is the six bases behind spacer 2;
//   N1, spacer, N2 (I8_single): window bc[0:18]; N1 is bc[0 : spacer position], N2 the six bases behind the spacer;
//     for both: N1 of <= 3 or >= 9 bases and an N2 that runs past the end reject the row, and set_barcode (:281-326)
//     makes N1 + N2, a short N1 padded with 'S' (quality '?'), a long one cut to five bases + 'L';
//   fixed barcode (NEBIO: window bc[18:28], barcode bc[0:17]; TAKARA: window bc[0:19], barcode bc[0:12]): the spacer only
//     has to be there, its position is not used.
// check_umi_quality (:340-352): more than `max_below` barcode qualities under `min_q`, or a mean under `avg_q`, rejects the row.
//
// Each spacer search is spacerSearch (:147-153): regex.findall of the spacer, and only when that finds nothing
// {1s<=2}, and only when that finds nothing {2i+2d+1s<=2}; the first non-empty list decides.  With FUZZY false only the
// exact stage runs and a row it finds nothing for is handed back (DCB_BC_HOST).  The fuzzy stages as regex runs them
// (pinned against it by tests/test_barcode_sim.py, case by case):
//   {1s<=2}         leftmost, non-overlapping windows of the spacer's length within Hamming distance 2;
//   {2i+2d+1s<=2}   reached only when no such window exists in the range, which leaves one deleted spacer base or one
//                   inserted base and no substitution: leftmost start, a deletion at any spacer position, an insertion
//                   only between two spacer bases, non-overlapping.
// Where N1 and N2 lie does not come from where the search matched but from str.find of the matched TEXT with a running
// offset (getSpacerPositions, :166-172): text 1 from 0, text 2 from len(text 1), which for a fuzzy spacer 1 of another
// length than the oligo's can find a later occurrence of text 2, or none (-1).  Kept as the host does it.
// Rows with symbols outside ACGTN, a quality string of another length or a region longer than 250 are always handed back,
// and so are fixed-barcode regions shorter than the barcode (the reference would cut the barcode short) whose spacer the
// search finds: without the fuzzy stages before any search, with them once the search has found it (NEBIO's window starts
// behind its 17-symbol barcode, so such a region of NEBIO is always DCB_BC_FAIL_NOSPACER).
#ifndef DCB_BARCODE_CORE_CUH
#define DCB_BARCODE_CORE_CUH

#include "../../include/dcb.h"

#include <stdint.h>

#if defined(__CUDACC__)
#define BC_HD __host__ __device__ __forceinline__
#else
#define BC_HD inline
#endif

enum { BC_TWO_SPACERS = 0, BC_N1_SPACER_N2 = 1, BC_FIXED = 2 };   // BcParams::layout
struct BcParams { char sp1[32], sp2[32]; int layout, lo, hi, bclen, len1, len2, allow_ns, min_q, max_below; double avg_q; };

// spacers, window of spacer 1 and barcode length per design (collapse.py:172-189, 367-479); false: not a DCB_OLIGO_*
inline bool bc_params(const dcb_bc_params& prm, BcParams& P) {
    P = BcParams{};
    const char *sp1, *sp2 = "";
    switch (prm.oligo) {
    case DCB_OLIGO_M13:       sp1 = "GTCGTGACTGGGAAAACCCTGG"; sp2 = "GTCGTGAT"; P.layout = BC_TWO_SPACERS; break;
    case DCB_OLIGO_I8:        sp1 = "GTCGTGAT"; sp2 = "GTCGTGAT"; P.layout = BC_TWO_SPACERS; break;
    case DCB_OLIGO_I8_SINGLE: sp1 = "ATCACGAC"; P.layout = BC_N1_SPACER_N2; break;
    case DCB_OLIGO_NEBIO:     sp1 = "TACGGG"; P.layout = BC_FIXED; P.lo = 18; P.hi = 28; P.bclen = 17; break;
    case DCB_OLIGO_TAKARA:    sp1 = "GTACGGG"; P.layout = BC_FIXED; P.lo = 0; P.hi = 19; P.bclen = 12; break;
    default: return false;
    }
    while (sp1[P.len1]) { P.sp1[P.len1] = sp1[P.len1]; P.len1++; }
    while (sp2[P.len2]) { P.sp2[P.len2] = sp2[P.len2]; P.len2++; }
    if (P.layout != BC_FIXED) { P.lo = 0; P.hi = 10 + P.len1; P.bclen = 12; }
    P.allow_ns = prm.allow_ns; P.min_q = prm.min_q; P.max_below = prm.max_below; P.avg_q = prm.avg_q;
    return true;
}

// first occurrence of pat[0:plen] in s[from:to), -1 if none (str.find; regex.findall steps through these)
BC_HD int bc_find(const unsigned char* s, int from, int to, const unsigned char* pat, int plen) {
    for (int p = from; p + plen <= to; p++) {
        int k = 0;
        while (k < plen && s[p + k] == pat[k]) k++;
        if (k == plen) return p;
    }
    return -1;
}
BC_HD int bc_count(const unsigned char* s, int from, int to, const unsigned char* pat, int plen, int& first) {
    int n = 0;
    first = -1;
    for (int p = bc_find(s, from, to, pat, plen); p >= 0; p = bc_find(s, p + plen, to, pat, plen)) { if (!n) first = p; n++; }
    return n;
}
// t[0:L-1] is pat[0:L] with one symbol deleted: a common prefix and a common suffix that together cover the text
BC_HD bool bc_one_deletion(const unsigned char* t, const unsigned char* pat, int L) {
    int a = 0, b = 0;
    while (a < L - 1 && t[a] == pat[a]) a++;
    while (b < L - 1 && t[L - 2 - b] == pat[L - 1 - b]) b++;
    return a + b >= L - 1;
}
// t[0:L+1] is pat[0:L] with one symbol inserted at k, 1 <= k <= L - 1 (not before the first base nor after the last)
BC_HD bool bc_one_insertion(const unsigned char* t, const unsigned char* pat, int L) {
    int a = 0, b = 0;
    while (a < L && t[a] == pat[a]) a++;
    while (b < L && t[L - b] == pat[L - 1 - b]) b++;
    const int k_lo = L - b > 1 ? L - b : 1, k_hi = a < L - 1 ? a : L - 1;
    return k_lo <= k_hi;
}

struct BcHits {
    int n;        // hits of the stage that decided (0: none in any stage)
    int at, len;  // first hit: start and length of the matched text
    bool fuzzy;   // decided by {1s<=2} or {2i+2d+1s<=2}: the matched text differs from the spacer
};
template <bool FUZZY>
BC_HD void bc_search(const unsigned char* s, int from, int to, const unsigned char* pat, int plen, BcHits& h) {
    h.n = bc_count(s, from, to, pat, plen, h.at);
    h.len = plen;
    h.fuzzy = false;
    if (!FUZZY || h.n) return;
    h.fuzzy = true;
    for (int p = from; p + plen <= to;) {                                    // {1s<=2}
        int miss = 0;
        for (int k = 0; k < plen && miss <= 2; k++) miss += s[p + k] != pat[k];
        if (miss <= 2) { if (!h.n) h.at = p; h.n++; p += plen; }
        else p++;
    }
    if (h.n) return;
    for (int p = from; p + plen - 1 <= to;) {                                // {2i+2d+1s<=2}
        int len = 0;
        if (bc_one_deletion(s + p, pat, plen)) len = plen - 1;
        else if (p + plen + 1 <= to && bc_one_insertion(s + p, pat, plen)) len = plen + 1;
        if (len) { if (!h.n) { h.at = p; h.len = len; } h.n++; p += len; }
        else p++;
    }
}

struct BcRow { uint8_t status, n1len, match; uint64_t code; };

// One row: s[0:L] the barcode region, q[0:qlen] its quality string.  -> status (DCB_BC_*), n1len, code as dcb_barcodes
// reports them; match = 1 when a placed row (DCB_BC_OK, DCB_BC_FAIL_QUALITY) took a fuzzy text for either spacer.
template <bool FUZZY>
BC_HD BcRow bc_row(const unsigned char* s, int L, const unsigned char* q, int qlen, const BcParams& P) {
    BcRow r;
    r.status = DCB_BC_HOST; r.n1len = 0; r.match = 0; r.code = 0;
    if (L > 250 || qlen != L) return r;
    bool has_n = false, odd = false;
    for (int p = 0; p < L; p++) {
        const unsigned char c = s[p];
        has_n |= c == 'N';
        odd |= !(c == 'A' || c == 'C' || c == 'G' || c == 'T' || c == 'N');
    }
    if (has_n && !P.allow_ns) { r.status = DCB_BC_FAIL_N; return r; }                      // collapse.py:388-392
    const bool cut_short = P.layout == BC_FIXED && L < P.bclen;          // the reference would cut the barcode short
    if (odd || (!FUZZY && cut_short)) return r;
    const unsigned char* sp1 = (const unsigned char*)P.sp1;
    const unsigned char* sp2 = (const unsigned char*)P.sp2;
    const int hi = L < P.hi ? L : P.hi;
    BcHits h1, h2;
    bc_search<FUZZY>(s, P.lo, hi, sp1, P.len1, h1);                                          // :405-413
    if (!FUZZY && h1.n == 0) return r;                                                       // the fuzzy searches decide
    if (h1.n != 1) { r.status = DCB_BC_FAIL_NOSPACER; return r; }
    if (cut_short) return r;
    // the barcode symbols (A C G T N S L = 0..6) and their qualities
    uint64_t cd = (uint64_t)P.bclen << 58;
    int qsum = 0, qn = 0, below = 0, k = 0;
    auto sym = [](unsigned char c) -> uint64_t { return c == 'A' ? 0 : c == 'C' ? 1 : c == 'G' ? 2 : c == 'T' ? 3 : 4; };
    auto addq = [&](int v) { qsum += v; qn++; below += v < P.min_q; };
    bool fuzzy = h1.fuzzy;
    if (P.layout == BC_FIXED) {                                                             // set_barcode: bc[0:bclen], q[0:bclen]
        for (; k < P.bclen; k++) { cd |= sym(s[k]) << (3 * k); addq((int)q[k] - 33); }
    } else {
        int w0 = h1.at, w1 = -1;
        if (P.layout == BC_TWO_SPACERS) {
            bc_search<FUZZY>(s, P.len1, L, sp2, P.len2, h2);                                 // :417-422
            if (!FUZZY && h2.n == 0) return r;
            if (h2.n != 1) { r.status = DCB_BC_FAIL_NOT2; return r; }
            w1 = h2.at;
            fuzzy |= h2.fuzzy;
        }
        if (fuzzy) {                                                                         // getSpacerPositions
            w0 = bc_find(s, 0, L, s + h1.at, h1.len);
            if (P.layout == BC_TWO_SPACERS) w1 = bc_find(s, h1.len, L, s + h2.at, h2.len);
        }
        int b1s = 0, b1e = w0, b2s = w0 + h1.len;                                           // I8_single: N1, spacer, N2
        if (P.layout == BC_TWO_SPACERS) { b1s = w0 + h1.len; b1e = w1; b2s = w1 + h2.len; }
        const int b2e = b2s + 6, n1 = b1e - b1s;
        if (n1 <= 3) { r.status = DCB_BC_FAIL_N1SHORT; return r; }                          // :241-254
        if (n1 >= 9) { r.status = DCB_BC_FAIL_N1LONG; return r; }
        if (b2e > L) { r.status = DCB_BC_FAIL_N2END; return r; }
        r.n1len = (uint8_t)n1;
        // 12 symbols; a long N1 has no pad quality (11 values)
        const int take1 = n1 > 6 ? 5 : n1;
        for (int p = 0; p < take1; p++, k++) { cd |= sym(s[b1s + p]) << (3 * k); addq((int)q[b1s + p] - 33); }
        if (n1 < 6) for (int p = n1; p < 6; p++, k++) { cd |= 5ull << (3 * k); addq('?' - 33); }   // 'S', quality '?'
        if (n1 > 6) { cd |= 6ull << (3 * k); k++; }                                               // 'L'; "?" * (6 - n1) is empty
        for (int p = 0; p < 6; p++, k++) { cd |= sym(s[b2s + p]) << (3 * k); addq((int)q[b2s + p] - 33); }
    }
    r.code = cd;
    r.match = fuzzy ? 1 : 0;
    const bool bad_q = below > P.max_below || (double)qsum / (double)qn < P.avg_q;            // :350-352
    r.status = bad_q ? DCB_BC_FAIL_QUALITY : DCB_BC_OK;
    return r;
}

#endif
