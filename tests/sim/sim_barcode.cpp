// Host build of csrc/barcode_core.cuh (tests/test_barcode_sim.py): one row at a time, as dcb_barcodes_kernel runs it.
#include "../../decombinator_b200/csrc/barcode_core.cuh"

#include <stdint.h>

extern "C" {

// -> 0, or -1 for an oligo without a device path; status / n1len / code / match as dcb_barcodes_fuzzy reports them.
int sim_barcode_row(int oligo, int allow_ns, int min_q, int max_below, double avg_q, int fuzzy, const char* bc, int len,
                    const char* q, int qlen, uint8_t* status, uint8_t* n1len, uint64_t* code, uint8_t* match) {
    const dcb_bc_params prm = {oligo, allow_ns, min_q, max_below, avg_q};
    BcParams P;
    if (!bc_params(prm, P)) return -1;
    const unsigned char* s = (const unsigned char*)bc;
    const unsigned char* qq = (const unsigned char*)q;
    const BcRow r = fuzzy ? bc_row<true>(s, len, qq, qlen, P) : bc_row<false>(s, len, qq, qlen, P);
    *status = r.status; *n1len = r.n1len; *code = r.code; *match = r.match;
    return 0;
}

// bc_one_deletion (insertion == 0: t holds L - 1 symbols) or bc_one_insertion (insertion != 0: L + 1 symbols) of t against pat[0:L]
int sim_one_edit(int insertion, const char* t, const char* pat, int L) {
    const unsigned char* tt = (const unsigned char*)t;
    const unsigned char* pp = (const unsigned char*)pat;
    return insertion ? bc_one_insertion(tt, pp, L) : bc_one_deletion(tt, pp, L);
}

}
