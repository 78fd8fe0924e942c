// Host build of csrc/translate_core.cuh (tests/test_translate_sim.py): one row at a time, as the kernels of
// csrc/translate.cu size and write it, over the table blob of dcb_translate_tables_blob.
#include "../../decombinator_b200/csrc/translate_core.cuh"

#include <stdint.h>

extern "C" {

// -> length of the row's .tsv line written to out (cap bytes), 0 with *flags != 0 (the row is the host's), -1: cap too small.
// productive / flags as the size kernel reports them; plain: the decombinator_id check of the size kernel.
long sim_translate_row(const uint8_t* blob, uint32_t v, uint32_t j, uint32_t vdel, uint32_t jdel, const uint8_t* ins, int il,
                       const uint8_t* id, int id_len, int64_t seq_id, int64_t freq, int64_t cluster, int nbc, char* out, long cap,
                       int* flags, int* productive) {
    const TrTables t = tr_tables(blob);
    TrRow r;
    tr_row(t, v, j, vdel, jdel, ins, il, r);
    if (!tr_plain(id, id_len)) r.flags |= TR_F_QUOTE;
    *flags = r.flags;
    *productive = r.productive;
    if (r.flags) return 0;
    TrLine L;
    L.seq_id = seq_id; L.freq = freq; L.cluster = cluster; L.nbc = nbc != 0; L.id = id; L.id_len = id_len;
    const uint64_t n = tr_line_len(t, r, L, v, j);
    if ((long)n > cap) return -1;
    char* end = tr_write(t, r, L, v, j, out);
    return (long)(end - out) == (long)n ? (long)n : -2;
}

}
