// Host build of csrc/inflate_core.cuh (tests/test_inflate_sim.py): one decoder at a time, as the kernels of
// csrc/inflate.cu run it, with the tables in plain host arrays (stride 1).
#include "../../decombinator_b200/csrc/inflate_core.cuh"

#include <stdint.h>
#include <stdlib.h>
#include <vector>

extern "C" {

// res: status, landed, produced, end_bit, n_members, n_blocks.  marker != 0: out is uint16_t symbols, else bytes.
// Buffers of exactly the sizes given (cap elements, mend_cap / blocks_cap entries) so that the sanitizer build sees any
// access beyond them.
int sim_inflate(const uint8_t* in, uint64_t n, uint64_t start, uint64_t limit, const uint64_t* cand, uint32_t ncand, int gzip,
                int marker, void* out, uint64_t cap, uint64_t* mend_pos, uint32_t* mend_crc, uint32_t* mend_isize, uint32_t mend_cap,
                uint64_t* blocks, uint32_t blocks_cap, uint64_t* res) {
    std::vector<uint16_t> u16(INF_TAB_U16);
    std::vector<uint8_t> u8(INF_TAB_U8);
    InfTab<1> t = inf_tab<1>(u16.data(), u8.data(), 0);
    InfJob J;
    J.in = in; J.n = n; J.start = start; J.limit = limit; J.cand = cand; J.ncand = ncand; J.gzip = gzip; J.marker = marker;
    J.mend_pos = mend_pos; J.mend_crc = mend_crc; J.mend_isize = mend_isize; J.mend_cap = mend_cap;
    J.blocks = blocks; J.blocks_cap = blocks_cap;
    const InfResult R = marker ? inf_decode<uint16_t, 1>(J, t, (uint16_t*)out, cap) : inf_decode<uint8_t, 1>(J, t, (uint8_t*)out, cap);
    res[0] = (uint64_t)(int64_t)R.status; res[1] = R.landed; res[2] = R.produced; res[3] = R.end_bit; res[4] = R.n_members;
    res[5] = R.n_blocks;
    return R.status;
}

int sim_dyn_ok(const uint8_t* in, uint64_t n, uint64_t bit) {
    std::vector<uint16_t> u16(INF_VTAB_U16);
    std::vector<uint8_t> u8(INF_VTAB_U8);
    return inf_dyn_ok<1>(in, n, bit, u16.data(), u8.data(), 0) ? 1 : 0;
}

// Every bit offset in [lo, hi) that passes the validator, up to cap of them -> count found
uint64_t sim_find_all(const uint8_t* in, uint64_t n, uint64_t lo, uint64_t hi, uint64_t* out, uint64_t cap) {
    uint16_t u16[INF_VTAB_U16];
    uint8_t u8[INF_VTAB_U8];
    uint64_t m = 0;
    for (uint64_t b = lo; b < hi; b++)
        if (inf_dyn_ok<1>(in, n, b, u16, u8, 0)) {
            if (m < cap) out[m] = b;
            m++;
        }
    return m;
}

void sim_resolve(const uint16_t* sym, uint64_t n, const uint8_t* window, uint8_t* out) {
    for (uint64_t i = 0; i < n; i++) out[i] = inf_resolve(sym[i], window);
}

uint32_t sim_chain(const int* status, const uint32_t* landed, uint32_t n, uint32_t* chain, int* bad) {
    uint32_t bad_chunk = 0;
    return inf_chain(status, landed, n, chain, bad, &bad_chunk);
}

uint32_t sim_crc32(const uint8_t* p, uint64_t n) {
    uint32_t table[256];
    for (uint32_t i = 0; i < 256; i++) table[i] = inf_crc_entry(i);
    return inf_crc32(0, p, n, table);
}

uint32_t sim_crc_combine(uint32_t a, uint32_t b, uint64_t len_b) { return inf_crc_combine(a, b, inf_crc_shift(len_b)); }

}

#ifdef SIM_MAIN
// Sanitizer build: argv[1] a small .gz file; decodes every truncation and every single-byte change of it, in byte
// mode from the member header and in marker mode from the first block, each into heap buffers of exactly the sizes
// passed.  Prints the number of decodes per status; an out-of-bounds access ends the run with a sanitizer report.
#include <stdio.h>
#include <map>

static int run_one(const std::vector<uint8_t>& data, uint64_t cap, std::map<int, long>& seen) {
    uint8_t* in = (uint8_t*)malloc(data.size() ? data.size() : 1);
    for (size_t i = 0; i < data.size(); i++) in[i] = data[i];
    InfBits b;
    b.init(in, data.size(), 0);
    if (data.size() < 10 || inf_gzip_header(b) != 0) { free(in); seen[INF_E_HEADER]++; return 0; }
    const uint64_t start = b.pos();
    uint64_t mp[2], res[6], blocks[4];
    uint32_t mc[2], mi[2];
    const uint64_t cand[2] = {start + 7, start + 800};
    uint8_t* out8 = (uint8_t*)malloc(cap);
    uint16_t* out16 = (uint16_t*)malloc(cap * 2);
    int st = sim_inflate(in, data.size(), start, ~0ull, nullptr, 0, 1, 0, out8, cap, mp, mc, mi, 2, blocks, 4, res);
    seen[st]++;
    st = sim_inflate(in, data.size(), start, start + 4000, cand, 2, 1, 1, out16, cap, mp, mc, mi, 2, blocks, 4, res);
    seen[100 + st]++;
    free(out8); free(out16); free(in);
    return 0;
}

int main(int argc, char** argv) {
    if (argc < 2) return 2;
    FILE* f = fopen(argv[1], "rb");
    if (!f) return 2;
    std::vector<uint8_t> data;
    for (int c; (c = fgetc(f)) != EOF;) data.push_back((uint8_t)c);
    fclose(f);
    const uint64_t cap = argc > 2 ? strtoull(argv[2], nullptr, 10) : 4096;
    std::map<int, long> seen;
    for (size_t len = 0; len < data.size(); len++) run_one(std::vector<uint8_t>(data.begin(), data.begin() + len), cap, seen);
    for (size_t i = 0; i < data.size(); i++)
        for (int x = 1; x < 256; x++) {
            std::vector<uint8_t> d = data;
            d[i] ^= (uint8_t)x;
            run_one(d, cap, seen);
        }
    for (auto& kv : seen) printf("%d %ld\n", kv.first, kv.second);
    return 0;
}
#endif
