// dcb_internal.h -- definitions shared by the translation units of libdcb.so (not installed).
#ifndef DCB_INTERNAL_H
#define DCB_INTERNAL_H

#include "../../include/dcb.h"
#include "dcb_tables.h"

#include <map>
#include <string>
#include <vector>

struct dcb_tagset {
    int n_tags = 0, split = 0, is_v = 0, lmin = 0;
    std::vector<std::string> tags;
    std::vector<uint32_t> general;  // DcbGene + tags + keyword sets + germline regions (general kernel)
    std::vector<uint32_t> core;     // DcbGene + tags only (exact-tag kernels)
    std::vector<uint32_t> index;    // DcbSeedIndex of this gene alone
};

// Seed index over one gene (other pointer null) or over both genes of a chain (equal lmin).
bool dcb_build_seed_index(const std::vector<std::string>* gene_v, const std::vector<std::string>* gene_j, int lmin,
                          int wbits, std::vector<uint32_t>& out);

// Sampled half-tag index over both genes of a chain (DcbHalfIndex); false when a half keyword is too short for it.
bool dcb_build_half_index(const dcb_tagset* v, const dcb_tagset* j, std::vector<uint32_t>& out);

extern "C" int dcb_packed_alloc(uint64_t n, uint32_t slot_words, uint32_t n_exc, dcb_packed** out);
extern "C" int dcb_pack_words(const char* ascii, const uint64_t* off, const uint32_t* len, uint64_t first, uint64_t count, uint32_t uniform_len,
                              int revcomp, uint32_t slot_words, uint32_t* words, int n_threads, int* clean);

// The light context of collapse.cu, for the other entry points that hang off it (translate.cu).
int dcb_dist_device(const dcb_dist* d);
void* dcb_dist_stream(const dcb_dist* d);
void dcb_dist_set_last_ms(dcb_dist* d, double ms);

#if defined(__GNUC__)
__attribute__((format(printf, 1, 2)))
#endif
void dcb_set_error(const char* fmt, ...);

#endif
