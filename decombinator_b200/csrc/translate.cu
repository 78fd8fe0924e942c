// translate.cu -- the translate stage on the GPU (sm_100a): DCR rows -> the lines of the AIRR .tsv.
//
//   dcb_translate_tables_build  the chain's germline tables (import_gene_information, translate.py:123-254) as one
//                               blob: gene records, a 4096-entry codon table over 4-bit IUPAC masks, a string pool.
//   dcb_translate               get_cdr3 (translate.py:257-357) for every row and the DataFrame.to_csv line of each
//                               kept row.  Two passes over the rows -- size each line (and flag rows outside the
//                               envelope), exclusive scan, write each line at its offset -- then one copy of the text
//                               into page-locked host memory.  Every block stages the blob in shared memory first: the
//                               per-row work is lookups into the germline regions and the codon table.
// One thread per row: a row is a few hundred bytes of text built from table lookups, and nothing is shared between
// rows but the tables.
#include "dcb_internal.h"
#include "translate_core.cuh"

#include <cub/device/device_scan.cuh>
#include <cuda_runtime.h>

#include <cstring>
#include <string>
#include <vector>

#define CUDA_TRY(expr)                                                                          \
    do {                                                                                        \
        cudaError_t e__ = (expr);                                                               \
        if (e__ != cudaSuccess) {                                                               \
            dcb_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
            return DCB_ENOGPU;                                                                  \
        }                                                                                       \
    } while (0)

struct dcb_translate_tables {
    std::vector<uint8_t> blob;
};

namespace {

struct DevBuf {
    void* p = nullptr;
    ~DevBuf() { if (p) cudaFree(p); }
    cudaError_t alloc(size_t bytes) { if (p) { cudaFree(p); p = nullptr; } return cudaMalloc(&p, bytes ? bytes : 16); }
    template <class T> T* as() { return static_cast<T*>(p); }
};

struct EventPair {
    cudaEvent_t a = nullptr, b = nullptr;
    ~EventPair() { if (a) cudaEventDestroy(a); if (b) cudaEventDestroy(b); }
};

struct RowArgs {
    const uint8_t* text;
    const uint32_t *v, *j, *vdel, *jdel;
    const uint64_t *id_off, *ins_off;
    const uint32_t *id_len, *ins_len;
    const int64_t *freq, *cluster;
    uint64_t n;
    int npf, nbc;
};

__device__ __forceinline__ const uint8_t* stage_tables(const uint8_t* blob, uint32_t bytes, uint8_t* smem) {
    const uint4* src = (const uint4*)blob;
    uint4* dst = (uint4*)smem;
    for (uint32_t i = threadIdx.x; i < bytes / 16; i += blockDim.x) dst[i] = src[i];
    __syncthreads();
    return smem;
}

__global__ void __launch_bounds__(256)
dcb_translate_size_kernel(const uint8_t* __restrict__ blob, uint32_t blob_bytes, RowArgs A, uint64_t* __restrict__ line_len,
                          uint8_t* __restrict__ productive, uint8_t* __restrict__ row_flags, unsigned int* __restrict__ n_flagged) {
    extern __shared__ __align__(16) uint8_t smem[];
    const TrTables t = tr_tables(stage_tables(blob, blob_bytes, smem));
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= A.n) return;
    TrRow r;
    const uint8_t* ins = A.text + A.ins_off[i];
    tr_row(t, A.v[i], A.j[i], A.vdel[i], A.jdel[i], ins, (int)A.ins_len[i], r);
    if (!tr_plain(A.text + A.id_off[i], (int)A.id_len[i])) r.flags |= TR_F_QUOTE;
    row_flags[i] = (uint8_t)r.flags;
    productive[i] = r.productive;
    if (r.flags) {
        atomicAdd(n_flagged, 1u);
        line_len[i] = 0;
        return;
    }
    TrLine L;
    L.seq_id = (int64_t)i + 1; L.freq = A.freq[i]; L.cluster = A.cluster[i]; L.nbc = A.nbc != 0;
    L.id = A.text + A.id_off[i]; L.id_len = (int)A.id_len[i];
    line_len[i] = (A.npf && !r.productive) ? 0 : tr_line_len(t, r, L, A.v[i], A.j[i]);
}

__global__ void __launch_bounds__(256)
dcb_translate_write_kernel(const uint8_t* __restrict__ blob, uint32_t blob_bytes, RowArgs A, const uint64_t* __restrict__ line_off,
                           const uint64_t* __restrict__ line_len, char* __restrict__ out) {
    extern __shared__ __align__(16) uint8_t smem[];
    const TrTables t = tr_tables(stage_tables(blob, blob_bytes, smem));
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= A.n || line_len[i] == 0) return;
    TrRow r;
    tr_row(t, A.v[i], A.j[i], A.vdel[i], A.jdel[i], A.text + A.ins_off[i], (int)A.ins_len[i], r);
    TrLine L;
    L.seq_id = (int64_t)i + 1; L.freq = A.freq[i]; L.cluster = A.cluster[i]; L.nbc = A.nbc != 0;
    L.id = A.text + A.id_off[i]; L.id_len = (int)A.id_len[i];
    tr_write(t, r, L, A.v[i], A.j[i], out + line_off[i]);
}

// Bio.Seq's standard table over IUPAC codes (translate.py: _ambiguous_codon)
void build_codon_table(uint8_t* out) {
    static const char* bases = "TCAG";
    static const char* amino = "FFLLSSSSYY**CC*WLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG";
    auto base_bit = [](char b) { return b == 'A' ? 1 : b == 'C' ? 2 : b == 'G' ? 4 : 8; };
    for (int m = 0; m < 4096; m++) {
        const int m1 = m >> 8, m2 = (m >> 4) & 15, m3 = m & 15;
        out[m] = 0;
        if (!m1 || !m2 || !m3) continue;
        std::string aas;
        for (int a = 0; a < 4; a++)
            for (int b = 0; b < 4; b++)
                for (int c = 0; c < 4; c++) {
                    if (!(m1 & base_bit(bases[a])) || !(m2 & base_bit(bases[b])) || !(m3 & base_bit(bases[c]))) continue;
                    const char x = amino[16 * a + 4 * b + c];
                    if (aas.find(x) == std::string::npos) aas += x;
                }
        auto within = [&](const char* set) { for (char x : aas) if (!std::strchr(set, x)) return false; return true; };
        char aa;
        if (aas.size() == 1) aa = aas[0];
        else if (aas.find('*') != std::string::npos) aa = 'X';
        else if (within("DN")) aa = 'B';
        else if (within("EQ")) aa = 'Z';
        else if (within("IL")) aa = 'J';
        else aa = 'X';
        out[m] = (uint8_t)aa;
    }
}

bool plain_text(const char* s) {
    for (; *s; s++)
        if ((unsigned char)*s < 0x20 || (unsigned char)*s >= 0x7F || *s == '"') return false;
    return true;
}

}  // namespace

extern "C" {

int dcb_translate_tables_build(int n_v, const char* const* v_regions, const char* const* v_calls, const int32_t* v_pos,
                               const char* const* v_residue, const char* const* v_cdr1, const char* const* v_cdr2, int n_j,
                               const char* const* j_regions, const char* const* j_calls, const int32_t* j_pos,
                               const char* const* j_motif, dcb_translate_tables** out) {
    if (!out || n_v < 0 || n_j < 0 || (n_v && (!v_regions || !v_calls || !v_pos || !v_residue || !v_cdr1 || !v_cdr2)) ||
        (n_j && (!j_regions || !j_calls || !j_pos || !j_motif))) {
        dcb_set_error("dcb_translate_tables_build: null argument");
        return DCB_EINVAL;
    }
    *out = nullptr;
    std::vector<TrGene> genes((size_t)n_v + n_j);
    std::string pool;
    auto add = [&](const char* s, uint32_t& off, uint16_t& len) -> bool {
        const size_t n = std::strlen(s);
        if (n > 0xFFFF) return false;
        off = (uint32_t)pool.size(); len = (uint16_t)n;
        pool += s;
        return true;
    };
    for (int g = 0; g < n_v + n_j; g++) {
        const bool is_v = g < n_v;
        const int k = is_v ? g : g - n_v;
        TrGene& G = genes[g];
        std::memset(&G, 0, sizeof(G));
        const char* region = is_v ? v_regions[k] : j_regions[k];
        const char* call = is_v ? v_calls[k] : j_calls[k];
        for (const char* p = region; *p; p++)
            if (*p < 'A' || *p > 'Z' || tr_mask((uint8_t)*p) == 0) {
                dcb_set_error("dcb_translate_tables_build: %s gene %d: region symbol '%c' outside upper-case IUPAC", is_v ? "V" : "J", k, *p);
                return DCB_EUNSUPPORTED;
            }
        if (std::strlen(region) > DCB_TR_MAX_SEQ) {
            dcb_set_error("dcb_translate_tables_build: %s gene %d: region longer than %d", is_v ? "V" : "J", k, DCB_TR_MAX_SEQ);
            return DCB_EUNSUPPORTED;
        }
        if (!plain_text(call) || (is_v && (!plain_text(v_cdr1[k]) || !plain_text(v_cdr2[k])))) {
            dcb_set_error("dcb_translate_tables_build: %s gene %d: a name or CDR the .tsv would quote", is_v ? "V" : "J", k);
            return DCB_EUNSUPPORTED;
        }
        if (!add(region, G.region_off, G.region_len) || !add(call, G.call_off, G.call_len)) {
            dcb_set_error("dcb_translate_tables_build: string too long");
            return DCB_EUNSUPPORTED;
        }
        if (is_v) {
            if (!add(v_cdr1[k], G.cdr1_off, G.cdr1_len) || !add(v_cdr2[k], G.cdr2_off, G.cdr2_len)) {
                dcb_set_error("dcb_translate_tables_build: string too long");
                return DCB_EUNSUPPORTED;
            }
            G.pos = v_pos[k];
            const char* r = v_residue[k];
            G.res[0] = std::strlen(r) == 1 ? (uint8_t)r[0] : 0;       // a longer (or empty) residue never matches
        } else {
            G.pos = j_pos[k];
            const char* m = j_motif[k];
            bool ok = std::strlen(m) == 4;
            for (int q = 0; ok && q < 4; q++) ok = (m[q] >= 'A' && m[q] <= 'Z') || m[q] == '.';
            if (!ok) {
                dcb_set_error("dcb_translate_tables_build: J gene %d: motif '%s' is not four capital letters or '.'", k, m);
                return DCB_EUNSUPPORTED;
            }
            std::memcpy(G.res, m, 4);
        }
    }
    auto up16 = [](size_t x) { return (x + 15) & ~(size_t)15; };
    TrHeader h;
    std::memset(&h, 0, sizeof(h));
    h.magic = DCB_TR_MAGIC; h.n_v = (uint32_t)n_v; h.n_j = (uint32_t)n_j;
    h.genes_off = (uint32_t)up16(sizeof(TrHeader));
    h.codon_off = (uint32_t)up16(h.genes_off + genes.size() * sizeof(TrGene));
    h.pool_off = h.codon_off + 4096;
    const size_t total = up16(h.pool_off + pool.size());
    if (total > 160 * 1024) {
        dcb_set_error("dcb_translate_tables_build: tables of %zu bytes exceed the 160 KiB staged in shared memory", total);
        return DCB_EUNSUPPORTED;
    }
    h.bytes = (uint32_t)total;
    auto* t = new dcb_translate_tables();
    t->blob.assign(total, 0);
    std::memcpy(t->blob.data(), &h, sizeof(h));
    if (!genes.empty()) std::memcpy(t->blob.data() + h.genes_off, genes.data(), genes.size() * sizeof(TrGene));
    build_codon_table(t->blob.data() + h.codon_off);
    std::memcpy(t->blob.data() + h.pool_off, pool.data(), pool.size());
    *out = t;
    return DCB_OK;
}

void dcb_translate_tables_free(dcb_translate_tables* t) { delete t; }

int dcb_translate_tables_blob(const dcb_translate_tables* t, const uint8_t** bytes, size_t* n_bytes) {
    if (!t || !bytes || !n_bytes) { dcb_set_error("dcb_translate_tables_blob: null argument"); return DCB_EINVAL; }
    *bytes = t->blob.data();
    *n_bytes = t->blob.size();
    return DCB_OK;
}

int dcb_translate(dcb_dist* d, const dcb_translate_tables* t, const char* text, uint64_t text_bytes, const uint32_t* v, const uint32_t* j,
                  const uint32_t* vdel, const uint32_t* jdel, const uint64_t* id_off, const uint32_t* id_len, const uint64_t* ins_off,
                  const uint32_t* ins_len, const int64_t* freq, const int64_t* cluster, uint64_t n, int nonproductive_filter,
                  int nobarcoding, uint8_t* productive, uint8_t* row_flags, uint64_t* n_flagged, char** out, uint64_t* out_bytes) {
    if (!d) {
        int n_dev = 0;
        if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0) {
            (void)cudaGetLastError();
            dcb_set_error("dcb_translate: no CUDA device available (there is no CPU fallback)");
            return DCB_ENOGPU;
        }
    }
    if (!d || !t || !n_flagged || !out || !out_bytes ||
        (n && (!text || !v || !j || !vdel || !jdel || !id_off || !id_len || !ins_off || !ins_len || !freq || !cluster || !productive || !row_flags))) {
        dcb_set_error("dcb_translate: null argument");
        return DCB_EINVAL;
    }
    *out = nullptr; *out_bytes = 0; *n_flagged = 0;
    if (n == 0) return DCB_OK;
    for (uint64_t i = 0; i < n; i++)
        if (id_off[i] + id_len[i] > text_bytes || ins_off[i] + ins_len[i] > text_bytes) {
            dcb_set_error("dcb_translate: row %llu reaches beyond the text", (unsigned long long)i);
            return DCB_EINVAL;
        }
    CUDA_TRY(cudaSetDevice(dcb_dist_device(d)));
    cudaStream_t s = (cudaStream_t)dcb_dist_stream(d);
    const uint32_t blob_bytes = (uint32_t)t->blob.size();
    CUDA_TRY(cudaFuncSetAttribute(dcb_translate_size_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)blob_bytes));
    CUDA_TRY(cudaFuncSetAttribute(dcb_translate_write_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)blob_bytes));
    DevBuf d_blob, d_text, d_cols, d_off, d_len, d_scan, d_tmp, d_prod, d_flags, d_cnt, d_out;
    CUDA_TRY(d_blob.alloc(blob_bytes));
    CUDA_TRY(d_text.alloc(text_bytes + 16));
    // v, j, vdel, jdel, id_len, ins_len (u32); id_off, ins_off, freq, cluster (8 bytes)
    const size_t c4 = n * 4, c8 = n * 8;
    CUDA_TRY(d_cols.alloc(6 * c4 + 4 * c8 + 64));
    uint8_t* cols = d_cols.as<uint8_t>();
    uint8_t* c8base = cols + ((6 * c4 + 15) & ~(size_t)15);
    CUDA_TRY(d_len.alloc(c8 + 8));
    CUDA_TRY(d_off.alloc(c8 + 8));
    CUDA_TRY(d_prod.alloc(n));
    CUDA_TRY(d_flags.alloc(n));
    CUDA_TRY(d_cnt.alloc(16));
    CUDA_TRY(cudaMemcpyAsync(d_blob.p, t->blob.data(), blob_bytes, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(d_text.p, text, text_bytes, cudaMemcpyHostToDevice, s));
    const void* src4[6] = {v, j, vdel, jdel, id_len, ins_len};
    for (int k = 0; k < 6; k++) CUDA_TRY(cudaMemcpyAsync(cols + k * c4, src4[k], c4, cudaMemcpyHostToDevice, s));
    const void* src8[4] = {id_off, ins_off, freq, cluster};
    for (int k = 0; k < 4; k++) CUDA_TRY(cudaMemcpyAsync(c8base + k * c8, src8[k], c8, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemsetAsync(d_cnt.p, 0, 16, s));
    RowArgs A;
    A.text = d_text.as<uint8_t>();
    A.v = (const uint32_t*)(cols); A.j = (const uint32_t*)(cols + c4); A.vdel = (const uint32_t*)(cols + 2 * c4);
    A.jdel = (const uint32_t*)(cols + 3 * c4); A.id_len = (const uint32_t*)(cols + 4 * c4); A.ins_len = (const uint32_t*)(cols + 5 * c4);
    A.id_off = (const uint64_t*)(c8base); A.ins_off = (const uint64_t*)(c8base + c8);
    A.freq = (const int64_t*)(c8base + 2 * c8); A.cluster = (const int64_t*)(c8base + 3 * c8);
    A.n = n; A.npf = nonproductive_filter != 0; A.nbc = nobarcoding != 0;
    const unsigned blocks = (unsigned)((n + 255) / 256);
    EventPair ev;
    CUDA_TRY(cudaEventCreate(&ev.a)); CUDA_TRY(cudaEventCreate(&ev.b));
    CUDA_TRY(cudaEventRecord(ev.a, s));
    dcb_translate_size_kernel<<<blocks, 256, blob_bytes, s>>>(d_blob.as<uint8_t>(), blob_bytes, A, d_len.as<uint64_t>(), d_prod.as<uint8_t>(),
                                                              d_flags.as<uint8_t>(), d_cnt.as<unsigned int>());
    CUDA_TRY(cudaGetLastError());
    // exclusive scan over n + 1 entries: the last offset is the text's size
    CUDA_TRY(cudaMemsetAsync(d_len.as<uint64_t>() + n, 0, 8, s));
    size_t tmp_bytes = 0;
    CUDA_TRY(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, d_len.as<uint64_t>(), d_off.as<uint64_t>(), (int64_t)(n + 1), s));
    CUDA_TRY(d_tmp.alloc(tmp_bytes));
    CUDA_TRY(cub::DeviceScan::ExclusiveSum(d_tmp.p, tmp_bytes, d_len.as<uint64_t>(), d_off.as<uint64_t>(), (int64_t)(n + 1), s));
    unsigned int flagged = 0;
    uint64_t total = 0;
    CUDA_TRY(cudaMemcpyAsync(&flagged, d_cnt.p, 4, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(&total, d_off.as<uint64_t>() + n, 8, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(productive, d_prod.p, n, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(row_flags, d_flags.p, n, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    *n_flagged = flagged;
    if (flagged) return DCB_OK;          // the caller takes the host path for the whole call: no text
    CUDA_TRY(d_out.alloc(total + 16));
    dcb_translate_write_kernel<<<blocks, 256, blob_bytes, s>>>(d_blob.as<uint8_t>(), blob_bytes, A, d_off.as<uint64_t>(), d_len.as<uint64_t>(),
                                                               d_out.as<char>());
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaEventRecord(ev.b, s));
    char* host = nullptr;
    CUDA_TRY(cudaMallocHost((void**)&host, total + 1));
    cudaError_t e = cudaMemcpyAsync(host, d_out.p, total, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) {
        cudaFreeHost(host);
        dcb_set_error("dcb_translate: copy of the text failed: %s", cudaGetErrorString(e));
        return DCB_ENOGPU;
    }
    host[total] = 0;
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ev.a, ev.b) == cudaSuccess) dcb_dist_set_last_ms(d, ms);   // both kernels and the scan
    *out = host;
    *out_bytes = total;
    return DCB_OK;
}

}  // extern "C"
