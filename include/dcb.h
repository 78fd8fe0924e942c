/*
 * dcb.h -- C ABI of libdcb.so, the B200-native `decombine` hot path.
 *
 * The reference (innate2adaptive/decombinator, /root/reference) is pure Python and has no FFI
 * of its own; the drop-in boundary is the stage function decombinator(inputargs)
 * (src/decombinator/decombine.py:881) and, inside it, the per-read contract dcr(read, inputargs)
 * (decombine.py:534).  Each entry point below names the reference interface it replaces, as
 * file:line under /root/reference/src/decombinator/.  INTEGRATION.md shows the ctypes binding a
 * maintainer would add to the reference to call them.
 *
 * Conventions: plain pointers and sizes only; every function returning int returns 0 on success
 * and a negative DCB_E* code on failure, with text from dcb_last_error(); no exceptions cross the
 * boundary; a context is used by one host thread at a time and launches on its own stream
 * (or the one given with dcb_ctx_set_stream).  There is NO CPU fallback: compute entry points
 * fail with DCB_ENOGPU when no CUDA device is usable.
 */
#ifndef DCB_H
#define DCB_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DCB_ABI_VERSION 1

enum {
    DCB_OK = 0,
    DCB_EINVAL = -1,   /* bad argument */
    DCB_ENOGPU = -2,   /* no usable CUDA device / CUDA error */
    DCB_ENOMEM = -3,
    DCB_EUNSUPPORTED = -4, /* input outside what the tables support (e.g. tag longer than 32 nt) */
    DCB_EIO = -5
};

const char* dcb_last_error(void);
int dcb_abi_version(void);

/* ---------------------------------------------------------------------------------------------
 * Counters: the keys of the reference's `counts` Counter that dcr() and its callees bump
 * (decombine.py:279-584; written to the summary at decombine.py:1131-1195).
 * ------------------------------------------------------------------------------------------- */
enum dcb_counter {
    DCB_C_verr1 = 0,
    DCB_C_verr2,
    DCB_C_jerr1,
    DCB_C_jerr2,
    DCB_C_dcrfilter_intertagN,
    DCB_C_dcrfilter_toolong_intertag,
    DCB_C_dcrfilter_imposs_deletion,
    DCB_C_dcrfilter_tag_overlap,
    DCB_C_multiple_v_matches,
    DCB_C_v_del_failed_tag_at_end,
    DCB_C_v_del_failed,
    DCB_C_foundv1notv2,
    DCB_C_foundv2notv1,
    DCB_C_no_vtags_found,
    DCB_C_multiple_j_matches,
    DCB_C_j_del_failed,
    DCB_C_foundj1notj2,
    DCB_C_foundj2notj1,
    DCB_C_no_j_assigned,
    DCB_C_VJ_assignment_failed,
    DCB_NCOUNTERS
};
/* Name of counter i as spelled in the reference ("verr1", ...), or NULL. */
const char* dcb_counter_name(int i);

/* ---------------------------------------------------------------------------------------------
 * Tag tables.  Replaces get_v_tags/get_j_tags + the six AcoraBuilder automata of
 * import_tcr_info (decombine.py:681-746, 820-866): one call per gene.
 *   tags[i], jumps[i] : columns 0 and 1 of the .tags file       (decombine.py:826-835)
 *   regions[i]        : upper-cased FASTA record i               (decombine.py:690-696)
 *   half_split        : v_half_split / j_half_split              (decombine.py:657-661)
 * Tags and regions must be pure ACGT, 4 <= len(tag) <= 32, n <= 255 (DCB_EUNSUPPORTED otherwise).
 * Host only; no GPU needed.
 * ------------------------------------------------------------------------------------------- */
typedef struct dcb_tagset dcb_tagset;
dcb_tagset* dcb_tagset_build(const char* const* tags, const int32_t* jumps, const char* const* regions,
                             int n, int half_split, int is_v);
void dcb_tagset_free(dcb_tagset*);
/* Total bytes of the flattened table blobs (what thread blocks stage in shared memory). */
size_t dcb_tagset_table_bytes(const dcb_tagset*);
/* Introspection (tests): which = 0 the general-kernel blob, 1 the tag records of the exact-tag kernels,
 * 2 this gene's seed index. */
int dcb_tagset_blob(const dcb_tagset*, int which, const uint32_t** words, size_t* n_words);
/* Seed index over BOTH genes of a chain (built by dcb_ctx_create when V and J share the seed geometry).
 * Writes up to cap words; *n_words is the size needed; returns DCB_EUNSUPPORTED when the geometries differ. */
int dcb_tagset_union_index(const dcb_tagset* v, const dcb_tagset* j, uint32_t* out, size_t cap, size_t* n_words);
/* Sampled half-tag index of a chain (csrc/dcb_tables.h, DcbHalfIndex): what the half-tag kernel finds the occurrences of
   the acora half-tag automata with (decombine.py:730-746 build them; findall at :294, :339, :422, :473).  Same calling
   convention; DCB_EUNSUPPORTED when a half tag of the chain is shorter than 10 bases (the kernel then does not run). */
int dcb_tagset_half_index(const dcb_tagset* v, const dcb_tagset* j, uint32_t* out, size_t cap, size_t* n_words);
/* Union suffix filter of the six keyword sets of a chain (csrc/dcb_tables.h, DcbSuffixFilter): what the general kernel
   marks candidate keyword positions with.  Same calling convention as dcb_tagset_union_index. */
int dcb_tagset_suffix_filter(const dcb_tagset* v, const dcb_tagset* j, uint32_t* out, size_t cap, size_t* n_words);

/* ---------------------------------------------------------------------------------------------
 * Packed reads: 2 bits per base (A=0 C=1 G=2 T=3, base i of a read in bits [2*(i%16), +2) of
 * word i/16), one fixed-size slot of `slot_words` 32-bit words per read (a multiple of 4, so a
 * slot is read with 128-bit loads).  Any other symbol is packed as 0 and listed in the sparse
 * exception arrays (sorted by read): kind 1 = 'N', kind 2 = anything else.  `flags` has one bit
 * per read that is set when the read has exceptions.  Buffers are page-locked when a GPU is
 * present so they can be streamed to HBM with cudaMemcpyAsync.
 * ------------------------------------------------------------------------------------------- */
typedef struct dcb_packed {
    uint64_t n_reads;
    uint32_t slot_words;   /* 32-bit words per read slot */
    uint32_t uniform_len;  /* != 0: every read has this length and `lens` may be ignored */
    uint32_t max_len;
    uint32_t n_exc;
    uint32_t* words;       /* n_reads * slot_words */
    uint16_t* lens;        /* n_reads */
    uint32_t* flags;       /* ceil(n_reads/32) */
    uint32_t* exc_read;    /* n_exc : read index */
    uint16_t* exc_pos;     /* n_exc : base position in the ORIENTED read */
    uint8_t*  exc_kind;    /* n_exc : 1 = 'N', 2 = other */
    void* owner;           /* internal */
} dcb_packed;

/* Replaces the string handling of the main loop for the V(D)J read: `vdj = record1[1]`
 * (decombine.py:965-977) and, when revcomp != 0, revcomp(vdj) (decombine.py:182-184, 1000)
 * with Bio.Seq's complement table.  ascii/off/len describe n reads inside one byte buffer.
 * Allocates *out (free with dcb_packed_free).  Host only; multi-threaded. */
int dcb_pack_reads(const char* ascii, const uint64_t* off, const uint32_t* len, uint64_t n, int revcomp,
                   int n_threads, dcb_packed** out);
void dcb_packed_free(dcb_packed*);
/* The host's share of dcb_decombine_ascii: reads [first, first + count) of nothing but A / C / G / T packed (AVX2, n_threads
 * host threads) into the caller's buffer of count * slot_words words, in the layout of dcb_packed.words.  *clean = 0 when
 * another symbol turned up (or the CPU has no AVX2): the buffer is then void.  off == NULL: contiguous reads of uniform_len. */
int dcb_pack_words(const char* ascii, const uint64_t* off, const uint32_t* len, uint64_t first, uint64_t count, uint32_t uniform_len,
                   int revcomp, uint32_t slot_words, uint32_t* words, int n_threads, int* clean);
/* ---------------------------------------------------------------------------------------------
 * FASTQ ingest (host): the record index of a FASTQ text held in memory.  Replaces the reference's
 * parser readfq (decombine.py:228-265) for files in the strict layout (four lines per record, '\n'
 * line ends, ASCII, quality at least as long as its sequence): name = header after '@' up to the
 * first space, sequence / quality = the second / fourth line, all as (offset, length) into `text`,
 * so sequences go to dcb_pack_reads without a copy.  strict == 0 (and n_records == 0): the text is
 * not in that layout and the caller must use the general parser.
 * ------------------------------------------------------------------------------------------- */
typedef struct dcb_fastq_index {
    uint64_t n_records;
    uint64_t* name_off; uint32_t* name_len;
    uint64_t* seq_off;  uint32_t* seq_len;
    uint64_t* qual_off; uint32_t* qual_len;
    int32_t strict;
} dcb_fastq_index;
int dcb_fastq_index_build(const char* text, uint64_t n_bytes, int n_threads, dcb_fastq_index** out);
void dcb_fastq_index_free(dcb_fastq_index*);
/* Number of the n byte ranges (off[i], len[i]) of text that contain `symbol` (the barcode "N" count,
   decombine.py:985-989). */
uint64_t dcb_count_ranges_with(const char* text, const uint64_t* off, const uint32_t* len, uint64_t n, int symbol,
                               int n_threads);

/* Inverse of the packer for one read (tests): writes len chars, exceptions as 'N' / '?'. */
int dcb_unpack_read(const dcb_packed*, uint64_t i, char* dst, uint32_t cap);

/* ---------------------------------------------------------------------------------------------
 * Per-read result: what dcr() returns (decombine.py:572-581) as a 16-byte record.  The insert
 * string is oriented_read[ins_start:ins_end]; tcrseq / tcrQ are sliced with
 * [v_seq_start:j_seq_end] on the host (decombine.py:1015-1020).
 * ------------------------------------------------------------------------------------------- */
typedef struct dcb_result {
    uint8_t status;        /* 0: dcr() returned None; 1: rearrangement found */
    uint8_t frame;         /* 0: the packed orientation; 1: its reverse complement (-or both, 2nd try) */
    uint8_t v, j;          /* recom[0], recom[1] */
    uint16_t vdel, jdel;   /* recom[2], recom[3] */
    uint16_t ins_start;    /* end_v + 1 */
    uint16_t ins_end;      /* start_j */
    uint16_t v_seq_start;  /* recom[5] */
    uint16_t j_seq_end;    /* recom[6] */
} dcb_result;

/* One string per read as (offset, length) into a text buffer (a column of the FASTQ index above). */
typedef struct dcb_column { const char* text; const uint64_t* off; const uint32_t* len; } dcb_column;

/* Row assembly of the reference's main loop (decombine.py:1015-1039) for every read with status 1, in read
 * order: v, j, vdel, jdel, insert, read id, tcrseq, tcrQ, barcode, barcode quality (+ v_tail when given), fields
 * joined by `sep`, one row per line, into ONE malloc'ed buffer (free with dcb_buffer_free).  packed_revcomp:
 * the batch was packed as the reverse complement (-or reverse / both); a result of frame 1 is the other strand.
 * With sep = ", " the buffer is the .n12 text of write_out_intermediate (io.py:480-513). */
int dcb_format_rows(const dcb_result* res, uint64_t n, int packed_revcomp, const dcb_column* ids, const dcb_column* vdj,
                    const dcb_column* vdjqual, const dcb_column* bc, const dcb_column* bcq, const dcb_column* v_tail,
                    const char* sep, int n_threads, char** out, uint64_t* out_bytes, uint64_t* n_rows);
/* What collapse builds per decombined row before it groups them (collapse.py:560-590), for all rows at once: three lines
 * per row -- tcrseq; str(row[:5]), i.e. "['v', 'j', 'vdel', 'jdel', 'insert']"; and "|".join((that, tcrseq, tcrQ, read id)). */
int dcb_format_collapse_rows(const dcb_result* res, uint64_t n, int packed_revcomp, const dcb_column* ids, const dcb_column* vdj,
                             const dcb_column* vdjqual, int n_threads, char** out, uint64_t* out_bytes, uint64_t* n_rows);
/* The `collapse` command's input: index of an .n12 text (ten fields per row joined by ", ", as write_out_intermediate
 * writes them, io.py:480-513) -- off / len are n_rows x 10, row-major, malloc'ed (dcb_buffer_free); *n_rows = 0 when the
 * text is not of that shape (the caller then splits the lines as the reference does, collapse.py:523-530) -- and the
 * three lines of dcb_format_collapse_rows built from the fields of the rows with keep[i] != 0 (*n_rows = UINT64_MAX:
 * a field holds a quote or a backslash, str() would write it differently; the caller builds the strings itself). */
int dcb_n12_index(const char* text, uint64_t n_bytes, int n_threads, uint64_t** off, uint32_t** len, uint64_t* n_rows);
int dcb_n12_collapse_rows(const char* text, const uint64_t* off, const uint32_t* len, uint64_t n, const uint8_t* keep, int n_threads,
                          char** out, uint64_t* out_bytes, uint64_t* n_rows);
void dcb_buffer_free(char*);
/* Compressed FASTQ (the reference reads it through gzip.open, decombine.py:118-123): the blocks of a BGZF file -- raw deflate
 * data raw[start[k], end[k]) of isize[k] bytes each, its CRC-32 behind it -- inflated side by side into out + out_off[k]. */
int dcb_bgzf_inflate(const unsigned char* raw, const uint64_t* start, const uint64_t* end, const uint32_t* isize, const uint64_t* out_off,
                     uint64_t n_blocks, unsigned char* out, int n_threads);

/* The order-dependent grouping of collapse's read_in_data (collapse.py:595-682) over columns instead of a Python loop over
 * rows: per barcode, rows in input order found / join / kill the barcode's group (rules: csrc/group.cpp).  Host logic; the
 * sequence comparisons it needs (are_seqs_equivalent, collapse.py:355-360) are the caller's to fetch from the GPU:
 *   dcb_group_create(seqs joined by '\n', barcode code and global row index per row)
 *   loop: dcb_group_step -> n_pairs; 0: done.  dcb_group_pairs (sizes with symbols == NULL, then the arrays) is a batch
 *         for dcb_lev_leq (coded = 1) / dcb_lev_leq_bytes (coded = 0); dcb_group_verdicts feeds the answers back
 *   dcb_group_result (sizes with rows == NULL, then the arrays): surviving groups in the reference's dict order with
 *         their barcode code, tick (the row index at which the group took its place), a row holding the proto-sequence, and their member rows (first[g] .. first[g + 1]). */
typedef struct dcb_group dcb_group;
int dcb_group_create(const char* seqs, uint64_t seqs_bytes, uint64_t n, const uint64_t* code, const uint64_t* idx, dcb_group** out);
int dcb_group_step(dcb_group*, uint64_t* n_pairs);
int dcb_group_pairs(dcb_group*, uint64_t* n_seqs, uint64_t* n_symbols, uint8_t* symbols, uint64_t* off, uint32_t* len, uint32_t* a, uint32_t* b,
                    int* coded);
int dcb_group_verdicts(dcb_group*, const uint8_t* same, uint64_t n_pairs);
int dcb_group_result(dcb_group*, uint64_t* n_groups, uint64_t* n_members, uint64_t* dropped, uint64_t* dead, uint64_t* code, uint64_t* tick,
                     uint32_t* proto_row, uint64_t* first, uint32_t* rows);
void dcb_group_free(dcb_group*);


typedef struct dcb_params {
    int32_t both_frames;   /* -or both: retry the reverse complement of the packed read when the first try fails
                              (decombine.py:1005-1010); reads are then packed in the FIRST orientation tried */
    int32_t allow_ns;      /* inputargs["allowNs"]      (decombine.py:553-556) */
    int32_t lenthreshold;  /* inputargs["lenthreshold"] (decombine.py:557-560) */
    int32_t force_general; /* testing: 1 = send every read through the general (fallback) kernel;
                              2 = exact-tag search without the flat kernel (the bit-filter kernels only);
                              3 = no half-tag kernel (the flat kernel's queue goes straight to the general kernel) */
} dcb_params;

/* ---------------------------------------------------------------------------------------------
 * Context: one per GPU.  Owns the device copies of the tag tables, the device batch buffers and
 * a stream.  Replaces the module globals import_tcr_info() sets up (decombine.py:593-746).
 * ------------------------------------------------------------------------------------------- */
typedef struct dcb_ctx dcb_ctx;
dcb_ctx* dcb_ctx_create(int device, const dcb_tagset* v, const dcb_tagset* j, const dcb_params* p);
void dcb_ctx_destroy(dcb_ctx*);
/* Launch on an externally owned cudaStream_t (e.g. torch's current stream) instead of the ctx's own. */
int dcb_ctx_set_stream(dcb_ctx*, void* cuda_stream);

/* The batched dcr(): replaces the body of the hot loop `for records in zipfqs: ... dcr(...)`
 * (decombine.py:963-1010) for n reads.  HOST buffers in, HOST buffers out: streams the packed
 * batch to HBM in chunks on two streams (upload, kernels and download of different chunks
 * overlap), copies the n result records back and ADDS this batch's counter deltas to
 * counters[DCB_NCOUNTERS].  Synchronous on return. */
int dcb_decombine_batch(dcb_ctx*, const dcb_packed* reads, dcb_result* out, uint64_t* counters);

/* The same from ASCII: replaces the string handling in front of dcr() -- `vdj = record1[1]` (decombine.py:965-977) and,
 * when revcomp != 0, revcomp(vdj) (decombine.py:182-184, 1000) -- AND the hot loop, in one call.  The text is streamed
 * to HBM in chunks and packed there (csrc/pack_device.cuh: bit-identical to dcb_pack_reads); no packed copy is made on
 * the host.  Read i is ascii[off[i] .. off[i] + len[i]); offsets must not decrease inside the batch (FASTQ order).
 * off == NULL: the reads are contiguous, read i at i * uniform_len.  uniform_len != 0: every read has that length and
 * len is ignored.  Chunks of nothing but A / C / G / T are shared between the device packer and the host threads
 * (dcb_pack_words): page-locked text from both ends, the device taking chunks from the front and the host threads from
 * the back; pageable text by the host threads until the first chunk with another symbol.  Chunks with other symbols are
 * packed by the device.  The environment variable DCB_HOST_SHARE = 0 makes the device pack every chunk; a value other
 * than 0 or 1 fails the call with DCB_EINVAL. */
int dcb_decombine_ascii(dcb_ctx*, const char* ascii, const uint64_t* off, const uint32_t* len, uint64_t n, uint32_t uniform_len,
                        int revcomp, dcb_result* out, uint64_t* counters);
/* The device packer alone: its output copied back into a host dcb_packed (free with dcb_packed_free); tests compare it
 * with dcb_pack_reads.  dcb_pack_device_ms: device time (CUDA events) of the last call, copies of the text included. */
int dcb_pack_device(dcb_ctx*, const char* ascii, const uint64_t* off, const uint32_t* len, uint64_t n, uint32_t uniform_len,
                    int revcomp, dcb_packed** out);
int dcb_pack_device_ms(dcb_ctx*, double* ms);
/* How the chunks of the last dcb_decombine_ascii call were packed: by the host threads (clean reads, dcb_pack_words: a
 * quarter of the text's bytes cross the link) or by the device (the text itself crosses the link).  With
 * DCB_HOST_SHARE = 0 the host packs none. */
int dcb_last_pack_shares(dcb_ctx*, uint32_t* host_chunks, uint32_t* device_chunks);

/* Page-locked host memory for result records (so that the device->host copies of dcb_decombine_batch run
 * asynchronously, overlapped with the uploads); NULL when no GPU is usable. */
void* dcb_pinned_alloc(size_t bytes);
void dcb_pinned_free(void*);

/* Same work with the batch resident in HBM (bench `value`, multi-step pipelines):
 *   dcb_upload          : host packed batch -> ctx-owned device buffers (synchronous)
 *   dcb_run_resident    : launch the kernels on the resident batch; asynchronous on the ctx stream.  The kernels of
 *                         consecutive steps are chained by programmatic dependent launch; the environment variable
 *                         DCB_PDL = 0 launches them plainly behind a memset of the counters, a value other than 0 or 1
 *                         fails the call with DCB_EINVAL
 *   dcb_download        : wait, copy results + ADD counter deltas of the last run
 */
int dcb_upload(dcb_ctx*, const dcb_packed* reads);
int dcb_run_resident(dcb_ctx*);
int dcb_download(dcb_ctx*, dcb_result* out, uint64_t* counters);

/* Per-kernel device time of the resident steps, accumulated since the last reset, and the number of launches timed.
 * A launch's time runs from the start of its first block to the end of its last block (%globaltimer, stamped by the
 * kernels themselves: no host event sits between the launches of a step).
 * slot 0: exact-tag matching kernel, slot 1: general kernel, slot 2: half-tag kernel. */
#define DCB_NTIMERS 4
int dcb_timing_reset(dcb_ctx*);
int dcb_timing_enable(dcb_ctx*, int on);
int dcb_timing_get(dcb_ctx*, double ms[DCB_NTIMERS], uint64_t launches[DCB_NTIMERS]);
/* Number of reads of the last run that the exact-tag kernel could not finish (queued for the next kernel), and the
   number that reached the general kernel (the same, unless the half-tag kernel ran in between). */
int dcb_last_deferred(dcb_ctx*, uint64_t* n);
int dcb_last_general(dcb_ctx*, uint64_t* n);
/* "dcb_halftag_kernel" when the half-tag kernel runs between the exact-tag and the general kernel for the resident batch
   (chains whose half tags all have >= 10 bases, one frame), else "". */
const char* dcb_halftag_kernel_name(const dcb_ctx*);
/* Name of the exact-tag kernel chosen for the resident batch ("dcb_exact_kernel_flat", "dcb_exact_kernel_spec" or
   "dcb_exact_kernel"); a static string, "" before any batch. */
const char* dcb_exact_kernel_name(const dcb_ctx*);

/* ---------------------------------------------------------------------------------------------
 * Distance primitives of the collapse step (no tag tables needed: their own light context).
 * ------------------------------------------------------------------------------------------- */
typedef struct dcb_dist dcb_dist;
dcb_dist* dcb_dist_create(int device);
void dcb_dist_destroy(dcb_dist*);

/* UMI neighbour search.  Replaces
 *     matches = prsnn.symdel(umi_list, max_edits=barcode_threshold, output_type="coo_matrix")
 *     matches = sparse.triu(matches); matches.sum_duplicates()                 (collapse.py:735-742)
 * codes[i]: UMI i, 3 bits per symbol (symbol k in bits [3k, 3k+3); the caller picks the alphabet, <= 8 symbols),
 *           length (<= 19) in bits [58, 64).
 * With codes != NULL the sorted list of pairs (row < col, Levenshtein(codes[row], codes[col]) <= max_edits,
 * ascending (row, col) = the order make_clusters walks the COO matrix in, collapse.py:773) is computed on the GPU
 * and kept; *n_pairs is its length.  With keys != NULL the kept list is copied out as row << 32 | col
 * (DCB_ENOMEM when cap is too small).  Typical use: one call with keys == NULL to size, one with codes == NULL. */
int dcb_umi_pairs(dcb_dist*, const uint64_t* codes, uint32_t n, int max_edits, uint64_t* keys, uint64_t cap,
                  uint64_t* n_pairs);
/* One GPU's share of the same search when n_parts GPUs hold the same list (an all-gather of the UMI codes): part p verifies
 * the runs of equal deletion variants whose variant hashes to p (the tile pairs numbered p modulo n_parts on the all-pairs
 * path).  The union of the parts' lists is the list of dcb_umi_pairs; a pair can be in more than one part. */
int dcb_umi_pairs_part(dcb_dist*, const uint64_t* codes, uint32_t n, int max_edits, uint32_t part, uint32_t n_parts,
                       uint64_t* keys, uint64_t cap, uint64_t* n_pairs);

/* Batch of are_seqs_equivalent(seq1, seq2, lev_threshold_fraction) (collapse.py:355-360; called at :601, :778):
 *     verdict[t] = polyleven.levenshtein(A, B) <= len(shorter of A, B) * frac        (compared in double)
 * for A = sequence a[t], B = sequence b[t].  Sequences: one byte per symbol (codes 0..7, the caller picks the
 * alphabet), sequence i at symbols[off[i] .. off[i] + len[i]), len <= 512. */
int dcb_lev_leq(dcb_dist*, const uint8_t* symbols, const uint64_t* off, const uint32_t* len, uint32_t n_seqs,
                const uint32_t* a, const uint32_t* b, uint64_t n_pairs, double frac, uint8_t* verdict);
/* The same over arbitrary byte symbols (a batch with more than eight distinct characters: lower case, the whole IUPAC
 * alphabet); the pattern then takes eight bit planes instead of three. */
int dcb_lev_leq_bytes(dcb_dist*, const uint8_t* symbols, const uint64_t* off, const uint32_t* len, uint32_t n_seqs,
                      const uint32_t* a, const uint32_t* b, uint64_t n_pairs, double frac, uint8_t* verdict);
/* Barcode extraction of the collapse step, per decombined row: replaces, for rows whose spacers are found EXACTLY,
 * get_barcode_positions (collapse.py:367-479), set_barcode (:281-326) and check_umi_quality (:340-352), for every
 * ligation-oligo design of -ol.  bc / q: the barcode region of the row (field 8 of an .n12 row) and its quality string
 * (field 9), as (offset, length) into two text buffers.  Per row:
 *   status  DCB_BC_OK, the failure the reference would count (DCB_BC_FAIL_*), or DCB_BC_HOST: an exact search of spacer 1
 *           in its window (or of spacer 2) found nothing, so the reference's fuzzy regular-expression searches decide; so
 *           also for a symbol outside ACGTN, a quality string of another length, a region longer than 250, and (TAKARA) a
 *           region shorter than the 12-symbol barcode: the caller runs the reference's own code on these rows.
 *           M13, I8: any DCB_BC_FAIL_*; I8_single: all but DCB_BC_FAIL_NOT2; NEBIO, TAKARA: DCB_BC_FAIL_N,
 *           DCB_BC_FAIL_NOSPACER (two or more exact hits in the window) and DCB_BC_FAIL_QUALITY;
 *   n1len   M13, I8, I8_single: length of N1 (4..8) once the spacers are placed (also for DCB_BC_FAIL_QUALITY): 6 = plain,
 *           < 6 padded with 'S', > 6 cut to five bases + 'L' (the readdata_short_barcode / readdata_long_barcode
 *           counters); NEBIO, TAKARA: 0 (no N1);
 *   code    the barcode as dcb_umi_pairs takes it: 3 bits per symbol, A C G T N S L = 0..6, length in bits [58, 64):
 *           N1 + N2 in 12 symbols (M13, I8, I8_single), bc[0:17] (NEBIO), bc[0:12] (TAKARA). */
enum { DCB_BC_OK = 0, DCB_BC_FAIL_N = 1, DCB_BC_FAIL_NOSPACER = 2, DCB_BC_FAIL_NOT2 = 3, DCB_BC_FAIL_N1SHORT = 4, DCB_BC_FAIL_N1LONG = 5,
       DCB_BC_FAIL_N2END = 6, DCB_BC_FAIL_QUALITY = 7, DCB_BC_HOST = 255 };
enum { DCB_OLIGO_M13 = 0, DCB_OLIGO_I8 = 1, DCB_OLIGO_I8_SINGLE = 2, DCB_OLIGO_NEBIO = 3, DCB_OLIGO_TAKARA = 4 };   /* other values: DCB_EUNSUPPORTED */
typedef struct dcb_bc_params {
    int32_t oligo;       /* DCB_OLIGO_* (inputargs["oligo"]) */
    int32_t allow_ns;    /* inputargs["allowNs"] */
    int32_t min_q;       /* inputargs["minbcQ"] */
    int32_t max_below;   /* inputargs["bcQbelowmin"] */
    double avg_q;        /* inputargs["avgQthreshold"] */
} dcb_bc_params;
int dcb_barcodes(dcb_dist*, const char* bc_text, const uint64_t* bc_off, const uint32_t* bc_len, const char* q_text,
                 const uint64_t* q_off, const uint32_t* q_len, uint64_t n, const dcb_bc_params* prm, uint8_t* status,
                 uint8_t* n1len, uint64_t* code);

/* ---------------------------------------------------------------------------------------------
 * Translate stage: get_cdr3 (translate.py:257-357) for DCR rows and the AIRR .tsv line of each, as
 * DataFrame.to_csv(sep="\t", index=False) writes it (io.py:516-548).
 *
 * Tables of one chain (host only, no GPU needed), from what import_gene_information reads
 * (translate.py:123-254): per V gene the upper-cased region, the call (name cut at '*'), the conserved
 * residue's position and residue, CDR1 / CDR2 ("" where there are none); per J gene the region, the call,
 * the motif window start and the motif.  Motifs must be four symbols, each a capital letter or '.',
 * regions upper-case IUPAC of at most 1024 bases, names and CDRs printable ASCII without '"'
 * (DCB_EUNSUPPORTED otherwise: the caller keeps the host path).
 * ------------------------------------------------------------------------------------------- */
typedef struct dcb_translate_tables dcb_translate_tables;
int dcb_translate_tables_build(int n_v, const char* const* v_regions, const char* const* v_calls, const int32_t* v_pos,
                               const char* const* v_residue, const char* const* v_cdr1, const char* const* v_cdr2, int n_j,
                               const char* const* j_regions, const char* const* j_calls, const int32_t* j_pos,
                               const char* const* j_motif, dcb_translate_tables** out);
void dcb_translate_tables_free(dcb_translate_tables*);
/* The flattened blob the kernels stage in shared memory (tests compile csrc/translate_core.cuh over it). */
int dcb_translate_tables_blob(const dcb_translate_tables*, const uint8_t** bytes, size_t* n_bytes);

/* Row flags of dcb_translate: the row is outside the device path (the host would raise, or write it otherwise). */
enum { DCB_TR_SYMBOL = 1,   /* an insert symbol outside IUPAC and U (either case) */
       DCB_TR_GENE = 2,     /* v or j out of range */
       DCB_TR_CINDEX = 4,   /* the conserved-C index lies beyond the protein */
       DCB_TR_QUOTE = 8,    /* decombinator_id holds '"', a control or a non-ASCII byte (to_csv would quote or re-encode) */
       DCB_TR_LONG = 16 };  /* the rebuilt sequence is longer than 1024 bases */

/* n rows as columns.  decombinator_id of row i is text[id_off[i], + id_len[i]) (written verbatim), its insert
 * text[ins_off[i], + ins_len[i]); freq / cluster: duplicate_count and av_UMI_cluster_size.  Row i is line
 * sequence_id = i + 1.  nonproductive_filter (-npf) drops the lines of non-productive rows; nobarcoding (-nbc)
 * writes duplicate_count 1 and an empty av_UMI_cluster_size.  Out: productive[i], row_flags[i] (DCB_TR_*),
 * *n_flagged; when no row is flagged, *out is the text of the kept lines (no header) in page-locked memory
 * (free with dcb_pinned_free), *out_bytes its size; with flagged rows *out is NULL.  d == NULL and no CUDA
 * device: DCB_ENOGPU. */
int dcb_translate(dcb_dist*, const dcb_translate_tables*, const char* text, uint64_t text_bytes, const uint32_t* v, const uint32_t* j,
                  const uint32_t* vdel, const uint32_t* jdel, const uint64_t* id_off, const uint32_t* id_len, const uint64_t* ins_off,
                  const uint32_t* ins_len, const int64_t* freq, const int64_t* cluster, uint64_t n, int nonproductive_filter,
                  int nobarcoding, uint8_t* productive, uint8_t* row_flags, uint64_t* n_flagged, char** out, uint64_t* out_bytes);

/* Device time of the last dcb_umi_pairs (pair search, incl. its sorts on the deletion-neighbourhood path),
   dcb_lev_leq kernel or dcb_translate kernels and scan (CUDA events). */
int dcb_dist_last_ms(dcb_dist*, double* ms);
/* How the last dcb_umi_pairs searched: "deletion neighbourhoods" (max_edits <= 2 and a long list: what symdel does,
   collapse.py:735-740) or "all pairs" (short lists, max_edits > 2).  The environment variable DCB_UMI_SYMDEL_MIN moves
   the switch-over (default 4096 UMIs). */
const char* dcb_dist_last_method(const dcb_dist*);

/* ---------------------------------------------------------------------------------------------
 * Synthetic workload generator (SURVEY.md 8d): deterministic in (seed, read index).
 * ------------------------------------------------------------------------------------------- */
typedef struct dcb_synth_params {
    uint64_t seed;
    uint32_t read_len;     /* R1 length */
    uint32_t read2_len;    /* R2 length (barcode read); 0 = none */
    uint32_t sub_rate;     /* per-base substitution probability * 2^32 */
    uint32_t n_rate;       /* per-base N probability * 2^32 */
    uint32_t junk_rate;    /* probability * 2^32 that a read is random sequence (no TCR) */
    uint32_t umi_pool;     /* != 0: read i is a copy of molecule i % umi_pool (same rearrangement, same UMI) */
    uint32_t sub_rate2;    /* per-base substitution probability * 2^32 in R2 (the barcode read) */
    uint32_t reserved;
} dcb_synth_params;
typedef struct dcb_synth dcb_synth;
dcb_synth* dcb_synth_create(const dcb_synth_params* p, int n_sets, const char* const* const* v_regions,
                            const int* n_v, const char* const* const* j_regions, const int* n_j);
void dcb_synth_destroy(dcb_synth*);
/* r1: n*read_len bytes; r2: n*read2_len bytes or NULL.  No terminators. */
int dcb_synth_reads(const dcb_synth*, uint64_t first_index, uint64_t n, char* r1, char* r2, int n_threads);

#ifdef __cplusplus
}
#endif
#endif /* DCB_H */
