"""ctypes binding of libdcb.so (include/dcb.h).  Thin: every call is a C-ABI call.

The library is built in-tree by ``decombinator_b200.build``.  There is no Python or CPU fallback
for the compute entry points: if the library is missing it is built, if that fails or no GPU is
usable the call raises.
"""
import ctypes
import os

import numpy as np

from . import build as _build

_HERE = os.path.dirname(os.path.abspath(__file__))

NCOUNTERS = 20
NTIMERS = 4

RESULT_DTYPE = np.dtype([
    ("status", "u1"), ("frame", "u1"), ("v", "u1"), ("j", "u1"),
    ("vdel", "<u2"), ("jdel", "<u2"), ("ins_start", "<u2"), ("ins_end", "<u2"),
    ("v_seq_start", "<u2"), ("j_seq_end", "<u2"),
])
assert RESULT_DTYPE.itemsize == 16


class DcbError(RuntimeError):
    pass


class CPacked(ctypes.Structure):
    _fields_ = [
        ("n_reads", ctypes.c_uint64), ("slot_words", ctypes.c_uint32), ("uniform_len", ctypes.c_uint32),
        ("max_len", ctypes.c_uint32), ("n_exc", ctypes.c_uint32),
        ("words", ctypes.POINTER(ctypes.c_uint32)), ("lens", ctypes.POINTER(ctypes.c_uint16)),
        ("flags", ctypes.POINTER(ctypes.c_uint32)), ("exc_read", ctypes.POINTER(ctypes.c_uint32)),
        ("exc_pos", ctypes.POINTER(ctypes.c_uint16)), ("exc_kind", ctypes.POINTER(ctypes.c_uint8)),
        ("owner", ctypes.c_void_p),
    ]


class CParams(ctypes.Structure):
    _fields_ = [("both_frames", ctypes.c_int32), ("allow_ns", ctypes.c_int32), ("lenthreshold", ctypes.c_int32),
                ("force_general", ctypes.c_int32)]


class CBcParams(ctypes.Structure):
    _fields_ = [("oligo", ctypes.c_int32), ("allow_ns", ctypes.c_int32), ("min_q", ctypes.c_int32), ("max_below", ctypes.c_int32),
                ("avg_q", ctypes.c_double)]


BC_OK, BC_FAIL_N, BC_FAIL_NOSPACER, BC_FAIL_NOT2, BC_FAIL_N1SHORT, BC_FAIL_N1LONG, BC_FAIL_N2END, BC_FAIL_QUALITY, BC_HOST = 0, 1, 2, 3, 4, 5, 6, 7, 255
OLIGOS_ON_DEVICE = {"m13": 0, "i8": 1, "i8_single": 2, "nebio": 3, "takara": 4}   # -ol (lower case) -> DCB_OLIGO_*
BC_LENGTH = {"m13": 12, "i8": 12, "i8_single": 12, "nebio": 17, "takara": 12}      # symbols of the barcode dcb_barcodes assembles
BC_FIXED = ("nebio", "takara")                  # designs whose barcode is a fixed slice of the region (no N1 / N2)


class CSynthParams(ctypes.Structure):
    _fields_ = [("seed", ctypes.c_uint64), ("read_len", ctypes.c_uint32), ("read2_len", ctypes.c_uint32),
                ("sub_rate", ctypes.c_uint32), ("n_rate", ctypes.c_uint32), ("junk_rate", ctypes.c_uint32),
                ("umi_pool", ctypes.c_uint32), ("sub_rate2", ctypes.c_uint32), ("reserved", ctypes.c_uint32)]


_lib = None


def lib():
    """Load (building if needed) libdcb.so and declare the prototypes of include/dcb.h."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("DCB_LIB") or _build.build()   # DCB_LIB: a tuning build of the same sources (tools/variants.sh)
    L = ctypes.CDLL(path)
    vp, i32, u64, u32 = ctypes.c_void_p, ctypes.c_int, ctypes.c_uint64, ctypes.c_uint32
    cpp = ctypes.POINTER(ctypes.c_char_p)
    L.dcb_last_error.restype = ctypes.c_char_p
    L.dcb_abi_version.restype = i32
    L.dcb_counter_name.restype = ctypes.c_char_p
    L.dcb_counter_name.argtypes = [i32]
    L.dcb_tagset_build.restype = vp
    L.dcb_tagset_build.argtypes = [cpp, ctypes.POINTER(ctypes.c_int32), cpp, i32, i32, i32]
    L.dcb_tagset_free.argtypes = [vp]
    L.dcb_tagset_table_bytes.restype = ctypes.c_size_t
    L.dcb_tagset_table_bytes.argtypes = [vp]
    L.dcb_tagset_blob.argtypes = [vp, i32, ctypes.POINTER(ctypes.POINTER(ctypes.c_uint32)), ctypes.POINTER(ctypes.c_size_t)]
    L.dcb_tagset_union_index.argtypes = [vp, vp, vp, ctypes.c_size_t, ctypes.POINTER(ctypes.c_size_t)]
    L.dcb_tagset_suffix_filter.argtypes = [vp, vp, vp, ctypes.c_size_t, ctypes.POINTER(ctypes.c_size_t)]
    L.dcb_tagset_half_index.argtypes = [vp, vp, vp, ctypes.c_size_t, ctypes.POINTER(ctypes.c_size_t)]
    L.dcb_fastq_index_build.argtypes = [vp, u64, i32, ctypes.POINTER(ctypes.POINTER(CFastqIndex))]
    L.dcb_fastq_index_free.argtypes = [ctypes.POINTER(CFastqIndex)]
    L.dcb_fastq_index_free.restype = None
    L.dcb_count_ranges_with.argtypes = [vp, vp, vp, u64, i32, i32]
    L.dcb_count_ranges_with.restype = u64
    L.dcb_format_rows.argtypes = [vp, u64, i32] + [ctypes.POINTER(CColumn)] * 6 + [ctypes.c_char_p, i32,
                                  ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(u64), ctypes.POINTER(u64)]
    L.dcb_buffer_free.argtypes = [ctypes.c_void_p]
    L.dcb_buffer_free.restype = None
    L.dcb_format_collapse_rows.argtypes = [vp, u64, i32] + [ctypes.POINTER(CColumn)] * 3 + [i32, ctypes.POINTER(ctypes.c_void_p),
                                           ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint64)]
    L.dcb_format_collapse_rows.restype = ctypes.c_int
    L.dcb_n12_index.argtypes = [vp, u64, i32, ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(u64)]
    L.dcb_n12_index.restype = ctypes.c_int
    L.dcb_n12_collapse_rows.argtypes = [vp, vp, vp, u64, vp, i32, ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(u64), ctypes.POINTER(u64)]
    L.dcb_n12_collapse_rows.restype = ctypes.c_int
    pu64 = ctypes.POINTER(u64)
    L.dcb_bgzf_inflate.argtypes = [vp, vp, vp, vp, vp, u64, vp, i32]
    L.dcb_bgzf_inflate.restype = ctypes.c_int
    L.dcb_group_create.argtypes = [vp, u64, u64, vp, vp, ctypes.POINTER(ctypes.c_void_p)]
    L.dcb_group_step.argtypes = [vp, pu64]
    L.dcb_group_pairs.argtypes = [vp, pu64, pu64, vp, vp, vp, vp, vp, ctypes.POINTER(ctypes.c_int)]
    L.dcb_group_verdicts.argtypes = [vp, vp, u64]
    L.dcb_group_result.argtypes = [vp, pu64, pu64, pu64, pu64, vp, vp, vp, vp, vp]
    L.dcb_group_free.argtypes = [vp]
    L.dcb_group_free.restype = None
    for f in (L.dcb_group_create, L.dcb_group_step, L.dcb_group_pairs, L.dcb_group_verdicts, L.dcb_group_result):
        f.restype = ctypes.c_int
    L.dcb_pack_reads.argtypes = [vp, vp, vp, u64, i32, i32, ctypes.POINTER(ctypes.POINTER(CPacked))]
    L.dcb_packed_free.argtypes = [ctypes.POINTER(CPacked)]
    L.dcb_pack_words.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_uint32,
                                 ctypes.c_int, ctypes.c_uint32, ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(ctypes.c_int)]
    L.dcb_pack_words.restype = ctypes.c_int
    L.dcb_unpack_read.argtypes = [ctypes.POINTER(CPacked), u64, ctypes.c_char_p, u32]
    L.dcb_ctx_create.restype = vp
    L.dcb_ctx_create.argtypes = [i32, vp, vp, ctypes.POINTER(CParams)]
    L.dcb_ctx_destroy.argtypes = [vp]
    L.dcb_ctx_set_stream.argtypes = [vp, vp]
    L.dcb_decombine_batch.argtypes = [vp, ctypes.POINTER(CPacked), vp, vp]
    L.dcb_decombine_ascii.argtypes = [vp, vp, vp, vp, u64, u32, i32, vp, vp]
    L.dcb_pack_device.argtypes = [vp, vp, vp, vp, u64, u32, i32, ctypes.POINTER(ctypes.POINTER(CPacked))]
    L.dcb_pack_device_ms.argtypes = [vp, ctypes.POINTER(ctypes.c_double)]
    L.dcb_last_pack_shares.argtypes = [vp, ctypes.POINTER(ctypes.c_uint32), ctypes.POINTER(ctypes.c_uint32)]
    L.dcb_last_pack_shares.restype = ctypes.c_int
    L.dcb_pinned_alloc.restype = vp
    L.dcb_pinned_alloc.argtypes = [ctypes.c_size_t]
    L.dcb_pinned_free.argtypes = [vp]
    L.dcb_upload.argtypes = [vp, ctypes.POINTER(CPacked)]
    L.dcb_run_resident.argtypes = [vp]
    L.dcb_download.argtypes = [vp, vp, vp]
    L.dcb_timing_reset.argtypes = [vp]
    L.dcb_timing_enable.argtypes = [vp, i32]
    L.dcb_timing_get.argtypes = [vp, vp, vp]
    L.dcb_last_deferred.argtypes = [vp, ctypes.POINTER(u64)]
    L.dcb_last_general.argtypes = [vp, ctypes.POINTER(u64)]
    L.dcb_halftag_kernel_name.argtypes = [vp]
    L.dcb_halftag_kernel_name.restype = ctypes.c_char_p
    L.dcb_exact_kernel_name.argtypes = [vp]
    L.dcb_exact_kernel_name.restype = ctypes.c_char_p
    L.dcb_dist_create.restype = vp
    L.dcb_dist_create.argtypes = [i32]
    L.dcb_dist_destroy.argtypes = [vp]
    L.dcb_umi_pairs.argtypes = [vp, vp, u32, i32, vp, u64, ctypes.POINTER(u64)]
    L.dcb_umi_pairs_part.argtypes = [vp, vp, u32, i32, u32, u32, vp, u64, ctypes.POINTER(u64)]
    L.dcb_lev_leq.argtypes = [vp, vp, vp, vp, u32, vp, vp, u64, ctypes.c_double, vp]
    L.dcb_lev_leq_bytes.argtypes = [vp, vp, vp, vp, u32, vp, vp, u64, ctypes.c_double, vp]
    L.dcb_barcodes.argtypes = [vp, vp, vp, vp, vp, vp, vp, u64, ctypes.POINTER(CBcParams), vp, vp, vp]
    L.dcb_dist_last_ms.argtypes = [vp, ctypes.POINTER(ctypes.c_double)]
    L.dcb_dist_last_method.argtypes = [vp]
    L.dcb_dist_last_method.restype = ctypes.c_char_p
    L.dcb_synth_create.restype = vp
    L.dcb_synth_create.argtypes = [ctypes.POINTER(CSynthParams), i32, ctypes.POINTER(cpp), ctypes.POINTER(ctypes.c_int),
                                   ctypes.POINTER(cpp), ctypes.POINTER(ctypes.c_int)]
    L.dcb_synth_destroy.argtypes = [vp]
    L.dcb_synth_reads.argtypes = [vp, u64, u64, vp, vp, i32]
    _lib = L
    return L


def _check(rc, what):
    if rc != 0:
        raise DcbError("%s failed (%d): %s" % (what, rc, lib().dcb_last_error().decode()))


def counter_names():
    L = lib()
    return [L.dcb_counter_name(i).decode() for i in range(NCOUNTERS)]


def _carr(strings):
    arr = (ctypes.c_char_p * len(strings))()
    arr[:] = [s.encode() if isinstance(s, str) else s for s in strings]
    return arr


class TagTables:
    """dcb_tagset: the flattened automaton/bitmap tables of one gene (V or J)."""

    def __init__(self, tags, jumps, regions, half_split, is_v):
        L = lib()
        n = len(tags)
        self._h = L.dcb_tagset_build(_carr(tags), (ctypes.c_int32 * n)(*jumps), _carr(list(regions)[:n]), n,
                                     int(half_split), int(is_v))
        if not self._h:
            raise DcbError("dcb_tagset_build: " + L.dcb_last_error().decode())

    @property
    def handle(self):
        return self._h

    def table_bytes(self):
        return lib().dcb_tagset_table_bytes(self._h)

    def blob(self, which):
        p = ctypes.POINTER(ctypes.c_uint32)()
        n = ctypes.c_size_t()
        _check(lib().dcb_tagset_blob(self._h, which, ctypes.byref(p), ctypes.byref(n)), "dcb_tagset_blob")
        return np.ctypeslib.as_array(p, shape=(n.value,))

    def __del__(self):
        try:
            if self._h:
                lib().dcb_tagset_free(self._h)
                self._h = None
        except Exception:
            pass


def union_index(vt: "TagTables", jt: "TagTables"):
    """Seed index over both genes (what dcb_ctx_create builds), or None when their seed geometries differ."""
    n = ctypes.c_size_t()
    if lib().dcb_tagset_union_index(vt.handle, jt.handle, None, 0, ctypes.byref(n)) != 0:
        return None
    out = np.zeros(n.value, dtype=np.uint32)
    _check(lib().dcb_tagset_union_index(vt.handle, jt.handle, out.ctypes.data, n.value, ctypes.byref(n)), "dcb_tagset_union_index")
    return out


def half_index(vt: "TagTables", jt: "TagTables"):
    """Sampled half-tag index of the chain (what the half-tag kernel searches with), or None when a half tag is too short."""
    n = ctypes.c_size_t()
    if lib().dcb_tagset_half_index(vt.handle, jt.handle, None, 0, ctypes.byref(n)) != 0:
        return None
    out = np.zeros(n.value, dtype=np.uint32)
    _check(lib().dcb_tagset_half_index(vt.handle, jt.handle, out.ctypes.data, n.value, ctypes.byref(n)), "dcb_tagset_half_index")
    return out


def suffix_filter(vt: "TagTables", jt: "TagTables"):
    """Union suffix filter of the chain's six keyword sets (what the general kernel marks candidate positions with)."""
    n = ctypes.c_size_t()
    _check(lib().dcb_tagset_suffix_filter(vt.handle, jt.handle, None, 0, ctypes.byref(n)), "dcb_tagset_suffix_filter")
    out = np.zeros(n.value, dtype=np.uint32)
    _check(lib().dcb_tagset_suffix_filter(vt.handle, jt.handle, out.ctypes.data, n.value, ctypes.byref(n)), "dcb_tagset_suffix_filter")
    return out


class Packed:
    """dcb_packed: 2-bit packed read slots (+ sparse non-ACGT list) in page-locked host memory."""

    def __init__(self, ptr):
        self._p = ptr

    @property
    def c(self):
        return self._p

    @property
    def n_reads(self):
        return int(self._p.contents.n_reads)

    @property
    def slot_words(self):
        return int(self._p.contents.slot_words)

    @property
    def n_exc(self):
        return int(self._p.contents.n_exc)

    @property
    def uniform_len(self):
        return int(self._p.contents.uniform_len)

    @property
    def max_len(self):
        return int(self._p.contents.max_len)

    def arrays(self):
        """Every array of the batch as numpy copies (words, lens, flags, exc_read, exc_pos, exc_kind)."""
        c, n, ne = self._p.contents, self.n_reads, self.n_exc

        def arr(ptr, count):
            return np.ctypeslib.as_array(ptr, shape=(max(1, count),))[:count].copy()
        return {"words": arr(c.words, n * self.slot_words), "lens": arr(c.lens, n), "flags": arr(c.flags, (n + 31) // 32),
                "exc_read": arr(c.exc_read, ne), "exc_pos": arr(c.exc_pos, ne), "exc_kind": arr(c.exc_kind, ne)}

    def words(self):
        c = self._p.contents
        return np.ctypeslib.as_array(c.words, shape=(max(1, self.n_reads * self.slot_words),))[: self.n_reads * self.slot_words]

    def nbytes(self):
        c = self._p.contents
        n = self.n_reads
        return n * self.slot_words * 4 + n * 2 + ((n + 31) // 32) * 4 + c.n_exc * 7

    def h2d_bytes(self):
        """Bytes dcb_decombine_batch copies to the device for this batch."""
        c = self._p.contents
        n = self.n_reads
        return n * self.slot_words * 4 + (0 if c.uniform_len else n * 2) + ((((n + 31) // 32) * 4 + c.n_exc * 7) if c.n_exc else 0)

    def unpack(self, i):
        buf = ctypes.create_string_buffer(self.max_len + 1)
        n = lib().dcb_unpack_read(self._p, i, buf, self.max_len + 1)
        if n < 0:
            raise DcbError("dcb_unpack_read")
        return buf.raw[:n].decode()

    def free(self):
        if self._p is not None:
            lib().dcb_packed_free(self._p)
            self._p = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class CColumn(ctypes.Structure):
    _fields_ = [("text", ctypes.c_void_p), ("off", ctypes.c_void_p), ("len", ctypes.c_void_p)]


def format_rows(res, packed_revcomp, columns, sep, n_threads=None):
    """dcb_format_rows: the rows of every decombined read as one text buffer (fields joined by sep, one row per line).

    columns: (ids, vdj, vdjqual, bc, bcq, v_tail-or-None), each an object with .buf (bytes), .off (uint64), .len (uint32).
    -> (bytes, number of rows)"""
    keep, cols = [], []
    for col in columns:
        if col is None:
            cols.append(None)
            continue
        buf = np.frombuffer(col.buf, dtype=np.uint8)
        off = np.ascontiguousarray(col.off, dtype=np.uint64)
        ln = np.ascontiguousarray(col.len, dtype=np.uint32)
        keep.append((buf, off, ln))
        cols.append(ctypes.pointer(CColumn(buf.ctypes.data, off.ctypes.data, ln.ctypes.data)))
    res = np.ascontiguousarray(res)
    out, nbytes, nrows = ctypes.c_void_p(), ctypes.c_uint64(), ctypes.c_uint64()
    nt = n_threads or min(32, os.cpu_count() or 1)
    _check(lib().dcb_format_rows(res.ctypes.data, len(res), int(bool(packed_revcomp)), *cols, sep.encode("ascii"), nt,
                                 ctypes.byref(out), ctypes.byref(nbytes), ctypes.byref(nrows)), "dcb_format_rows")
    return NativeText(out.value, nbytes.value), int(nrows.value)


def pack_words(buf, off, length, revcomp, slot_words, uniform_len=0, first=0, count=None, n_threads=None, out=None):
    """dcb_pack_words: reads of nothing but A / C / G / T packed by the host threads into a uint32 array of
    count * slot_words words.  -> (words, clean); clean False: another symbol turned up, the words are void."""
    buf = np.frombuffer(buf, dtype=np.uint8) if not isinstance(buf, np.ndarray) else buf
    if off is not None:
        off = np.ascontiguousarray(off, dtype=np.uint64)
    if length is not None:
        length = np.ascontiguousarray(length, dtype=np.uint32)
    n = len(off) if off is not None else (len(buf) // uniform_len if uniform_len else 0)
    count = n - first if count is None else count
    words = out if out is not None else np.empty(count * slot_words, dtype=np.uint32)
    clean = ctypes.c_int(0)
    _check(lib().dcb_pack_words(buf.ctypes.data, off.ctypes.data if off is not None else None,
                                length.ctypes.data if length is not None else None, int(first), int(count), int(uniform_len),
                                int(bool(revcomp)), int(slot_words), words.ctypes.data,
                                n_threads or min(32, os.cpu_count() or 1), ctypes.byref(clean)), "dcb_pack_words")
    return words, bool(clean.value)


def format_collapse_rows(res, packed_revcomp, columns, n_threads=None):
    """dcb_format_collapse_rows: three lines per decombined read -- tcrseq, str(row[:5]) and the "|"-joined
    (str(row[:5]), tcrseq, tcrQ, read id) collapse files its rows under.  columns: (ids, vdj, vdjqual, ...).
    -> (NativeText, number of rows)"""
    keep, cols = [], []
    for col in columns[:3]:
        buf = np.frombuffer(col.buf, dtype=np.uint8)
        off = np.ascontiguousarray(col.off, dtype=np.uint64)
        ln = np.ascontiguousarray(col.len, dtype=np.uint32)
        keep.append((buf, off, ln))
        cols.append(ctypes.pointer(CColumn(buf.ctypes.data, off.ctypes.data, ln.ctypes.data)))
    res = np.ascontiguousarray(res)
    out, nbytes, nrows = ctypes.c_void_p(), ctypes.c_uint64(), ctypes.c_uint64()
    nt = n_threads or min(32, os.cpu_count() or 1)
    _check(lib().dcb_format_collapse_rows(res.ctypes.data, len(res), int(bool(packed_revcomp)), *cols, nt,
                                          ctypes.byref(out), ctypes.byref(nbytes), ctypes.byref(nrows)), "dcb_format_collapse_rows")
    return NativeText(out.value, nbytes.value), int(nrows.value)


def n12_index(text, n_threads=None):
    """dcb_n12_index: (off, len) arrays of shape (rows, 10) over an .n12 text (uint8 array), or None when the text is not ten
    ", "-joined fields per row."""
    off, ln, n = ctypes.c_void_p(), ctypes.c_void_p(), ctypes.c_uint64(0)
    _check(lib().dcb_n12_index(text.ctypes.data, len(text), n_threads or min(32, os.cpu_count() or 1), ctypes.byref(off), ctypes.byref(ln),
                               ctypes.byref(n)), "dcb_n12_index")
    if n.value == 0:
        return None
    try:
        o = np.ctypeslib.as_array(ctypes.cast(off, ctypes.POINTER(ctypes.c_uint64)), shape=(n.value * 10,)).reshape(n.value, 10).copy()
        l = np.ctypeslib.as_array(ctypes.cast(ln, ctypes.POINTER(ctypes.c_uint32)), shape=(n.value * 10,)).reshape(n.value, 10).copy()
    finally:
        lib().dcb_buffer_free(off)
        lib().dcb_buffer_free(ln)
    return o, l


def n12_collapse_rows(text, off, ln, keep, n_threads=None):
    """dcb_n12_collapse_rows -> (NativeText, rows) or None when a field cannot be written the way str() writes it."""
    off, ln = np.ascontiguousarray(off, dtype=np.uint64), np.ascontiguousarray(ln, dtype=np.uint32)
    keep = np.ascontiguousarray(keep, dtype=np.uint8)
    out, nbytes, nrows = ctypes.c_void_p(), ctypes.c_uint64(), ctypes.c_uint64()
    _check(lib().dcb_n12_collapse_rows(text.ctypes.data, off.ctypes.data, ln.ctypes.data, len(off), keep.ctypes.data,
                                       n_threads or min(32, os.cpu_count() or 1), ctypes.byref(out), ctypes.byref(nbytes),
                                       ctypes.byref(nrows)), "dcb_n12_collapse_rows")
    if nrows.value == 0xFFFFFFFFFFFFFFFF:
        return None
    return NativeText(out.value, nbytes.value), int(nrows.value)


def bgzf_inflate(raw, start, end, isize, out_off, out, n_threads=None):
    """dcb_bgzf_inflate: raw / out are uint8 arrays (views of the compressed file and of the buffer to fill)."""
    start, end = np.ascontiguousarray(start, dtype=np.uint64), np.ascontiguousarray(end, dtype=np.uint64)
    isize, out_off = np.ascontiguousarray(isize, dtype=np.uint32), np.ascontiguousarray(out_off, dtype=np.uint64)
    _check(lib().dcb_bgzf_inflate(raw.ctypes.data, start.ctypes.data, end.ctypes.data, isize.ctypes.data, out_off.ctypes.data, len(start),
                                  out.ctypes.data, n_threads or min(32, os.cpu_count() or 1)), "dcb_bgzf_inflate")


class Grouping:
    """dcb_group: the grouping of collapse's read_in_data over columns (csrc/group.cpp).  seqs: bytes of the rows' inter-tag
    sequences joined by newlines; code / idx: barcode code and global row index per row.  ``run(verdicts)`` drives the
    rounds: verdicts(symbols, off, len, a, b) -> bool array is the caller's route to the GPU (Dist.lev_leq)."""

    def __init__(self, seqs, code, idx):
        self._seqs = seqs                                  # the library reads the text in place
        self._buf = np.frombuffer(seqs, dtype=np.uint8)
        self._h = ctypes.c_void_p()
        code = np.ascontiguousarray(code, dtype=np.uint64)
        idx = np.ascontiguousarray(idx, dtype=np.uint64)
        _check(lib().dcb_group_create(self._buf.ctypes.data if len(self._buf) else None, len(self._buf), len(code), code.ctypes.data,
                                      idx.ctypes.data, ctypes.byref(self._h)), "dcb_group_create")

    def run(self, verdicts):
        L = lib()
        n_pairs = ctypes.c_uint64()
        while True:
            _check(L.dcb_group_step(self._h, ctypes.byref(n_pairs)), "dcb_group_step")
            if n_pairs.value == 0:
                break
            ns, nsym, coded = ctypes.c_uint64(), ctypes.c_uint64(), ctypes.c_int()
            _check(L.dcb_group_pairs(self._h, ctypes.byref(ns), ctypes.byref(nsym), None, None, None, None, None, None), "dcb_group_pairs")
            sym = np.zeros(max(1, nsym.value), dtype=np.uint8)
            off, ln = np.zeros(ns.value, dtype=np.uint64), np.zeros(ns.value, dtype=np.uint32)
            a, b = np.zeros(n_pairs.value, dtype=np.uint32), np.zeros(n_pairs.value, dtype=np.uint32)
            _check(L.dcb_group_pairs(self._h, ctypes.byref(ns), ctypes.byref(nsym), sym.ctypes.data, off.ctypes.data, ln.ctypes.data,
                                     a.ctypes.data, b.ctypes.data, ctypes.byref(coded)), "dcb_group_pairs")
            same = np.ascontiguousarray(verdicts(sym[:nsym.value], off, ln, a, b), dtype=np.uint8)
            _check(L.dcb_group_verdicts(self._h, same.ctypes.data, len(same)), "dcb_group_verdicts")

    def result(self):
        """-> (code uint64[g], tick uint64[g], proto_row uint32[g], first uint64[g + 1], rows uint32[members], dropped, dead)"""
        L = lib()
        ng, nm, dr, dd = ctypes.c_uint64(), ctypes.c_uint64(), ctypes.c_uint64(), ctypes.c_uint64()
        args = [ctypes.byref(ng), ctypes.byref(nm), ctypes.byref(dr), ctypes.byref(dd)]
        _check(L.dcb_group_result(self._h, *args, None, None, None, None, None), "dcb_group_result")
        code, tick, proto = np.zeros(ng.value, dtype=np.uint64), np.zeros(ng.value, dtype=np.uint64), np.zeros(ng.value, dtype=np.uint32)
        first, rows = np.zeros(ng.value + 1, dtype=np.uint64), np.zeros(max(1, nm.value), dtype=np.uint32)
        _check(L.dcb_group_result(self._h, *args, code.ctypes.data, tick.ctypes.data, proto.ctypes.data, first.ctypes.data, rows.ctypes.data),
               "dcb_group_result")
        return code, tick, proto, first, rows[:nm.value], int(dr.value), int(dd.value)

    def close(self):
        if self._h:
            lib().dcb_group_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class NativeText:
    """A text buffer malloc'ed by the library (dcb_format_rows), handed on WITHOUT a copy: `.a` is a uint8 array over it,
    bytes(obj) / obj.tobytes() copy, the buffer is freed with the object."""

    def __init__(self, ptr, nbytes):
        self._p, self._n = ptr, int(nbytes)
        self.a = np.frombuffer((ctypes.c_uint8 * max(1, self._n)).from_address(ptr), dtype=np.uint8, count=self._n)

    def __len__(self):
        return self._n

    def tobytes(self):
        return self.a.tobytes()

    __bytes__ = tobytes

    def decode(self, *a):
        return self.tobytes().decode(*a)

    def __del__(self):
        try:
            if self._p:
                self.a = None
                lib().dcb_buffer_free(self._p)
                self._p = None
        except Exception:
            pass


class CFastqIndex(ctypes.Structure):
    _fields_ = [("n_records", ctypes.c_uint64),
                ("name_off", ctypes.POINTER(ctypes.c_uint64)), ("name_len", ctypes.POINTER(ctypes.c_uint32)),
                ("seq_off", ctypes.POINTER(ctypes.c_uint64)), ("seq_len", ctypes.POINTER(ctypes.c_uint32)),
                ("qual_off", ctypes.POINTER(ctypes.c_uint64)), ("qual_len", ctypes.POINTER(ctypes.c_uint32)),
                ("strict", ctypes.c_int32)]


def fastq_index(data, n_threads=None):
    """dcb_fastq_index_build over FASTQ text in memory (bytes / uint8 array).

    -> dict of numpy arrays (name_off, name_len, seq_off, seq_len, qual_off, qual_len), or None when the text is not in
    the strict four-line layout (the caller then uses the general parser)."""
    buf = np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else data
    out = ctypes.POINTER(CFastqIndex)()
    nt = n_threads or min(32, os.cpu_count() or 1)
    rc = lib().dcb_fastq_index_build(buf.ctypes.data if len(buf) else None, len(buf), nt, ctypes.byref(out))
    try:
        _check(rc, "dcb_fastq_index_build")
        ix = out.contents
        if not ix.strict:
            return None
        n = int(ix.n_records)
        res = {}
        owner = _FastqIndexOwner(out)      # the arrays are views of the index's own memory: it lives as long as any of them
        out = None
        for name, ctype, dt in (("name_off", ctypes.c_uint64, np.uint64), ("name_len", ctypes.c_uint32, np.uint32),
                                ("seq_off", ctypes.c_uint64, np.uint64), ("seq_len", ctypes.c_uint32, np.uint32),
                                ("qual_off", ctypes.c_uint64, np.uint64), ("qual_len", ctypes.c_uint32, np.uint32)):
            if not n:
                res[name] = np.zeros(0, dt)
                continue
            carr = (ctype * n).from_address(ctypes.addressof(getattr(ix, name).contents))
            carr._owner = owner
            res[name] = np.frombuffer(carr, dtype=dt, count=n)
        return res
    finally:
        if out:
            lib().dcb_fastq_index_free(out)


class _FastqIndexOwner:
    def __init__(self, ptr):
        self._p = ptr

    def __del__(self):
        try:
            if self._p:
                lib().dcb_fastq_index_free(self._p)
                self._p = None
        except Exception:
            pass


def count_ranges_with(buf, off, length, symbol, n_threads=None):
    """How many of the byte ranges (off[i], length[i]) of buf contain `symbol` (one character)."""
    buf = np.frombuffer(buf, dtype=np.uint8) if not isinstance(buf, np.ndarray) else buf
    off = np.ascontiguousarray(off, dtype=np.uint64)
    length = np.ascontiguousarray(length, dtype=np.uint32)
    if len(off) == 0:
        return 0
    nt = n_threads or min(32, os.cpu_count() or 1)
    return int(lib().dcb_count_ranges_with(buf.ctypes.data, off.ctypes.data, length.ctypes.data, len(off), ord(symbol), nt))


class PinnedBytes:
    """A page-locked uint8 buffer (dcb_pinned_alloc) as a numpy array `.a`; host->device copies from it run at link speed."""

    def __init__(self, src):
        src = np.ascontiguousarray(src, dtype=np.uint8).reshape(-1)
        self._n = len(src)
        self._p = lib().dcb_pinned_alloc(self._n + 64)
        if not self._p:
            raise DcbError("dcb_pinned_alloc: " + lib().dcb_last_error().decode())
        self.a = np.frombuffer((ctypes.c_uint8 * (self._n + 64)).from_address(self._p), dtype=np.uint8, count=self._n)
        self.a[:] = src

    def free(self):
        if self._p:
            self.a = None
            lib().dcb_pinned_free(self._p)
            self._p = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def pack_arrays(buf, off, length, revcomp, n_threads=None) -> Packed:
    """dcb_pack_reads over reads stored in one uint8 buffer (off: uint64 offsets, length: uint32)."""
    buf = np.ascontiguousarray(buf, dtype=np.uint8)
    off = np.ascontiguousarray(off, dtype=np.uint64)
    length = np.ascontiguousarray(length, dtype=np.uint32)
    out = ctypes.POINTER(CPacked)()
    nt = n_threads or min(32, os.cpu_count() or 1)
    _check(lib().dcb_pack_reads(buf.ctypes.data, off.ctypes.data, length.ctypes.data, len(off), int(bool(revcomp)), nt,
                                ctypes.byref(out)), "dcb_pack_reads")
    return Packed(out)


def pack_strings(reads, revcomp, n_threads=1) -> Packed:
    bufs = [r.encode("latin-1") if isinstance(r, str) else r for r in reads]
    length = np.array([len(b) for b in bufs], dtype=np.uint32)
    off = np.zeros(len(bufs), dtype=np.uint64)
    if len(bufs) > 1:
        off[1:] = np.cumsum(length[:-1], dtype=np.uint64)
    buf = np.frombuffer(b"".join(bufs) + b"\0", dtype=np.uint8)
    return pack_arrays(buf, off, length, revcomp, n_threads)


class Context:
    """dcb_ctx: device tables + batch buffers + stream of one GPU."""

    def __init__(self, vset: TagTables, jset: TagTables, device=0, both_frames=False, allow_ns=False,
                 lenthreshold=130, force_general=False):
        L = lib()
        prm = CParams(int(bool(both_frames)), int(bool(allow_ns)), int(lenthreshold), int(force_general))
        self._keep = (vset, jset)
        self._h = L.dcb_ctx_create(int(device), vset.handle, jset.handle, ctypes.byref(prm))
        if not self._h:
            raise DcbError("dcb_ctx_create: " + L.dcb_last_error().decode())

    def set_stream(self, cuda_stream):
        _check(lib().dcb_ctx_set_stream(self._h, ctypes.c_void_p(cuda_stream)), "dcb_ctx_set_stream")

    def _pinned_results(self, n):
        """A page-locked result array of n records (dcb_pinned_alloc), kept and reused while it is large enough."""
        if getattr(self, "_pin_cap", 0) < n:
            if getattr(self, "_pin_ptr", None):
                lib().dcb_pinned_free(self._pin_ptr)
            self._pin_cap = max(n, 1)
            self._pin_ptr = lib().dcb_pinned_alloc(self._pin_cap * RESULT_DTYPE.itemsize)
            if not self._pin_ptr:
                raise DcbError("dcb_pinned_alloc: " + lib().dcb_last_error().decode())
        buf = (ctypes.c_uint8 * (n * RESULT_DTYPE.itemsize)).from_address(self._pin_ptr)
        return np.frombuffer(buf, dtype=RESULT_DTYPE, count=n)

    def decombine(self, packed: Packed, counters=None, pinned=False):
        """dcb_decombine_batch: host buffers in, host buffers out.  pinned=True returns a view of a page-locked buffer
        owned by this context (valid until the next pinned call) instead of a fresh array."""
        res = self._pinned_results(packed.n_reads) if pinned else np.zeros(packed.n_reads, dtype=RESULT_DTYPE)
        if counters is None:
            counters = np.zeros(NCOUNTERS, dtype=np.uint64)
        _check(lib().dcb_decombine_batch(self._h, packed.c, res.ctypes.data, counters.ctypes.data), "dcb_decombine_batch")
        return res, counters

    @staticmethod
    def _ascii_args(buf, off, length, uniform_len):
        buf = np.ascontiguousarray(buf, dtype=np.uint8) if not (isinstance(buf, np.ndarray) and buf.dtype == np.uint8 and buf.flags.c_contiguous) else buf
        n = len(length) if length is not None else (len(off) if off is not None else (len(buf) // uniform_len if uniform_len else 0))
        off = None if off is None else np.ascontiguousarray(off, dtype=np.uint64)
        length = None if (length is None or uniform_len) else np.ascontiguousarray(length, dtype=np.uint32)
        return buf, off, length, n

    def last_pack_shares(self):
        """(chunks packed by the host threads, chunks packed by the device) of the last decombine_ascii call."""
        a, b = ctypes.c_uint32(0), ctypes.c_uint32(0)
        _check(lib().dcb_last_pack_shares(self._h, ctypes.byref(a), ctypes.byref(b)), "dcb_last_pack_shares")
        return int(a.value), int(b.value)

    def decombine_ascii(self, buf, off, length, revcomp, uniform_len=0, counters=None, pinned=False):
        """dcb_decombine_ascii: ASCII reads in host memory in (read i = buf[off[i] : off[i] + length[i]]; off None = contiguous
        reads of uniform_len), result records in host memory out; the reads are packed on the device."""
        buf, off, length, n = self._ascii_args(buf, off, length, uniform_len)
        res = self._pinned_results(n) if pinned else np.zeros(n, dtype=RESULT_DTYPE)
        if counters is None:
            counters = np.zeros(NCOUNTERS, dtype=np.uint64)
        _check(lib().dcb_decombine_ascii(self._h, buf.ctypes.data if len(buf) else None, off.ctypes.data if off is not None else None,
                                         length.ctypes.data if length is not None else None, n, int(uniform_len), int(bool(revcomp)),
                                         res.ctypes.data, counters.ctypes.data), "dcb_decombine_ascii")
        self._n = n
        return res, counters

    def pack_device(self, buf, off, length, revcomp, uniform_len=0) -> Packed:
        """dcb_pack_device: the device packer's output as a host Packed (tests compare it with pack_arrays)."""
        buf, off, length, n = self._ascii_args(buf, off, length, uniform_len)
        out = ctypes.POINTER(CPacked)()
        _check(lib().dcb_pack_device(self._h, buf.ctypes.data if len(buf) else None, off.ctypes.data if off is not None else None,
                                     length.ctypes.data if length is not None else None, n, int(uniform_len), int(bool(revcomp)),
                                     ctypes.byref(out)), "dcb_pack_device")
        return Packed(out)

    def pack_device_ms(self):
        ms = ctypes.c_double()
        _check(lib().dcb_pack_device_ms(self._h, ctypes.byref(ms)), "dcb_pack_device_ms")
        return ms.value

    def upload(self, packed: Packed):
        _check(lib().dcb_upload(self._h, packed.c), "dcb_upload")
        self._n = packed.n_reads

    def run_resident(self):
        _check(lib().dcb_run_resident(self._h), "dcb_run_resident")

    def download(self, counters=None, want_results=True):
        res = np.zeros(self._n, dtype=RESULT_DTYPE) if want_results else None
        if counters is None:
            counters = np.zeros(NCOUNTERS, dtype=np.uint64)
        _check(lib().dcb_download(self._h, res.ctypes.data if want_results else None, counters.ctypes.data), "dcb_download")
        return res, counters

    def timing_enable(self, on=True):
        _check(lib().dcb_timing_enable(self._h, int(on)), "dcb_timing_enable")

    def timing_reset(self):
        _check(lib().dcb_timing_reset(self._h), "dcb_timing_reset")

    def timing_get(self):
        ms = np.zeros(NTIMERS, dtype=np.float64)
        n = np.zeros(NTIMERS, dtype=np.uint64)
        _check(lib().dcb_timing_get(self._h, ms.ctypes.data, n.ctypes.data), "dcb_timing_get")
        return ms, n

    def last_deferred(self):
        n = ctypes.c_uint64()
        _check(lib().dcb_last_deferred(self._h, ctypes.byref(n)), "dcb_last_deferred")
        return n.value

    def last_general(self):
        n = ctypes.c_uint64()
        _check(lib().dcb_last_general(self._h, ctypes.byref(n)), "dcb_last_general")
        return n.value

    def halftag_kernel_name(self):
        return lib().dcb_halftag_kernel_name(self._h).decode()

    def exact_kernel_name(self):
        return lib().dcb_exact_kernel_name(self._h).decode()

    def close(self):
        if self._h:
            lib().dcb_ctx_destroy(self._h)
            self._h = None
        if getattr(self, "_pin_ptr", None):
            lib().dcb_pinned_free(self._pin_ptr)
            self._pin_ptr = None
            self._pin_cap = 0

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_synth = None


def synth_lib():
    """libdcbsynth.so: the synthetic read generator in a library of its own, so that a process which only generates reads
    (bench.py --impl reference) never maps libdcb.so."""
    global _synth
    if _synth is None:
        L = ctypes.CDLL(_build.build_synth())
        cpp = ctypes.POINTER(ctypes.c_char_p)
        L.dcb_synth_create.restype = ctypes.c_void_p
        L.dcb_synth_create.argtypes = [ctypes.POINTER(CSynthParams), ctypes.c_int, ctypes.POINTER(cpp), ctypes.POINTER(ctypes.c_int),
                                       ctypes.POINTER(cpp), ctypes.POINTER(ctypes.c_int)]
        L.dcb_synth_destroy.argtypes = [ctypes.c_void_p]
        L.dcb_synth_reads.argtypes = [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int]
        _synth = L
    return _synth


class Synth:
    """dcb_synth: deterministic synthetic read generator (SURVEY.md 8d)."""

    def __init__(self, gene_sets, seed, read_len, read2_len=0, sub_rate=0.0, n_rate=0.0, junk_rate=0.0, umi_pool=0,
                 sub_rate2=0.0):
        """gene_sets: list of (v_regions, j_regions); read i is drawn from set i % len(gene_sets)."""
        L = synth_lib()
        self.read_len, self.read2_len = int(read_len), int(read2_len)

        def prob(x):
            return min(0xFFFFFFFF, int(round(x * 4294967296.0)))

        prm = CSynthParams(int(seed), self.read_len, self.read2_len, prob(sub_rate), prob(n_rate), prob(junk_rate),
                           int(umi_pool), prob(sub_rate2), 0)
        n = len(gene_sets)
        cpp = ctypes.POINTER(ctypes.c_char_p)
        self._keep = [(_carr(v), _carr(j)) for v, j in gene_sets]
        varr = (cpp * n)(*[ctypes.cast(k[0], cpp) for k in self._keep])
        jarr = (cpp * n)(*[ctypes.cast(k[1], cpp) for k in self._keep])
        nv = (ctypes.c_int * n)(*[len(v) for v, _ in gene_sets])
        nj = (ctypes.c_int * n)(*[len(j) for _, j in gene_sets])
        self._h = L.dcb_synth_create(ctypes.byref(prm), n, varr, nv, jarr, nj)
        if not self._h:
            raise DcbError("dcb_synth_create failed")

    def reads(self, first, n, want_r2=False, n_threads=None):
        r1 = np.empty(n * self.read_len, dtype=np.uint8)
        r2 = np.empty(n * self.read2_len, dtype=np.uint8) if (want_r2 and self.read2_len) else None
        nt = n_threads or min(32, os.cpu_count() or 1)
        if synth_lib().dcb_synth_reads(self._h, int(first), int(n), r1.ctypes.data, r2.ctypes.data if r2 is not None else None, nt) != 0:
            raise DcbError("dcb_synth_reads failed")
        return r1, r2

    def __del__(self):
        try:
            if self._h:
                synth_lib().dcb_synth_destroy(self._h)
                self._h = None
        except Exception:
            pass


# ---------------------------------------------------------------------------------------------------------
# collapse distance primitives
# ---------------------------------------------------------------------------------------------------------
UMI_MAX_LEN = 19
_BASE_ALPHABET = "ACGTNSL"


def _alphabet(strings, limit=8):
    """Symbol codes for the characters that occur (at most 8): A C G T N S L in that order, then whatever else."""
    present = set("".join(strings))
    order = [c for c in _BASE_ALPHABET if c in present] + sorted(present - set(_BASE_ALPHABET))
    if len(order) > limit:
        raise DcbError("more than %d distinct symbols: %r" % (limit, "".join(order)))
    return {c: i for i, c in enumerate(order)}


def encode_umis(umis):
    """list[str] -> uint64 codes for dcb_umi_pairs (3 bits per symbol, length in the top 6 bits)."""
    codes = _alphabet(umis)
    out = np.zeros(len(umis), dtype=np.uint64)
    for i, u in enumerate(umis):
        if len(u) > UMI_MAX_LEN:
            raise DcbError("UMI %r is longer than %d symbols" % (u, UMI_MAX_LEN))
        v = len(u) << 58
        for k, ch in enumerate(u):
            v |= codes[ch] << (3 * k)
        out[i] = v
    return out


def encode_umis_fixed(umis):
    """encode_umis with the FIXED alphabet A C G T N S L = 0..6 (what dcb_barcodes emits): the same code for the same UMI on
    every rank of a multi-GPU run, whatever symbols a rank happens to hold."""
    table = {c: i for i, c in enumerate(_BASE_ALPHABET)}
    out = np.zeros(len(umis), dtype=np.uint64)
    for i, u in enumerate(umis):
        if len(u) > UMI_MAX_LEN:
            raise DcbError("UMI %r is longer than %d symbols" % (u, UMI_MAX_LEN))
        v = len(u) << 58
        for k, ch in enumerate(u):
            if ch not in table:
                raise DcbError("UMI %r holds a symbol outside %s" % (u, _BASE_ALPHABET))
            v |= table[ch] << (3 * k)
        out[i] = v
    return out


def encode_seqs(seqs):
    """list[str] -> (symbols uint8, off uint64, len uint32) for dcb_lev_leq: codes 0..7 when the batch has at most eight
    distinct characters (the usual case), else the characters themselves (Dist.lev_leq then calls dcb_lev_leq_bytes)."""
    present = set("".join(seqs))
    table = np.arange(256, dtype=np.uint8)
    if len(present) <= 8:
        for ch, v in _alphabet(seqs).items():
            table[ord(ch)] = v
    elif any(ord(ch) > 255 for ch in present):
        raise DcbError("sequence symbols outside latin-1")
    length = np.array([len(x) for x in seqs], dtype=np.uint32)
    off = np.zeros(len(seqs), dtype=np.uint64)
    if len(seqs) > 1:
        off[1:] = np.cumsum(length[:-1], dtype=np.uint64)
    raw = np.frombuffer("".join(seqs).encode("latin-1"), dtype=np.uint8)
    return table[raw], off, length


class Dist:
    """dcb_dist: the GPU distance primitives of collapse (UMI neighbour pairs, bounded Levenshtein verdicts)."""

    def __init__(self, device=0):
        L = lib()
        self._h = L.dcb_dist_create(int(device))
        if not self._h:
            raise DcbError("dcb_dist_create: " + L.dcb_last_error().decode())

    def umi_pairs(self, codes, max_edits, part=0, n_parts=1):
        """-> (row, col) int64 arrays: every pair row < col within max_edits, ascending (row, col).  n_parts > 1: this
        GPU's share of a search split over n_parts GPUs (the union of the shares is the whole list)."""
        codes = np.ascontiguousarray(codes, dtype=np.uint64)
        n = ctypes.c_uint64()
        _check(lib().dcb_umi_pairs_part(self._h, codes.ctypes.data, len(codes), int(max_edits), int(part), int(n_parts), None, 0,
                                        ctypes.byref(n)), "dcb_umi_pairs")
        keys = np.zeros(n.value, dtype=np.uint64)
        if n.value:
            _check(lib().dcb_umi_pairs(self._h, None, 0, 0, keys.ctypes.data, n.value, ctypes.byref(n)), "dcb_umi_pairs")
        return (keys >> np.uint64(32)).astype(np.int64), (keys & np.uint64(0xFFFFFFFF)).astype(np.int64)

    def lev_leq(self, symbols, off, length, a, b, frac):
        """-> bool array: levenshtein(seq a[t], seq b[t]) <= len(shorter) * frac."""
        a = np.ascontiguousarray(a, dtype=np.uint32)
        b = np.ascontiguousarray(b, dtype=np.uint32)
        symbols = np.ascontiguousarray(symbols, dtype=np.uint8)
        off = np.ascontiguousarray(off, dtype=np.uint64)
        length = np.ascontiguousarray(length, dtype=np.uint32)
        out = np.zeros(len(a), dtype=np.uint8)
        wide = len(symbols) and int(symbols.max()) > 7
        _check((lib().dcb_lev_leq_bytes if wide else lib().dcb_lev_leq)(self._h, symbols.ctypes.data, off.ctypes.data, length.ctypes.data, len(length),
                                 a.ctypes.data, b.ctypes.data, len(a), float(frac), out.ctypes.data), "dcb_lev_leq")
        return out.astype(bool)

    def barcodes(self, bcs, quals, oligo, allow_ns, min_q, max_below, avg_q):
        """dcb_barcodes over lists of barcode-region strings and their quality strings.
        -> (status uint8, n1len uint8, code uint64) arrays; status BC_HOST rows are for the reference's fuzzy spacer search."""
        n = len(bcs)
        if n == 0:
            return np.zeros(0, dtype=np.uint8), np.zeros(0, dtype=np.uint8), np.zeros(0, dtype=np.uint64)
        try:
            bbuf = np.frombuffer("".join(bcs).encode("ascii") + b"\0", dtype=np.uint8)
            qbuf = np.frombuffer("".join(quals).encode("ascii") + b"\0", dtype=np.uint8)
        except UnicodeEncodeError:                       # non-ASCII text: every row takes the host path
            return np.full(n, BC_HOST, dtype=np.uint8), np.zeros(n, dtype=np.uint8), np.zeros(n, dtype=np.uint64)
        bl = np.fromiter((len(x) for x in bcs), dtype=np.uint32, count=n)
        ql = np.fromiter((len(x) for x in quals), dtype=np.uint32, count=n)
        bo = np.zeros(n, dtype=np.uint64)
        qo = np.zeros(n, dtype=np.uint64)
        if n > 1:
            np.cumsum(bl[:-1], dtype=np.uint64, out=bo[1:])
            np.cumsum(ql[:-1], dtype=np.uint64, out=qo[1:])
        return self.barcodes_arrays(bbuf, bo, bl, qbuf, qo, ql, oligo, allow_ns, min_q, max_below, avg_q)

    def barcodes_arrays(self, bbuf, bo, bl, qbuf, qo, ql, oligo, allow_ns, min_q, max_below, avg_q):
        """dcb_barcodes over (offset, length) columns into two uint8 text buffers."""
        n = len(bo)
        status, n1, code = np.full(n, BC_HOST, dtype=np.uint8), np.zeros(n, dtype=np.uint8), np.zeros(n, dtype=np.uint64)
        if n == 0:
            return status, n1, code
        bo, qo = np.ascontiguousarray(bo, dtype=np.uint64), np.ascontiguousarray(qo, dtype=np.uint64)
        bl, ql = np.ascontiguousarray(bl, dtype=np.uint32), np.ascontiguousarray(ql, dtype=np.uint32)
        prm = CBcParams(int(oligo), int(bool(allow_ns)), int(min_q), int(max_below), float(avg_q))
        _check(lib().dcb_barcodes(self._h, bbuf.ctypes.data, bo.ctypes.data, bl.ctypes.data, qbuf.ctypes.data, qo.ctypes.data,
                                  ql.ctypes.data, n, ctypes.byref(prm), status.ctypes.data, n1.ctypes.data, code.ctypes.data), "dcb_barcodes")
        return status, n1, code

    def last_ms(self):
        ms = ctypes.c_double()
        _check(lib().dcb_dist_last_ms(self._h, ctypes.byref(ms)), "dcb_dist_last_ms")
        return ms.value

    def last_method(self):
        return lib().dcb_dist_last_method(self._h).decode()

    def close(self):
        if self._h:
            lib().dcb_dist_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
