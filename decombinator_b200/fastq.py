"""FASTQ reading for the decombine path (reference decombine.py:118-179, 228-265).

``readfq`` keeps the exact record semantics of the reference's parser (Heng Li's readfq as shipped there:
the name is the header up to the first space, sequence and quality may span lines, and the last character
of every line is dropped unconditionally).  ``load_pairs`` materialises the records the main loop needs
(decombine.py:950-989) as flat byte buffers that go straight to ``dcb_pack_reads``.
"""
import gzip
import os
import struct
import zlib
import itertools
import mmap

import numpy as np


def opener_check(inputargs):
    """gzip.open for ``.gz`` inputs, else open (decombine.py:118-123)."""
    return gzip.open if inputargs["infile"].endswith(".gz") else open


def fastq_sanity(path, opener):
    """The three checks of fastq_check (decombine.py:126-179) on the first record.

    Returns False when the file holds fewer than four lines (the caller writes the stub summary and raises,
    as the reference does); raises ValueError for a malformed first record."""
    with opener(path, "rt") as fh:
        if sum(1 for _ in itertools.islice(fh, 4)) < 4:
            return False
        # the reference keeps reading from the same handle, i.e. it inspects lines 5-8
        rec = list(itertools.islice(fh, 0, 4))
    if rec[0][0] != "@":
        raise ValueError(f"Expected @ symbol at beginning of file for valid FASTQ. Found {rec[0][0]}.")
    if rec[2][0] != "+":
        raise ValueError(f"Expected + symbol at beginning of third line for valid FASTQ. Found {rec[2][0]}.")
    if len(rec[1]) != len(rec[3]):
        raise ValueError(
            f"Length of read to match length of read quality. Found read length = {len(rec[1])} and read quality length = {len(rec[3])}"
        )
    return True


def readfq(fp):
    """Generator of (name, seq, qual) with the reference parser's behaviour (decombine.py:228-265)."""
    pending = None
    while True:
        if not pending:
            for line in fp:
                if line[0] in ">@":
                    pending = line[:-1]
                    break
        if not pending:
            return
        name = pending[1:].partition(" ")[0]
        pending = None
        chunks = []
        for line in fp:
            if line[0] in "@+>":
                pending = line[:-1]
                break
            chunks.append(line[:-1])
        if not pending or pending[0] != "+":
            yield name, "".join(chunks), None
            if not pending:
                return
            continue
        seq = "".join(chunks)
        got, quals = 0, []
        complete = False
        for line in fp:
            quals.append(line[:-1])
            got += len(line) - 1
            if got >= len(seq):
                complete = True
                break
        if complete:
            pending = None
            yield name, seq, "".join(quals)
        else:
            yield name, seq, None
            return


class TextColumn:
    """One string per record, kept as (offset, length) into the raw FASTQ bytes and decoded on demand.

    Behaves like the list of str the general parser builds (len, integer index, slice, iteration); the rows of the
    result only ever need the strings of the reads that decombined."""

    __slots__ = ("buf", "off", "len")

    def __init__(self, buf, off, length):
        self.buf, self.off, self.len = buf, off, length

    def __len__(self):
        return len(self.off)

    def __getitem__(self, i):
        if isinstance(i, slice):
            return TextColumn(self.buf, self.off[i], self.len[i])
        o = int(self.off[i])
        return self.buf[o:o + int(self.len[i])].decode("ascii")

    def __iter__(self):
        buf = self.buf
        for o, n in zip(self.off.tolist(), self.len.tolist()):
            yield buf[o:o + n].decode("ascii")

    def count_containing(self, symbol):
        from . import _lib
        return _lib.count_ranges_with(self.buf, self.off, self.len, symbol)


def count_containing(column, symbol):
    """Records of a column (list of str or TextColumn) that contain `symbol`."""
    if isinstance(column, TextColumn):
        return column.count_containing(symbol)
    return sum(1 for s in column if symbol in s)


class ReadBatch:
    """Records of one decombine run: V(D)J reads as one byte buffer + per-record Python strings for the rows."""

    __slots__ = ("ids", "vdj", "vdjqual", "bc", "bcq", "v_tail", "buf", "off", "len")

    def __init__(self):
        self.ids, self.vdj, self.vdjqual, self.bc, self.bcq, self.v_tail = [], [], [], [], [], []
        self.buf = self.off = self.len = None

    def finalize(self):
        if isinstance(self.vdj, TextColumn):     # native index: the reads are packed straight from the file's bytes
            self.buf = np.frombuffer(self.vdj.buf, dtype=np.uint8)
            self.off = np.ascontiguousarray(self.vdj.off, dtype=np.uint64)
            self.len = np.ascontiguousarray(self.vdj.len, dtype=np.uint32)
            return self
        enc = [s.encode("latin-1", "replace") for s in self.vdj]
        self.len = np.fromiter((len(b) for b in enc), dtype=np.uint32, count=len(enc))
        self.off = np.zeros(len(enc), dtype=np.uint64)
        if len(enc) > 1:
            np.cumsum(self.len[:-1], dtype=np.uint64, out=self.off[1:])
        self.buf = np.frombuffer(b"".join(enc) + b"\0", dtype=np.uint8)
        return self

    def __len__(self):
        return len(self.vdj)

    def shard(self, lo, hi):
        """The records [lo, hi) as a batch of their own (multi-GPU runs: one contiguous shard per rank)."""
        part = ReadBatch()
        for name in ("ids", "vdj", "vdjqual", "bc", "bcq", "v_tail"):
            setattr(part, name, getattr(self, name)[lo:hi])
        return part.finalize()


def _clip(off, length, start, stop=None):
    """(offset, length) of s[start:stop] for every record s = (off, length); start, stop >= 0."""
    if start == 0 and stop is not None:          # a prefix (the barcode and its quality): one pass
        return off, np.minimum(length, np.uint32(stop)).astype(np.uint32, copy=False)
    n = length.astype(np.int64)
    a = np.minimum(n, start)
    b = n if stop is None else np.minimum(n, stop)
    return off + a.astype(np.uint64), np.maximum(b - a, 0).astype(np.uint32)


def _file_bytes(path, opener):
    """The file's text as a bytes-like object: a read-only memory map for plain files (no copy out of the page cache),
    the decompressed bytes for .gz."""
    if opener is open:
        try:
            with open(path, "rb") as fh:
                return mmap.mmap(fh.fileno(), 0, access=mmap.ACCESS_READ)
        except (ValueError, OSError):      # empty file, or a file system without mmap
            pass
    if opener is gzip.open:
        try:
            return gunzip_file(path)
        except Exception:                  # a damaged file: the gzip module then raises what the reference's reader raises
            pass
    with opener(path, "rb") as fh:
        return fh.read()


def _bgzf_blocks(raw):
    """[(first byte of the deflate data, one past its end, uncompressed size), ...] when the file is a chain of BGZF blocks
    (gzip members whose extra field 'BC' holds the member's size: bgzip, Illumina's converters), else None."""
    blocks, p, n = [], 0, len(raw)
    while p < n:
        if n - p < 18 or raw[p:p + 4] != b"\x1f\x8b\x08\x04":       # FLG = FEXTRA alone, as BGZF writes it
            return None
        xlen = struct.unpack_from("<H", raw, p + 10)[0]
        q, end, bsize = p + 12, p + 12 + xlen, None
        while q + 4 <= end:
            si1, si2, slen = raw[q], raw[q + 1], struct.unpack_from("<H", raw, q + 2)[0]
            if si1 == 66 and si2 == 67 and slen == 2:
                bsize = struct.unpack_from("<H", raw, q + 4)[0] + 1
            q += 4 + slen
        if bsize is None or p + bsize > n or bsize < 12 + xlen + 8:
            return None
        isize = struct.unpack_from("<I", raw, p + bsize - 4)[0]
        if isize:
            blocks.append((p + 12 + xlen, p + bsize - 8, isize))
        p += bsize
    return blocks or None


# BGZF files are inflated by the host threads: on the B200 box they beat one GPU decoder per 64 KB member (DESIGN §6).
BGZF_ON_DEVICE = False
# A single stream goes to the GPU unless its text is more than this many times the file's size (ISIZE of the last member
# over the file size).  One decoder thread per chunk writes its text serially, and highly compressible files have few
# chunks for a lot of text: on the B200 box the device inflated FASTQ of 6.5:1 at 2.8x the host's rate, and was slower
# than the host on synthetic FASTQ of 15:1 and 9:1 (constant quality strings) (DESIGN §6).
DEVICE_MAX_RATIO = 8


def _device_gunzip(raw, blocks):
    """The file inflated on the GPU (LOCAL_RANK selects it), or None: no usable device, a BGZF file (see BGZF_ON_DEVICE), or
    any failure of the device path -- a damaged file then reaches the host path, which raises what it raises today."""
    if blocks and not BGZF_ON_DEVICE:
        return None
    if not blocks and len(raw) >= 18 and int.from_bytes(raw[-4:], "little") > DEVICE_MAX_RATIO * len(raw):
        return None
    from . import _lib
    try:
        return _lib.gpu_inflate(raw, device=int(os.environ.get("LOCAL_RANK", "0")), members=blocks)
    except _lib.DcbError:
        return None


def gunzip_file(path, n_threads=None):
    """The decompressed bytes of a .gz file in an anonymous memory map (the same kind of object a plain file is read
    through).  A single stream or a chain of members is inflated on the GPU when one is usable (dcb_inflate_*, csrc/inflate.cu).
    Otherwise, and whenever the device path reports anything but success: a BGZF file is inflated block by block on all host
    threads (dcb_bgzf_inflate); any other gzip file -- one member or several -- is one deflate stream after the other,
    inflated in slices straight into the map."""
    with open(path, "rb") as fh:
        try:
            raw = mmap.mmap(fh.fileno(), 0, access=mmap.ACCESS_READ)
        except (ValueError, OSError):
            raw = fh.read()
    if len(raw) == 0:
        return b""
    blocks = _bgzf_blocks(raw)
    out = _device_gunzip(raw, blocks)
    if out is not None:
        return out
    if blocks:
        from . import _lib
        arr = np.array(blocks, dtype=np.uint64)
        out_off = np.zeros(len(blocks), dtype=np.uint64)
        np.cumsum(arr[:-1, 2], out=out_off[1:])
        total = int(arr[:, 2].sum())
        out = mmap.mmap(-1, total, flags=mmap.MAP_PRIVATE | mmap.MAP_ANONYMOUS)
        _lib.bgzf_inflate(np.frombuffer(raw, dtype=np.uint8), arr[:, 0], arr[:, 1], arr[:, 2], out_off, np.frombuffer(out, dtype=np.uint8),
                          n_threads)
        return out
    cap = max(1 << 20, 4 * len(raw))
    out = mmap.mmap(-1, cap, flags=mmap.MAP_PRIVATE | mmap.MAP_ANONYMOUS)      # (a shared anonymous map cannot grow)
    pos, at, step = 0, 0, 1 << 24
    d = zlib.decompressobj(31)
    pending = b""
    while True:
        if not pending:
            if at >= len(raw):
                break
            pending = raw[at:at + step]
            at += len(pending)
        chunk = d.decompress(pending, step)
        pending = d.unconsumed_tail
        if pos + len(chunk) > cap:
            cap = max(cap * 2, pos + len(chunk))
            out.resize(cap)
        out[pos:pos + len(chunk)] = chunk
        pos += len(chunk)
        if d.eof:                          # the end of a member: another one may follow (gzip files concatenate)
            rest = d.unused_data + pending
            while rest[:1] == b"\0":       # zero padding behind the last member, as the gzip module tolerates
                rest = rest[1:]
            pending = rest
            if not pending and at >= len(raw):
                break
            d = zlib.decompressobj(31)
    if not d.eof:
        raise EOFError("Compressed file ended before the end-of-stream marker was reached")
    if pos == 0:
        return b""
    out.resize(pos)
    return out


def load_pairs_native(inputargs, opener):
    """load_pairs through the native record index (dcb_fastq_index_build); None when a file is not in the strict
    four-line layout (the general parser then reproduces the reference's handling of everything else)."""
    from . import _lib
    bclength = inputargs["bclength"]
    if not isinstance(bclength, int) or bclength < 0 or inputargs["bc_read"] not in ("R1", "R2"):
        return None
    sampling = inputargs.get("sampling_analysis")
    batch = ReadBatch()
    if inputargs["bc_read"] == "R2":
        # both files are read (for .gz: decompressed -- zlib releases the GIL, and that is most of the wall time of a run on
        # compressed input) and indexed side by side: the line-start and record passes of one overlap the text scan of the other
        import threading
        box = {}

        def second():
            try:
                box["data2"] = _file_bytes(inputargs["infile"].replace("1.f", "2.f"), opener)
                box["ix2"] = _lib.fastq_index(box["data2"])
            except BaseException as e:      # raised again in the calling thread
                box["error"] = e
        th = threading.Thread(target=second)
        th.start()
        try:
            data1 = _file_bytes(inputargs["infile"], opener)
            ix1 = _lib.fastq_index(data1)
        finally:
            th.join()
        if "error" in box:
            raise box["error"]
        data2, ix2 = box["data2"], box.get("ix2")
        if ix1 is None or ix2 is None:
            return None
        n = min(len(ix1["seq_off"]), len(ix2["seq_off"]))            # zip() stops at the shorter file
        one = {k: v[:n] for k, v in ix1.items()}
        two = {k: v[:n] for k, v in ix2.items()}
        batch.ids = TextColumn(data1, one["name_off"], one["name_len"])
        batch.vdj = TextColumn(data1, one["seq_off"], one["seq_len"])
        batch.vdjqual = TextColumn(data1, one["qual_off"], one["qual_len"])
        batch.bc = TextColumn(data2, *_clip(two["seq_off"], two["seq_len"], 0, bclength))
        batch.bcq = TextColumn(data2, *_clip(two["qual_off"], two["qual_len"], 0, bclength))
        batch.v_tail = TextColumn(data2, *_clip(two["seq_off"], two["seq_len"], bclength, bclength + 31)) if sampling else []
    else:
        data1 = _file_bytes(inputargs["infile"], opener)
        ix1 = _lib.fastq_index(data1)
        if ix1 is None:
            return None
        # the reference zips the generator with itself: records 2k and 2k+1 are consumed together, the second only
        # feeds the sampling column
        n = len(ix1["seq_off"]) // 2
        one = {k: v[0:2 * n:2] for k, v in ix1.items()}
        two = {k: v[1:2 * n:2] for k, v in ix1.items()}
        batch.ids = TextColumn(data1, one["name_off"], one["name_len"])
        batch.vdj = TextColumn(data1, *_clip(one["seq_off"], one["seq_len"], bclength))
        batch.vdjqual = TextColumn(data1, *_clip(one["qual_off"], one["qual_len"], bclength))
        batch.bc = TextColumn(data1, *_clip(one["seq_off"], one["seq_len"], 0, bclength))
        batch.bcq = TextColumn(data1, *_clip(one["qual_off"], one["qual_len"], 0, bclength))
        batch.v_tail = TextColumn(data1, *_clip(two["seq_off"], two["seq_len"], bclength, bclength + 31)) if sampling else []
    return batch.finalize()


def load_pairs(inputargs, opener) -> ReadBatch:
    """The record handling at the top of the hot loop (decombine.py:950-983)."""
    if not inputargs.get("python_fastq"):
        native = load_pairs_native(inputargs, opener)
        if native is not None:
            return native
    bclength = inputargs["bclength"]
    batch = ReadBatch()
    fq1 = readfq(opener(inputargs["infile"], "rt"))
    if inputargs["bc_read"] == "R2":
        fq2 = readfq(opener(inputargs["infile"].replace("1.f", "2.f"), "rt"))
    elif inputargs["bc_read"] == "R1":
        fq2 = fq1  # the reference zips the generator with itself: two records are consumed per iteration
    else:
        raise UnboundLocalError("bc_read must be R1 or R2")  # the reference fails on the unbound fq1/fq2
    sampling = inputargs.get("sampling_analysis")
    for record1, record2 in zip(fq1, fq2):
        if inputargs["bc_read"] == "R2":
            batch.ids.append(record1[0])
            batch.vdj.append(record1[1])
            batch.vdjqual.append(record1[2])
            batch.bc.append(record2[1][:bclength])
            batch.bcq.append(record2[2][:bclength])
        else:
            batch.ids.append(record1[0])
            batch.vdj.append(record1[1][bclength:])
            batch.vdjqual.append(record1[2][bclength:])
            batch.bc.append(record1[1][0:bclength])
            batch.bcq.append(record1[2][0:bclength])
        if sampling:
            batch.v_tail.append(record2[1][bclength:bclength + 31])
    return batch.finalize()
