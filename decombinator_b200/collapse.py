"""Drop-in for the reference's ``decombinator.collapse`` module with its distance arithmetic on the GPU.

Same entry points and contracts as /root/reference/src/decombinator/collapse.py:

* ``collapsinator(inputargs, data=None) -> list[list]`` (collapse.py:979): same argument dict, same ``.freq`` rows
  (``[v, j, vdel, jdel, insert, n_umis, av_cluster_size]``), same summary CSV / optional side files;
* ``read_in_data``, ``cluster_UMIs``, ``get_barcode_positions``, ``findFirstSpacer`` ... keep their names and
  signatures (they are what the reference's own tests call);
* ``counts``: the module-level Counter.

What runs on the GPU (``libdcb.so``, include/dcb.h) are the two native dependencies of this stage:

* ``pyrepseq.nn.symdel`` + ``triu`` + ``sum_duplicates`` (collapse.py:735-742)  ->  ``dcb_umi_pairs``
* ``polyleven.levenshtein`` inside ``are_seqs_equivalent`` (collapse.py:355-360)  ->  ``dcb_lev_leq``, in batches:
  ``make_clusters`` asks for all its verdicts at once; ``read_in_data`` -- whose grouping is order dependent, but
  only among rows with the SAME barcode -- runs one small state machine per barcode and collects the verdicts the
  machines are waiting for into one batch per round.

Everything whose result depends on Python's own ordering rules stays host Python and reproduces them on purpose
(SURVEY.md Appendix A.7): dict insertion order incl. the re-insertion when a group's proto-sequence changes,
``Counter.most_common`` ties, the scipy row-major pair order, networkx's BFS component order and the iteration
order of a CPython ``set`` of ints (``list(subgraph)``), and banker's rounding of the average cluster size.
There is no CPU implementation of the distances here: without libdcb.so and a GPU these functions raise.
"""
import ast
import collections as coll
import gzip
import itertools
import operator
import os
import re
import sys
import time
from statistics import median

import numpy as np
import regex

from . import __version__, _lib

counts = coll.Counter()
_dist = None
MAX_SEQ_LEN = 512        # dcb_lev_leq (include/dcb.h); the reference's default -ln is 130

# spacer sequences per ligation oligo (collapse.py:172-190), first spacer then (if any) second
_OLIGOS = {
    "m13": {"spcr1": "GTCGTGACTGGGAAAACCCTGG", "spcr2": "GTCGTGAT"},
    "i8": {"spcr1": "GTCGTGAT", "spcr2": "GTCGTGAT"},
    "i8_single": {"spcr1": "ATCACGAC"},
    "nebio": {"spcr1": "TACGGG"},
    "takara": {"spcr1": "GTACGGG"},
}


def _gpu():
    """The dcb_dist context of this process (one per GPU; LOCAL_RANK selects the device under torchrun)."""
    global _dist
    if _dist is None:
        _dist = _lib.Dist(device=int(os.environ.get("LOCAL_RANK", "0")))
    return _dist


# ---------------------------------------------------------------------------------------------------------
# small helpers with the reference's names
# ---------------------------------------------------------------------------------------------------------
def num_check(poss_int):
    """Feasibly an integer >= 0? (collapse.py:74-82)"""
    try:
        return int(poss_int) >= 0
    except ValueError:
        return False


def is_dna(poss_dna):
    """collapse.py:85-87"""
    return set(poss_dna.upper()) <= set("ACGTN")


def get_qual_scores(qualstring):
    """FASTQ quality characters -> Q scores (collapse.py:329-332)"""
    return [ord(ch) - 33 for ch in qualstring]


def get_err_prob(Q):
    return 10 ** (-Q / 10)


def check_dcr_file(infile, opener):
    """Sanity check of the first five lines of an .n12 file (collapse.py:90-169)."""
    if not os.path.isfile(infile):
        print("Cannot find file, please double-check path.")
        return False
    print(os.path.getsize(infile))
    if os.path.getsize(infile) == 0:
        raise ValueError("Input file appears to be empty; please double-check path.")
    fail = "Input Decombinator file sanity check fail: "
    with opener(infile, "rt") as handle:
        for i in range(5):
            try:
                line = next(handle)
            except StopIteration:
                raise StopIteration(f"Input Decombinator file sanity check warning: {i} line(s) in input file.")
            if "," not in line:
                print(fail + "seemingly not comma-delimited text file.")
                return False
            f = line.rstrip().split(", ")
            if len(f) != 10:
                print(fail + "file does not contain the correct number of comma-delimited fields (ten).")
                return False
            if not all(num_check(x) for x in f[0:4]):
                print(fail + "integer components of Decombinator classifier not feasible (i.e. not integers >= zero).")
                return False
            if not is_dna(f[4]):
                print(fail + "Decombinator insert sequence field contains non-DNA sequence.")
                return False
            if not (is_dna(f[6]) and is_dna(f[8])):
                print(fail + "inter-tag and/or barcode sequence contains non-DNA sequences.")
                return False
            if not (all(set(num_check(x) for x in get_qual_scores(f[7]))) and all(set(num_check(x) for x in get_qual_scores(f[9])))):
                print(fail + "inter-tag and/or barcode quality strings do not appear to contain valid scores.")
                return False
            if len(f[6]) != len(f[7]) or len(f[8]) != len(f[9]):
                print(fail + "inter-tag and/or barcode sequence and quality string pairs are not of the same length.")
                return False
    return True


def getOligo(oligo_name):
    """collapse.py:172-190"""
    key = oligo_name.lower()
    if key not in _OLIGOS:
        print("Error: Failed to recognise oligo name. Please choose from " + str(list(_OLIGOS.keys())))
        sys.exit()
    return dict(_OLIGOS[key])


def findSubs(subseq, seq):
    """Up to two substitutions (collapse.py:193-196)."""
    return regex.findall("(" + subseq + "){1s<=2}", seq)


def findSubsInsOrDels(subseq, seq):
    """Up to two edits of which at most one substitution (collapse.py:199-202)."""
    return regex.findall("(" + subseq + "){2i+2d+1s<=2}", seq)


def spacerSearch(subseq, seq):
    """Exact, else substitutions, else indels (collapse.py:205-213)."""
    for finder in (regex.findall, findSubs, findSubsInsOrDels):
        found = finder(subseq, seq)
        if found:
            return found
    return found


def findFirstSpacer(oligo, seq, oligo_start, oligo_end):
    """collapse.py:216-220"""
    return list(spacerSearch(oligo["spcr1"], seq[oligo_start:oligo_end]))


def findSecondSpacer(oligo, seq):
    """collapse.py:223-228"""
    return list(spacerSearch(oligo["spcr2"], seq[len(oligo["spcr1"]):]))


def getSpacerPositions(bcseq, spacers):
    """str.find with a running start offset (collapse.py:231-238)."""
    positions, start = [], 0
    for sp in spacers:
        positions.append(bcseq.find(sp, start))
        start += len(sp)
    return positions


def filterShortandLongBarcodes(b1len, b2end, bcseq, counts):
    """collapse.py:241-254"""
    if b1len <= 3:
        counts["getbarcode_fail_n1tooshort"] += 1
    elif b1len >= 9:
        counts["getbarcode_fail_n1toolong"] += 1
    elif b2end > len(bcseq):
        counts["getbarcode_fail_n2pastend"] += 1
    else:
        return True
    return False


def logExactOrRegexMatch(spacers, oligo, counts):
    """collapse.py:257-261"""
    counts["getbarcode_pass_exactmatch" if spacers == list(oligo.values()) else "getbarcode_pass_regexmatch"] += 1


def logFuzzyMatching(b1len, bclength, spacers, oligo, counts):
    """collapse.py:264-278"""
    fuzzy = spacers != list(oligo.values())
    if b1len == bclength and fuzzy:
        counts["getbarcode_pass_fuzzymatch_rightlen"] += 1
    elif b1len in (4, 5) and fuzzy:
        counts["getbarcode_pass_fuzzymatch_short"] += 1
    elif b1len >= 7 and fuzzy:
        counts["getbarcode_pass_fuzzymatch_long"] += 1
    elif b1len == bclength:
        counts["getbarcode_pass_other"] += 1


def set_barcode(fields, bc_locs, inputargs):
    """Barcode + quality string from the located N1/N2 (collapse.py:281-326); N1 != 6 nt is padded with ``S`` or cut
    to five bases + ``L`` (quality ``?``; on the long branch ``"?" * negative`` is empty, as in the reference)."""
    seq, qual = fields[8], fields[9]
    if inputargs["oligo"].lower() in ("nebio", "takara"):
        return seq[bc_locs[0]:bc_locs[1]], qual[bc_locs[0]:bc_locs[1]]
    a, b, c, d = bc_locs
    n1 = b - a
    if n1 == 6:
        return seq[a:b] + seq[c:d], qual[a:b] + qual[c:d]
    pad = 6 - n1
    if n1 < 6:
        counts["readdata_short_barcode"] += 1
        return seq[a:b] + "S" * pad + seq[c:d], qual[a:b] + "?" * pad + qual[c:d]
    counts["readdata_long_barcode"] += 1
    return seq[a:a + 5] + "L" + seq[c:d], qual[a:a + 5] + "?" * pad + qual[c:d]


def check_umi_quality(qualstring, parameters):
    """True when the barcode FAILS: too many bases below the minimum, or mean below threshold (collapse.py:340-352)."""
    q = get_qual_scores(qualstring)
    return sum(x < parameters[0] for x in q) > parameters[1] or sum(q) / len(q) < parameters[2]


def _verdicts(pairs, lev_threshold_fraction):
    """[(seq_a, seq_b), ...] -> list of bool through ONE dcb_lev_leq launch."""
    if not pairs:
        return []
    index = {}
    for a, b in pairs:
        for x in (a, b):
            if x not in index:
                index[x] = len(index)
    seqs = list(index)
    sym, off, ln = _lib.encode_seqs(seqs)
    ia = np.fromiter((index[a] for a, _ in pairs), dtype=np.uint32, count=len(pairs))
    ib = np.fromiter((index[b] for _, b in pairs), dtype=np.uint32, count=len(pairs))
    return _gpu().lev_leq(sym, off, ln, ia, ib, lev_threshold_fraction).tolist()


def are_seqs_equivalent(seq1, seq2, lev_threshold_fraction):
    """Levenshtein distance <= len(shorter) * fraction (collapse.py:355-360); one-pair batch on the GPU."""
    return _verdicts([(seq1, seq2)], lev_threshold_fraction)[0]


def are_barcodes_equivalent(bc1, bc2, threshold):
    """collapse.py:363-364"""
    row, _ = _gpu().umi_pairs(_lib.encode_umis([bc1, bc2]), threshold)
    return len(row) == 1 or bc1 == bc2


def get_barcode_positions(bcseq, inputargs, counts):
    """Start/stop of N1 (and N2) in the barcode region, located through the spacers (collapse.py:367-479)."""
    name = inputargs["oligo"].lower()
    if name not in _OLIGOS:
        raise ValueError("The flag for the -ol input must be one of M13, I8, I8_single, NEBIO, or TAKARA.")
    if "N" in bcseq and inputargs["allowNs"] == False:  # noqa: E712
        counts["getbarcode_fail_N"] += 1
        return None
    oligo = getOligo(name)
    if name == "nebio":
        lo, hi = 18, 28
    elif name == "takara":
        lo, hi = 0, 19
    else:
        lo, hi = 0, 10 + len(oligo["spcr1"])
    spacers = findFirstSpacer(oligo, bcseq, lo, hi)
    if len(spacers) != 1:
        counts["getbarcode_fail_nospacerfound"] += 1
        return None
    fixed = name in ("nebio", "takara")
    if not fixed and name != "i8_single":
        spacers += findSecondSpacer(oligo, bcseq)
        if len(spacers) != 2:
            counts["getbarcode_fail_not2spacersfound"] += 1
            return None
    where = getSpacerPositions(bcseq, spacers)
    if fixed:
        bclength = 17 if name == "nebio" else 12
        logExactOrRegexMatch(spacers, oligo, counts)
        logFuzzyMatching(bclength, bclength, spacers, oligo, counts)
        return [0, bclength]
    bclength = 6
    if name == "i8_single":
        b1start, b1end = 0, where[0]
        b2start = where[0] + len(spacers[0])
    else:
        b1start, b1end = where[0] + len(spacers[0]), where[1]
        b2start = where[1] + len(spacers[1])
    b2end = b2start + bclength
    if not filterShortandLongBarcodes(b1end - b1start, b2end, bcseq, counts):
        return None
    logExactOrRegexMatch(spacers, oligo, counts)
    logFuzzyMatching(b1end - b1start, bclength, spacers, oligo, counts)
    return [b1start, b1end, b2start, b2end]


# ---------------------------------------------------------------------------------------------------------
# reading in: order-dependent grouping by exact barcode
# ---------------------------------------------------------------------------------------------------------
class _BarcodeMachine:
    """The grouping rules of read_in_data (collapse.py:595-682) for the rows of ONE barcode, in input order.

    A barcode owns at most one group: rows whose sequence is equivalent to the group's proto-sequence join it (and
    may change the proto-sequence to the new most common sequence, which re-inserts the group at the END of the
    reference's dict -- tracked as ``tick``); the first non-equivalent row kills the group and blacklists the barcode."""

    __slots__ = ("barcode", "rows", "pos", "proto", "members", "seq_count", "seq_first", "tick", "dead", "dropped")

    def __init__(self, barcode):
        self.barcode = barcode
        self.rows = []          # (row index, seq, dcretc)
        self.pos = 0
        self.proto = None
        self.members = None
        self.seq_count = None   # seq -> copies in the group
        self.seq_first = None   # seq -> position of its first copy (most_common(1) ties go to the earliest)
        self.tick = -1
        self.dead = False
        self.dropped = 0        # rows counted as multi_tcr_barcode_reads

    def run(self, cache):
        """Advance until the rows are used up (-> None) or a verdict is missing (-> the (proto, seq) pair needed)."""
        rows = self.rows
        while self.pos < len(rows):
            idx, seq, dcretc = rows[self.pos]
            if self.dead:
                self.dropped += 1
            elif self.members is None:
                self.proto, self.members, self.tick = seq, [dcretc], idx
                self.seq_count, self.seq_first = {seq: 1}, {seq: 0}
            else:
                if seq == self.proto:
                    same = True
                else:
                    key = (self.proto, seq) if self.proto <= seq else (seq, self.proto)
                    same = cache.get(key)
                    if same is None:
                        return key
                if same:
                    self.members.append(dcretc)
                    if seq not in self.seq_count:
                        self.seq_count[seq] = 0
                        self.seq_first[seq] = len(self.members) - 1
                    self.seq_count[seq] += 1
                    best = self.proto
                    if seq != best:
                        cs, cb = self.seq_count[seq], self.seq_count[best]
                        if cs > cb or (cs == cb and self.seq_first[seq] < self.seq_first[best]):
                            self.proto, self.tick = seq, idx
                else:
                    self.dead = True
                    self.dropped += 1
                    self.members = None
            self.pos += 1
        return None


_BC_SYMBOLS = np.frombuffer(b"ACGTNSL?", dtype=np.uint8)


def _fuzzy_on_device(d):
    """DCB_BC_FUZZY=0: the device leaves rows whose spacers are not found exactly to the host's regex path (A/B runs).
    A context that is not a _lib.Dist (the CPU tests install the oracle's, which hands every row back) takes the
    exact-search signature."""
    return os.environ.get("DCB_BC_FUZZY", "1") != "0" and isinstance(d, _lib.Dist)


def _device_barcodes(rows, inputargs, qp):
    """dcb_barcodes_fuzzy over the barcode regions of all rows at once: -> (status, barcode strings) or None when this
    oligo / option has no device path.  Rows with odd symbols, a ragged quality string or an overlong region come back with
    status BC_HOST (with DCB_BC_FUZZY=0 also rows whose spacers are not found exactly)."""
    name = inputargs["oligo"].lower()
    if name not in _lib.OLIGOS_ON_DEVICE or inputargs["sampling_analysis"] or not rows or "allowNs" not in inputargs:
        return None      # (without the allowNs key the reference fails on the first barcode that holds an N: host path)
    d = _gpu()
    fuzzy = _fuzzy_on_device(d)
    out = d.barcodes([r[8] for r in rows], [r[9] for r in rows], _lib.OLIGOS_ON_DEVICE[name],
                     inputargs["allowNs"] != False, qp[0], qp[1], qp[2], *((True,) if fuzzy else ()))  # noqa: E712
    status, n1, code = out[:3]
    text = _decode_barcodes(code, _lib.BC_LENGTH[name])      # BC_LENGTH[name] characters per row, back to back
    _count_device_barcodes(status, n1, name, out[3] if fuzzy else None)
    return status, text


def _decode_barcodes(code, width):
    """dcb_barcodes codes of `width` symbols -> their barcode strings, back to back in one str."""
    sym = (code[:, None] >> (np.uint64(3) * np.arange(width, dtype=np.uint64))[None, :]) & np.uint64(7)
    return _BC_SYMBOLS[sym.astype(np.intp)].tobytes().decode("ascii")


def _count_device_barcodes(status, n1, name, match=None):
    """The reference's counters for the rows decided on the device (collapse.py:241-278, 388-422, 546-553).  match (None:
    all 0) says which placed rows took a fuzzy spacer text: getbarcode_pass_regexmatch instead of _exactmatch, and
    logFuzzyMatching's classes by N1 length.  The fixed-barcode designs (NEBIO, TAKARA) have no N1: the reference passes
    their barcode length for it, so every placed row counts as N1 of the right length, none as a short or long barcode."""
    st = np.bincount(status, minlength=256)
    for key, k in (("getbarcode_fail_N", st[_lib.BC_FAIL_N]), ("getbarcode_fail_nospacerfound", st[_lib.BC_FAIL_NOSPACER]),
                   ("getbarcode_fail_not2spacersfound", st[_lib.BC_FAIL_NOT2]), ("getbarcode_fail_n1tooshort", st[_lib.BC_FAIL_N1SHORT]),
                   ("getbarcode_fail_n1toolong", st[_lib.BC_FAIL_N1LONG]), ("getbarcode_fail_n2pastend", st[_lib.BC_FAIL_N2END]),
                   ("readdata_fail_no_bclocs", int(st[_lib.BC_FAIL_N:_lib.BC_FAIL_N2END + 1].sum())),
                   ("readdata_fail_low_barcode_quality", st[_lib.BC_FAIL_QUALITY])):
        if k:
            counts[key] += int(k)
    placed = (status == _lib.BC_OK) | (status == _lib.BC_FAIL_QUALITY)         # spacers found, N1 / N2 in range
    fuzzy = placed & (match != 0) if match is not None else np.zeros_like(placed)
    exact = placed & ~fuzzy
    if name in _lib.BC_FIXED:
        right, short, long_ = placed, np.zeros_like(placed), np.zeros_like(placed)
    else:
        right, short, long_ = placed & (n1 == 6), placed & (n1 < 6), placed & (n1 > 6)
    for key, k in (("getbarcode_pass_exactmatch", exact.sum()), ("getbarcode_pass_regexmatch", fuzzy.sum()),
                   ("getbarcode_pass_fuzzymatch_rightlen", (fuzzy & right).sum()), ("getbarcode_pass_fuzzymatch_short", (fuzzy & short).sum()),
                   ("getbarcode_pass_fuzzymatch_long", (fuzzy & long_).sum()), ("getbarcode_pass_other", (exact & right).sum()),
                   ("readdata_short_barcode", short.sum()), ("readdata_long_barcode", long_.sum())):
        if k:
            counts[key] += int(k)


class N12Columns:
    """The rows of an .n12 FILE kept columnar (the `collapse` command's input, collapse.py:523-530): the text as one uint8
    array plus the (offset, length) of the ten fields of every row (dcb_n12_index).  Same protocol as
    decombine.RowsColumns: the barcode regions go to the device as columns into the text, the three strings collapse
    files a row under come from dcb_n12_collapse_rows, Python rows are only made for the rows the kernel hands back."""

    def __init__(self, text, off, ln):
        self.text, self.off, self.len = text, off, ln

    @classmethod
    def from_file(cls, path, opener):
        """None when the file is not plain ten-field ", "-joined ASCII rows ending in a newline (the caller then reads
        it line by line as the reference does)."""
        with opener(path, "rb") as handle:
            raw = handle.read()
        text = np.frombuffer(raw, dtype=np.uint8)
        if len(text) == 0 or bool((text >= 128).any()):
            return None
        index = _lib.n12_index(text)
        return None if index is None else cls(text, index[0], index[1])

    def __len__(self):
        return int(len(self.off))

    def barcode_columns(self):
        return (self.text, self.off[:, 8], self.len[:, 8], self.text, self.off[:, 9], self.len[:, 9])

    def subset_rows(self, keep):
        t, off, ln = self.text, self.off, self.len
        out = []
        for i in np.nonzero(keep)[0].tolist():
            a, b = int(off[i, 0]), int(off[i, 9]) + int(ln[i, 9])
            out.append(t[a:b].tobytes().decode("ascii").split(", "))
        return out

    def collapse_lines(self, keep):
        got = _lib.n12_collapse_rows(self.text, self.off, self.len, keep)
        if got is None:                                  # a quote or a backslash in a field: str() decides how it is written
            rows = self.subset_rows(keep)
            dcrs = [str(r[:5]) for r in rows]
            return [r[6] for r in rows], dcrs, ["|".join((d, r[6], r[7], r[5])) for d, r in zip(dcrs, rows)]
        blob, n = got
        lines = blob.tobytes().decode("ascii").split("\n")
        return lines[0:3 * n:3], lines[1:3 * n:3], lines[2:3 * n:3]


def _filter_columns(data, inputargs, barcode_quality_parameters, first_index=0):
    """_filter_rows for the columnar hand-over of `pipeline` (decombine.RowsColumns): the barcode regions and their
    qualities go to the device as (offset, length) columns into the FASTQ text -- no Python string per row -- and rows
    are only materialised for the reads the barcode kernel lets through or hands back.  Same results, same counters.
    None when this run has no device path for the barcodes (the caller then takes the rows)."""
    name = inputargs["oligo"].lower()
    if name not in _lib.OLIGOS_ON_DEVICE or inputargs["sampling_analysis"] or "allowNs" not in inputargs or len(data) == 0:
        return None
    d = _gpu()
    fuzzy = _fuzzy_on_device(d)
    out = d.barcodes_arrays(*data.barcode_columns(), _lib.OLIGOS_ON_DEVICE[name], inputargs["allowNs"] != False,  # noqa: E712
                            *barcode_quality_parameters, *((True,) if fuzzy else ()))
    status, n1, code = out[:3]
    _count_device_barcodes(status, n1, name, out[3] if fuzzy else None)
    ok, host = status == _lib.BC_OK, status == _lib.BC_HOST
    # rows whose barcode the kernel assembled: no Python row at all, the three strings collapse files them under come from
    # dcb_format_collapse_rows; rows it hands back (odd symbols, ragged quality strings) become Python rows as before
    seqs, dcrs, etcs = data.collapse_lines(ok)
    width = _lib.BC_LENGTH[name]
    text = _decode_barcodes(code[ok], width)
    fast = (seqs, dcrs, etcs, re.findall("." * width, text), (first_index + np.nonzero(ok)[0]).tolist())
    rows = data.subset_rows(host) if bool(host.any()) else []
    return rows, (first_index + np.nonzero(host)[0]).tolist(), fast, int(len(status))


def _filter_rows(data, inputargs, barcode_quality_parameters, dont_count, from_file, first_index=0):
    """The per-row part of read_in_data (collapse.py:523-593): barcode location, quality and length filters.

    The barcode of every row is located, assembled and quality-checked by ONE kernel launch (dcb_barcodes_fuzzy: the exact
    spacer search and the reference's fuzzy ones); only the rows it hands back -- odd symbols, ragged quality strings,
    regions over 250 bases -- go through get_barcode_positions / set_barcode / check_umi_quality on the host.

    -> ([(global row index, barcode, seq, dcretc), ...] for the rows that survive, Counter of str(dcr), rows seen).
    Rows are independent here, so a multi-GPU run calls this on each rank's shard (parallel.py)."""
    t0 = time.time()
    columnar = _filter_columns(data, inputargs, barcode_quality_parameters, first_index) if hasattr(data, "subset_rows") else None
    index = fast = None
    if columnar is not None:
        rows, index, fast, n_rows = columnar
        status = text = None                           # the rows left are the ones the kernel handed back
    else:
        rows = [line.rstrip("\n").split(", ") for line in data] if from_file else (data if isinstance(data, list) else list(data))
        dev = _device_barcodes(rows, inputargs, barcode_quality_parameters)
        n_rows = len(rows)
        status = dev[0].tolist() if dev is not None else None
        text = dev[1] if dev is not None else None
    kept = []
    input_dcr_counts = coll.Counter()
    counts["readdata_input_dcrs"] += n_rows
    lenthreshold, sampling = inputargs["lenthreshold"], inputargs["sampling_analysis"]
    n_long = n_ok = 0
    HOST, OK = _lib.BC_HOST, _lib.BC_OK
    width = _lib.BC_LENGTH.get(inputargs["oligo"].lower(), 0)
    for lcount, line in enumerate(rows):
        if lcount % 50000 == 0 and lcount != 0 and not dont_count:
            print("   Read in", lcount, "lines... ", round(time.time() - t0, 2), "seconds")
        st = status[lcount] if status is not None else HOST
        if st == OK:
            barcode, barcode_qualstring = text[width * lcount:width * (lcount + 1)], None
        elif st != HOST:
            continue                                  # rejected on the device, counted in _device_barcodes
        else:
            bc_locs = get_barcode_positions(line[8], inputargs, counts)
            if not bc_locs:
                counts["readdata_fail_no_bclocs"] += 1
                continue
            barcode, barcode_qualstring = set_barcode(line, bc_locs, inputargs)
            if check_umi_quality(barcode_qualstring, barcode_quality_parameters):
                counts["readdata_fail_low_barcode_quality"] += 1
                continue
        dcr = str(line[:5])
        input_dcr_counts[dcr] += 1
        seq = line[6]
        if len(seq) > lenthreshold:
            n_long += 1
            continue
        n_ok += 1
        if sampling:
            dcretc = "|".join([dcr, seq, line[7], line[5], barcode, barcode_qualstring, line[8], line[10]])
        else:
            dcretc = "|".join((dcr, seq, line[7], line[5]))
        kept.append((index[lcount] if index is not None else first_index + lcount, barcode, seq, dcretc))
    if fast is not None and fast[0]:
        seqs, dcrs, etcs, barcodes, idx = fast
        input_dcr_counts.update(dcrs)
        short = (np.fromiter(map(len, seqs), dtype=np.int64, count=len(seqs)) <= lenthreshold).tolist()
        part = list(itertools.compress(zip(idx, barcodes, seqs, etcs), short))
        n_long += len(seqs) - len(part)
        n_ok += len(part)
        if kept:                                       # both lists are in input order: one merge
            kept = part + kept
            kept.sort(key=operator.itemgetter(0))
        else:
            kept = part
    if n_long:
        counts["readdata_fail_overlong_intertag_seq"] += n_long
    if n_ok:
        counts["readdata_success"] += n_ok
    return kept, input_dcr_counts, n_rows


_BC_CODE = np.full(256, 255, dtype=np.uint8)
_BC_CODE[np.frombuffer(b"ACGTNSL", dtype=np.uint8)] = np.arange(7, dtype=np.uint8)


def _group_rows(kept, lev_threshold_fraction):
    """Order-dependent grouping by exact barcode (collapse.py:595-682) of rows given in global input order.

    -> ([(tick, barcode, proto, members), ...] of the surviving groups, rows dropped, barcodes blacklisted).  Only rows with
    the SAME barcode interact, so any partition of the barcodes (parallel.py: hash(barcode) % world) can be grouped
    independently and merged by ``tick`` afterwards.

    The rules run in the library over columns (dcb_group, csrc/group.cpp) when the barcodes are all of one length (up to
    UMI_MAX_LEN symbols of ACGTNSL) and the sequences are plain ASCII -- the usual case; anything else through the same
    rules in Python (_BarcodeMachine).
    Either way each round resolves, in ONE GPU batch, every sequence verdict some barcode waits for."""
    native = _group_rows_native(kept, lev_threshold_fraction) if len(kept) >= 64 and os.environ.get("DCB_GROUP_NATIVE", "1") != "0" else None
    if native is not None:
        return native
    machines = {}
    for idx, barcode, seq, dcretc in kept:
        m = machines.get(barcode)
        if m is None:
            m = machines[barcode] = _BarcodeMachine(barcode)
        m.rows.append((idx, seq, dcretc))
    # each round resolves, in one GPU batch, every verdict some machine waits for
    cache, waiting = {}, list(machines.values())
    while waiting:
        need, blocked = {}, []
        for m in waiting:
            key = m.run(cache)
            if key is not None:
                need[key] = None
                blocked.append(m)
        if need:
            keys = list(need)
            for key, verdict in zip(keys, _verdicts(keys, lev_threshold_fraction)):
                cache[key] = verdict
        waiting = blocked
    ms = list(machines.values())
    return ([(m.tick, m.barcode, m.proto, m.members) for m in ms if m.members is not None], sum(m.dropped for m in ms),
            sum(1 for m in ms if m.dead))


def _group_rows_native(kept, lev_threshold_fraction):
    """_group_rows through dcb_group; None when the rows are not of the shape it takes."""
    n = len(kept)
    idx_l, bc_l, seq_l, etc_l = zip(*kept)
    try:
        bcs = "".join(bc_l).encode("ascii")
        seqs = "\n".join(seq_l).encode("ascii")
    except UnicodeEncodeError:
        return None
    width = len(bc_l[0])                                              # 12, or 17 for NEBIO
    # (a sequence that holds a newline: not the library's shape)
    if not 0 < width <= _lib.UMI_MAX_LEN or len(bcs) != width * n or seqs.count(b"\n") != n - 1:
        return None
    sym = _BC_CODE[np.frombuffer(bcs, dtype=np.uint8)].reshape(n, width)
    if int(sym.max()) > 6 or len(set(map(len, bc_l))) != 1:
        return None
    code = (sym.astype(np.uint64) << (np.uint64(3) * np.arange(width, dtype=np.uint64))[None, :]).sum(axis=1, dtype=np.uint64)
    g = _lib.Grouping(seqs, code, np.fromiter(idx_l, dtype=np.uint64, count=n))
    try:
        g.run(lambda symbols, off, ln, a, b: _gpu().lev_leq(symbols, off, ln, a, b, lev_threshold_fraction))
        _, tick, proto, first, rows, dropped, dead = g.result()
    finally:
        g.close()
    rows, first, tick = rows.tolist(), first.tolist(), tick.tolist()
    groups = []
    for k, p in enumerate(proto.tolist()):
        members = rows[first[k]:first[k + 1]]
        groups.append((tick[k], bc_l[members[0]], seq_l[p],
                       list(operator.itemgetter(*members)(etc_l)) if len(members) > 1 else [etc_l[members[0]]]))
    return groups, dropped, dead


def _groups_to_dict(groups, input_dcr_counts, dropped, dead):
    """[(tick, barcode, proto, members)] -> the reference's ``barcode_dcretc`` dict (in its insertion order) + counters."""
    barcode_dcretc = coll.defaultdict(list)
    for _, barcode, proto, members in sorted(groups, key=lambda g: g[0]):
        barcode_dcretc["|".join([barcode, "0", proto])] = members
    if dropped:
        counts["multi_tcr_barcode_reads"] += dropped
    counts["readdata_barcode_dcretc_keys"] = len(barcode_dcretc)
    counts["number_input_unique_dcrs"] = len(input_dcr_counts)
    counts["number_input_total_dcrs"] = sum(input_dcr_counts.values())
    counts["multi_tcr_barcodes"] = dead
    return barcode_dcretc


def read_in_data(data, inputargs, barcode_quality_parameters, lev_threshold_fraction, dont_count, opener):
    """Filter the decombined rows, extract their barcodes and sort them into initial groups (collapse.py:482-701).

    Returns ``{"barcode|0|protoseq": [dcretc, ...]}`` in the reference's dict order."""
    if inputargs["command"] == "collapse":
        if not inputargs["dontcheckinput"]:
            if not check_dcr_file(data, opener):
                print("Please check that file contains suitable Decombinator output for collapsing.")
                print("Alternatively, disable the input file sanity check by changing the 'dontcheckinput' flag, i.e. '-di True'")
                sys.exit()
        columns = None
        if inputargs["oligo"].lower() in _lib.OLIGOS_ON_DEVICE and not inputargs["sampling_analysis"] and "allowNs" in inputargs:
            columns = N12Columns.from_file(data, opener)
        data = columns if columns is not None and len(columns) else opener(data, "rt")
    if not data:
        raise ValueError("No reads found in input file. Check .n12 and log files for errors.")

    print("Reading data in...")
    t0 = time.time()
    from_file = inputargs["command"] == "collapse" and not isinstance(data, N12Columns)
    kept, input_dcr_counts, n_lines = _filter_rows(data, inputargs, barcode_quality_parameters, dont_count, from_file)
    if from_file:
        data.close()
    groups, dropped, dead = _group_rows(kept, lev_threshold_fraction)
    barcode_dcretc = _groups_to_dict(groups, input_dcr_counts, dropped, dead)
    t1 = time.time()
    print("   Read in total of", n_lines, "lines")
    print("  ", counts["readdata_success"], "reads sorted into", len(barcode_dcretc), "initial groups")
    print("  ", round(t1 - t0, 2), "seconds")
    counts["time_readdata_s"] = t1
    return barcode_dcretc


# ---------------------------------------------------------------------------------------------------------
# clustering
# ---------------------------------------------------------------------------------------------------------
def create_clustering_objs(barcode_dcretc):
    """collapse.py:704-720"""
    barcode_dcretc_list = list(barcode_dcretc.items())
    umi_protoseq_tuple = [(key.split("|")[0], key.split("|")[2]) for key, _ in barcode_dcretc_list]
    return len(barcode_dcretc), barcode_dcretc_list, umi_protoseq_tuple


class _PairList:
    """What make_merge_groups returns: the ``row`` / ``col`` arrays of the reference's upper-triangular COO matrix."""

    def __init__(self, row, col):
        self.row, self.col = row, col

    def getnnz(self):
        return len(self.row)


def make_merge_groups(umi_protoseq_tuple, barcode_threshold, dont_count):
    """All UMI pairs within ``barcode_threshold`` edits, row < col, row-major order (collapse.py:723-751)."""
    umi_list = [u for u, _ in umi_protoseq_tuple]
    if len(umi_list) == 0:
        raise ValueError("No UMIs to cluster, check .n12 file for errors")
    print("Clustering UMIs...")
    print("  ", len(umi_list), "unique UMIs")
    row, col = _gpu().umi_pairs(_lib.encode_umis(umi_list), barcode_threshold)
    matches = _PairList(row, col)
    print("  ", matches.getnnz(), "UMIs within edit distance of", barcode_threshold)
    return matches


def _components(edges):
    """Connected components the way networkx yields them for a graph built by add_edge in this order: start nodes in
    node-insertion order, members gathered breadth first into a SET in discovery order (so that ``list(component)``
    has CPython's set iteration order, which the reference relies on, collapse.py:787-798)."""
    adj = {}
    for i, j in edges:
        adj.setdefault(i, {})
        adj.setdefault(j, {})
        adj[i][j] = None
        adj[j][i] = None
    done = set()
    for start in adj:
        if start in done:
            continue
        seen = {start}
        level = [start]
        while level:
            nxt = []
            for v in level:
                for w in adj[v]:
                    if w not in seen:
                        seen.add(w)
                        nxt.append(w)
            level = nxt
        done.update(seen)
        yield seen
    return


def make_clusters(merge_groups, barcode_dcretc_list, lev_threshold_fraction):
    """Merge the groups whose UMIs are neighbours AND whose proto-sequences are equivalent (collapse.py:754-809)."""
    pairs = list(zip(merge_groups.row.tolist(), merge_groups.col.tolist()))
    proto = [key.split("|")[2] for key, _ in barcode_dcretc_list]
    verdicts = _verdicts([(proto[i], proto[j]) for i, j in pairs], lev_threshold_fraction)
    edges = [p for p, ok in zip(pairs, verdicts) if ok]
    print("    ", len(edges), "merged UMIs")
    clusters = coll.defaultdict(list)
    in_graph = set()
    for component in _components(edges):
        order = list(component)
        in_graph.update(order)
        base = barcode_dcretc_list[order[0]][0]
        for k in order:
            clusters[base] += barcode_dcretc_list[k][1]
    for i, (key, members) in enumerate(barcode_dcretc_list):
        if i not in in_graph:
            clusters[key] = members
    return clusters


def write_clusters(clusters, inputargs):
    """collapse.py:812-848"""
    filename = "clusters_" + inputargs["chain"]
    ftype = ".psv.gz"
    count = 1
    while os.path.isfile(filename + ftype):
        filename = filename + str(count)
        count += 1
    filename += ftype
    print("   Writing clusters to directory: ", os.path.abspath(filename), "...")
    header = ["umi_id", "dcr", "inter_tag", "inter_tag_qual", "read_id", "umi", "umi_qual", "full_oligo", "v_tail"]
    with gzip.open(filename, "wt") as fh:
        fh.write("|".join(header) + "\n")
        for cluster_id, dcretc_list in clusters.items():
            name = ":".join(cluster_id.split("|")[:2])
            for dcretc in dcretc_list:
                fh.write(name + "|" + dcretc + "\n")


def cluster_UMIs(barcode_dcretc, inputargs, barcode_threshold, lev_threshold_fraction, dont_count, find_pairs=None):
    """Merge groups with neighbouring barcodes and equivalent proto-sequences (collapse.py:851-894).
    find_pairs: how to search the UMI pairs (default make_merge_groups on this GPU; parallel.py splits it over the ranks)."""
    print("Clustering barcode groups...")
    num_initial_groups, barcode_dcretc_list, umi_protoseq_tuple = create_clustering_objs(barcode_dcretc)
    t0 = time.time()
    matches = (find_pairs or make_merge_groups)(umi_protoseq_tuple, barcode_threshold, dont_count)
    print("  ", "comparing TCR sequences of similar UMIs...")
    clusters = make_clusters(matches, barcode_dcretc_list, lev_threshold_fraction)
    print("  ", num_initial_groups, "groups merged into", len(clusters), "clusters")
    print("  ", round(time.time() - t0, 10), "seconds")
    if inputargs["writeclusters"]:
        write_clusters(clusters, inputargs)
    return clusters


def _parse_dcr(dcr):
    """ast.literal_eval of str([v, j, vdel, jdel, insert]) -- five plain strings -- without compiling an expression per
    DCR (a second of a million-read run); anything that does not look like that goes through literal_eval."""
    if dcr.startswith("['") and dcr.endswith("']") and '"' not in dcr and "\\" not in dcr:
        parts = dcr[2:-2].split("', '")
        if len(parts) == 5 and not any("'" in x for x in parts):
            return parts
    return ast.literal_eval(dcr)


def _count_clusters(barcode_dcretc, inputargs, barcode_distance_threshold, lev_threshold_fraction, dont_count, outpath, file_id,
                    find_pairs=None):
    """cluster -> count (collapse.py:919-976), from the initial groups on."""
    clusters = cluster_UMIs(barcode_dcretc, inputargs, barcode_distance_threshold, lev_threshold_fraction, dont_count, find_pairs)

    print("Collapsing clusters...")
    t0 = time.time()
    collapsed = coll.Counter()
    cluster_sizes = coll.defaultdict(list)
    for members in clusters.values():
        # most common DCR of the cluster; ties go to the first one met (Counter.most_common semantics)
        dcrs = [x.split("|", 1)[0] for x in members]
        protodcr = dcrs[0] if dcrs.count(dcrs[0]) == len(dcrs) else coll.Counter(dcrs).most_common(1)[0][0]
        collapsed[protodcr] += 1
        cluster_sizes[protodcr].append(len(members))
    counts["number_output_unique_dcrs"] = len(collapsed)
    counts["number_output_total_dcrs"] = sum(collapsed.values())
    counts["median_barcodes_per_tcr"] = float(median(collapsed.values()))
    print("  ", round(time.time() - t0, 2), "seconds")

    print("Writing to variable...")
    out_data = []
    average_cluster_size_counter = coll.Counter()
    for dcr, dcr_count in collapsed.items():
        av_clus_size = round(sum(cluster_sizes[dcr]) / dcr_count)   # Python's round: half to even
        average_cluster_size_counter[av_clus_size] += 1
        out_data.append(_parse_dcr(dcr) + [dcr_count, av_clus_size])

    if inputargs["barcodeduplication"] == True:  # noqa: E712
        outfile = outpath + file_id + "_barcode_duplication.txt"
        with open(outfile, "w") as fh:
            for bc, copies in clusters.items():
                print(",".join(["|".join(bc.split("|")[:2]), str(len(copies))]), file=fh)
        print("barcode duplication data saved to", outfile)
    counts["outfilenam"] = "Saved to variable"
    return out_data, collapsed, average_cluster_size_counter


def collapsinate(data, inputargs, barcode_quality_parameters, lev_threshold_fraction, barcode_distance_threshold, outpath,
                 file_id, dont_count, opener=None):
    """read in -> cluster -> count (collapse.py:897-976)."""
    barcode_dcretc = read_in_data(data, inputargs, barcode_quality_parameters, lev_threshold_fraction, dont_count, opener)
    return _count_clusters(barcode_dcretc, inputargs, barcode_distance_threshold, lev_threshold_fraction, dont_count, outpath,
                           file_id)


def _write_summary(inputargs, file_id, average_cluster_size_counter):
    """Collapsing summary CSV (+ optional UMI histogram), collapse.py:1040-1224."""
    chainnams = {"a": "alpha", "b": "beta", "g": "gamma", "d": "delta"}
    chain_name = chainnams[inputargs["chain"].lower()]
    logpath = inputargs["outpath"] + f"Logs{os.sep}"
    sample_name = file_id.split(os.sep)[-1]
    if not os.path.exists(logpath):
        os.makedirs(logpath)
    date = time.strftime("%Y_%m_%d")
    stem = logpath + date + "_" + "dcr_" + sample_name + f"_{chain_name}" + "_Collapsing_Summary"
    summaryname = stem + ".csv"
    if os.path.exists(summaryname):
        for i in range(2, 10000):
            summaryname = stem + str(i) + ".csv"
            if not os.path.exists(summaryname):
                break
    inout_name = "_".join(f"{file_id}".split("_")[:-1]) + f"_{chain_name}"
    out = ["Property,Value", "Version," + str(__version__), "Directory," + os.getcwd(), "InputFile," + inout_name,
           "OutputFile," + inout_name, "DateFinished," + date, "TimeFinished," + time.strftime("%H:%M:%S"),
           "TimeTaken(Seconds)," + str(round(counts["time_taken_total_s"], 2)), ""]
    for s in ["extension", "dontgzip", "allowNs", "dontcheckinput", "barcodeduplication", "minbcQ", "bcQbelowmin",
              "bcthreshold", "lenthreshold", "percentlevdist", "avgQthreshold", "positionalbarcodes", "oligo"]:
        out.append(s + "," + str(inputargs[s]))
    counts["pc_input_dcrs"] = counts["number_input_total_dcrs"] / counts["readdata_input_dcrs"]
    counts["pc_uniq_dcr_kept"] = counts["number_output_unique_dcrs"] / counts["number_input_unique_dcrs"]
    counts["pc_total_dcr_kept"] = counts["number_output_total_dcrs"] / counts["number_input_total_dcrs"]
    counts["avg_input_tcr_size"] = counts["number_input_total_dcrs"] / counts["number_input_unique_dcrs"]
    counts["avg_output_tcr_size"] = counts["number_output_total_dcrs"] / counts["number_output_unique_dcrs"]
    counts["avg_RNA_duplication"] = 1 / counts["pc_total_dcr_kept"]
    out.append("")
    for label, key, nd in (("InputUncollapsedDCRLines", "readdata_input_dcrs", None),
                           ("UniqueDCRsPassingFilters", "number_input_unique_dcrs", None),
                           ("TotalDCRsPassingFilters", "number_input_total_dcrs", None),
                           ("PercentDCRPassingFilters(withbarcode)", "pc_input_dcrs", 3),
                           ("UniqueDCRsPostCollapsing", "number_output_unique_dcrs", None),
                           ("TotalDCRsPostCollapsing", "number_output_total_dcrs", None),
                           ("PercentUniqueDCRsKept", "pc_uniq_dcr_kept", 3),
                           ("PercentTotalDCRsKept", "pc_total_dcr_kept", 3),
                           ("AverageInputTCRAbundance", "avg_input_tcr_size", 3),
                           ("AverageOutputTCRAbundance", "avg_output_tcr_size", 3),
                           ("AverageRNAduplication", "avg_RNA_duplication", 3)):
        out.append(label + "," + str(counts[key] if nd is None else round(counts[key], nd)))
    out.append("")
    for label, key in (("BarcodeFail_ContainedNs", "getbarcode_fail_N"),
                       ("BarcodeFail_SpacersNotFound", "readdata_fail_no_bclocs"),
                       ("BarcodeFail_LowQuality", "readdata_fail_low_barcode_quality"),
                       ("NumberMultiTCRBarcodes", "multi_tcr_barcodes"),
                       ("NumberMultiTCRBarcodeReads", "multi_tcr_barcode_reads"),
                       ("MedianUMIsPerTCR", "median_barcodes_per_tcr")):
        out.append(label + "," + str(counts[key]))
    with open(summaryname, "w") as fh:
        print("\n".join(out), file=fh)

    if inputargs["UMIhistogram"]:
        hfileprefix = "_".join(summaryname.split("_")[:-2] + ["UMIhistogram"])
        if os.path.exists(hfileprefix + ".csv"):
            i = 1
            while os.path.exists(hfileprefix + str(i) + ".csv"):
                i += 1
            hfileprefix += str(i)
        hfilename = hfileprefix + ".csv"
        with open(hfilename, "w") as hfile:
            for av, count in sorted(average_cluster_size_counter.items()):
                print(str(av) + "," + str(count), file=hfile)
        print("\nAverage UMI cluster size histogram data saved to", hfilename)



def collapsinator(inputargs: dict, data: list = None) -> list:
    """Function wrapper for Collapsinator (collapse.py:979-1226)."""
    global counts
    print("Running Collapsinator version", __version__)
    if inputargs["extension"] == "n12":
        inputargs["extension"] = "freq"
    opener = gzip.open if inputargs["infile"].endswith(".gz") else open
    counts = coll.Counter()
    counts["start_time"] = time.time()
    barcode_quality_parameters = [inputargs["minbcQ"], inputargs["bcQbelowmin"], inputargs["avgQthreshold"]]
    lev_threshold_fraction = inputargs["percentlevdist"] / 100
    barcode_distance_threshold = inputargs["bcthreshold"]
    if inputargs["lenthreshold"] > MAX_SEQ_LEN:      # said before any work is done, not in the middle of the grouping
        raise ValueError("-ln %d: the sequence comparisons of this build take inter-tag sequences of up to %d bases"
                         % (inputargs["lenthreshold"], MAX_SEQ_LEN))
    if inputargs["command"] == "collapse":
        data = inputargs["infile"]
    file_id = inputargs["infile"].split("/")[-1].split(".")[0]
    dont_count = inputargs["dontcount"]

    out_data, collapsed, average_cluster_size_counter = collapsinate(
        data, inputargs, barcode_quality_parameters, lev_threshold_fraction, barcode_distance_threshold, "", file_id,
        dont_count, opener)

    counts["end_time"] = time.time()
    counts["time_taken_total_s"] = counts["end_time"] - counts["start_time"]

    if inputargs["suppresssummary"] == False:  # noqa: E712
        _write_summary(inputargs, file_id, average_cluster_size_counter)
    return out_data
