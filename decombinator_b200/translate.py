"""Drop-in for the reference's ``decombinator.translate`` module (CDR3translator): decombined / collapsed DCRs ->
AIRR-seq community ``.tsv`` rows.

Same entry points and contracts as /root/reference/src/decombinator/translate.py:

* ``cdr3translator(inputargs, data=None) -> pandas.DataFrame`` (translate.py:388-621): the 24 AIRR columns of
  ``out_headers``, one row per input DCR (non-productive ones too unless ``-npf``), the
  ``Logs/..._CDR3_Translation_Summary.csv`` file, the same exits for a bad chain / species;
* ``import_gene_information(inputargs)`` (translate.py:123-254) and ``get_cdr3(dcr, headers, inputargs)``
  (translate.py:257-357).

The work per row is rebuilding the nucleotide sequence from the germline regions, translating it, and four string
checks.  When a CUDA device is usable, ``dcb_translate`` (csrc/translate.cu) does that for every row and writes the
``.tsv`` lines itself; ``translate_tsv`` hands that text on without building a DataFrame (the command line writes it
as it is).  The host code below -- ``get_cdr3`` and the loop of ``_translate_host`` -- is the path without a device,
the path of a call with a row outside the kernels' envelope (``_lib.TR_*``: the host raises on it, or to_csv would
quote it), and the reference the tests compare the kernels with.  What is different from the reference is the
structure (one ``GeneTables`` object instead of a dozen module globals, the translation of every (V gene, deletion)
prefix cached because repertoires reuse them heavily) and that the translation itself is implemented here
(Bio.Seq.translate's standard-table semantics) instead of importing Biopython, which GPU nodes do not carry.  Quirks
kept on purpose, because the goldens depend on them or a user may:

* gene names are the second ``|`` field of the FASTA header, upper-cased, cut at ``*`` (translate.py:189-192, 293-294);
* "functionality" is column 3 of the ``.translate`` file (translate.py:217-219) -- the gene name, not the F/ORF/P
  flag of column 5, so the FunctionalityOfGermlineGenesUsed block of the summary counts only genes literally named
  ``F``/``ORF``/``P`` (i.e. it prints zeros);
* the conserved-cysteine test indexes the protein with ``position - 1`` under Python's rules (position 0 looks at the
  LAST residue; a position beyond the protein raises IndexError exactly as the reference does);
* the in-frame test is ``(len(sequence) - 1) % 3 == 0`` (translate.py:310).
"""
import collections as coll
import gzip
import os
import re
import sys
from time import strftime

import numpy as np

from . import __version__, _lib, tags

chainnams = tags.CHAINNAMS
counts = coll.Counter()
chain = None
_genes = None      # GeneTables of the last import_gene_information()
_dist = None       # dcb_dist of this process; False when no device is usable

out_headers = [
    "sequence_id", "v_call", "d_call", "j_call", "junction_aa", "duplicate_count", "sequence", "junction",
    "decombinator_id", "rev_comp", "productive", "sequence_aa", "cdr1_aa", "cdr2_aa", "vj_in_frame", "stop_codon",
    "conserved_c", "conserved_f", "sequence_alignment", "germline_alignment", "v_cigar", "d_cigar", "j_cigar",
    "av_UMI_cluster_size",
]

# ---------------------------------------------------------------------------------------------------------
# Translation: Bio.Seq.translate(table="Standard") semantics (what translate.py:304-306 calls): upper-cased input, the
# trailing partial codon dropped, '*' for stop codons; a codon with IUPAC ambiguity codes becomes the amino acid all of
# its expansions share, B / Z / J for {D,N} / {E,Q} / {I,L}, else X (also when only some expansions are stops).
# ---------------------------------------------------------------------------------------------------------
_BASES = "TCAG"
_AMINO = "FFLLSSSSYY**CC*WLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG"
_CODON = {a + b + c: _AMINO[16 * i + 4 * j + k] for i, a in enumerate(_BASES) for j, b in enumerate(_BASES)
          for k, c in enumerate(_BASES)}
_IUPAC = {"A": "A", "C": "C", "G": "G", "T": "T", "U": "T", "R": "AG", "Y": "CT", "S": "CG", "W": "AT", "K": "GT", "M": "AC",
          "B": "CGT", "D": "AGT", "H": "ACT", "V": "ACG", "N": "ACGT"}
_ambiguous_cache = {}


def _ambiguous_codon(codon):
    hit = _ambiguous_cache.get(codon)
    if hit is not None:
        return hit
    try:
        options = [_IUPAC[c] for c in codon]
    except KeyError:
        raise ValueError("Codon '%s' is invalid" % codon) from None      # Bio raises TranslationError here
    aas = {_CODON[a + b + c] for a in options[0] for b in options[1] for c in options[2]}
    if len(aas) == 1:
        aa = next(iter(aas))
    elif "*" in aas:
        aa = "X"
    elif aas <= {"D", "N"}:
        aa = "B"
    elif aas <= {"E", "Q"}:
        aa = "Z"
    elif aas <= {"I", "L"}:
        aa = "J"
    else:
        aa = "X"
    _ambiguous_cache[codon] = aa
    return aa


def translate_nt(seq):
    """str(Bio.Seq.Seq(seq).translate()) for the standard table."""
    s = seq.upper()
    get = _CODON.get
    out = []
    for i in range(0, len(s) - len(s) % 3, 3):
        codon = s[i:i + 3]
        out.append(get(codon) or _ambiguous_codon(codon))
    return "".join(out)


# ---------------------------------------------------------------------------------------------------------
# Gene tables
# ---------------------------------------------------------------------------------------------------------
def _fasta_records(text):
    """(id up to the first whitespace, upper-cased sequence) per record, as SeqIO.parse(..., "fasta") yields them."""
    recs, head, parts = [], None, []
    for raw in text.splitlines():
        if raw[:1] == ">":
            if head is not None:
                recs.append((head, "".join(parts).upper()))
            fields = raw[1:].split()
            head, parts = (fields[0] if fields else ""), []
        elif head is not None:
            parts.append(raw.strip())
    if head is not None:
        recs.append((head, "".join(parts).upper()))
    return recs


class GeneTables:
    """What import_gene_information() returns, for one chain (translate.py:123-254)."""

    def __init__(self, inputargs):
        species, tagset, tagdir, ch = inputargs["species"], inputargs["tags"], inputargs.get("tagfastadir"), inputargs["chain"]
        for gene in ("v", "j"):
            recs = _fasta_records(tags.read_tcr_text(species, tagset, ch, gene, "fasta", tagdir))
            setattr(self, gene + "_regions", [seq for _, seq in recs])
            setattr(self, gene + "_names", [head.upper().split("|")[1] for head, _ in recs])
            rows = [x.rstrip().split(",") for x in tags.read_tcr_text(species, tagset, ch, gene, "translate", tagdir).splitlines(True)]
            setattr(self, gene + "_translate_position", [int(r[1]) for r in rows])
            setattr(self, gene + "_translate_residue", [r[2] for r in rows])
            setattr(self, gene + "_functionality", [r[3] for r in rows])
        if species == "human":     # germline CDR1 / CDR2 exist for human V genes only (translate.py:221-245)
            rows = [x.rstrip().split(" ") for x in tags.read_tcr_text(species, tagset, ch, "v", "cdrs", tagdir).splitlines(True)]
            self.v_cdr1, self.v_cdr2 = [r[1] for r in rows], [r[2] for r in rows]
        else:
            self.v_cdr1 = self.v_cdr2 = [""] * len(self.v_regions)
        self._j_motif = [re.compile(p) for p in self.j_translate_residue]
        self._prefix_aa = {}

    def as_tuple(self):
        return (self.v_regions, self.j_regions, self.v_names, self.j_names, self.v_translate_position, self.v_translate_residue,
                self.j_translate_position, self.j_translate_residue, self.v_functionality, self.j_functionality, self.v_cdr1,
                self.v_cdr2)

    def protein(self, v, vdel, tail):
        """Translation of v_region[: len - vdel] + tail.  The codons that lie wholly inside the V part are translated once
        per (gene, deletion) -- a repertoire has a few hundred of those and up to millions of rows."""
        key = (v, vdel)
        hit = self._prefix_aa.get(key)
        if hit is None:
            region = self.v_regions[v]
            v_used = region if vdel == 0 else region[:-vdel]
            whole = len(v_used) - len(v_used) % 3
            hit = (v_used, translate_nt(v_used[:whole]), v_used[whole:])
            self._prefix_aa[key] = hit
        v_used, aa, rest = hit
        return v_used, aa + translate_nt(rest + tail)


def import_gene_information(inputargs):
    """Gene-specific information for the translation (translate.py:123-254); returns the reference's 12-tuple."""
    global chain, _genes
    chain = inputargs["chain"]
    if inputargs["tags"] == "extended" and inputargs["species"] == "mouse":
        print("Please note that there is currently no extended tag set for mouse TCR genes.\n"
              "Decombinator will now switch the tag set in use from 'extended' to 'original'.\n"
              "In future, consider editing the script to change the default, "
              "or use the appropriate flags (-sp mouse -tg original).")
        inputargs["tags"] = "original"
    if inputargs["tags"] == "extended" and chain in ("g", "d"):
        print("Please note that there is currently no extended tag set for gamma/delta TCR genes.\n"
              "Decombinator will now switch the tag set in use from 'extended' to 'original'.\n"
              "In future, consider editing the script to change the default, or use the appropriate flags.")
        inputargs["tags"] = "original"
    if inputargs["species"] not in ("human", "mouse"):
        print("Species not recognised. Please select either 'human' (default) or 'mouse'.\n"
              "If mouse is required by default, consider changing the default value in the script.")
        sys.exit()
    _genes = GeneTables(inputargs)
    return _genes.as_tuple()


def get_cdr3(dcr, headers, inputargs):
    """Productivity of one DCR-assigned rearrangement -> dict of output fields (translate.py:257-357).
    import_gene_information() must have run."""
    g = _genes
    out = dict.fromkeys(headers, "")
    from_file = inputargs["command"] == "translate"
    out["decombinator_id"] = (",".join(dcr)) if from_file else (", ".join(dcr))
    out["rev_comp"] = "F"
    v, j, vdel, jdel = int(dcr[0]), int(dcr[1]), int(dcr[2]), int(dcr[3])
    ins_nt = dcr[4][1:] if from_file else dcr[4]          # fields of a .freq line keep their leading space

    out["v_call"] = g.v_names[v].split("*")[0]
    out["j_call"] = g.j_names[j].split("*")[0]

    # 1-2. rebuild the nucleotide sequence from the assignment, translate it
    tail = ins_nt + g.j_regions[j][jdel:]
    v_used, aa = g.protein(v, vdel, tail)
    seq = v_used + tail
    out["sequence"], out["sequence_aa"] = seq, aa

    # 3-4. frame and stop codons
    in_frame = (len(seq) - 1) % 3 == 0
    out["vj_in_frame"] = "T" if in_frame else "F"
    has_stop = "*" in aa
    out["stop_codon"] = "T" if has_stop else "F"
    productive = in_frame and not has_stop

    # 5. conserved cysteine of the V gene (Python indexing on purpose, see the module docstring)
    start_cdr3 = end_cdr3 = 0
    if aa[g.v_translate_position[v] - 1] == g.v_translate_residue[v]:
        start_cdr3 = g.v_translate_position[v] - 1
        out["conserved_c"] = "T"
    else:
        productive = False
        out["conserved_c"] = "F"

    # 6. FGXG motif (or its equivalent for this J gene) downstream of it
    downstream = aa[start_cdr3:]
    jp = g.j_translate_position[j]
    if g._j_motif[j].findall(downstream[jp:jp + 4]):
        end_cdr3 = len(downstream) + jp + start_cdr3 + 1
        out["conserved_f"] = "T"
    else:
        productive = False
        out["conserved_f"] = "F"

    out["productive"] = "T" if productive else "F"
    if productive:
        out["junction_aa"] = aa[start_cdr3:end_cdr3]
        out["junction"] = seq[start_cdr3 * 3:3 * end_cdr3]
        out["cdr1_aa"] = g.v_cdr1[v]
        out["cdr2_aa"] = g.v_cdr2[v]
    return out


def findfile(filename):
    """translate.py:43-54"""
    try:
        open(str(filename), "rt").close()
    except Exception:
        print("Cannot find the specified input file. Please try again")
        sys.exit()


def sort_permissions(fl):
    if oct(os.stat(fl).st_mode)[4:] != "666":
        os.chmod(fl, 0o666)


def _resolve_chain(inputargs):
    """translate.py:398-429"""
    if not inputargs["chain"]:
        named = [x for x in ("alpha", "beta", "gamma", "delta") if x in inputargs["infile"].lower()]
        if len(named) == 1:
            return named[0][0]
    else:
        given = inputargs["chain"].upper()
        for letter, name in (("a", "ALPHA"), ("b", "BETA"), ("g", "GAMMA"), ("d", "DELTA")):
            if given in (letter.upper(), name, "TR" + letter.upper(), "TCR" + letter.upper()):
                return letter
    print("TCR chain not recognised. Please choose from a/b/g/d (case-insensitive).")
    sys.exit()


def _summary_file(logpath, stem):
    """First free name among Summary.csv, Summary2.csv, ... (translate.py:545-567)."""
    name = stem + ".csv"
    if not os.path.exists(name):
        return name, open(name, "wt")
    for i in range(2, 10000):
        name = stem + str(i) + ".csv"
        if not os.path.exists(name):
            return name, open(name, "wt")
    raise RuntimeError("no free summary file name")


def _device():
    """The dcb_dist context the device path runs on, or None when no CUDA device is usable."""
    global _dist
    if _dist is None:
        try:
            _dist = _lib.Dist(device=int(os.environ.get("LOCAL_RANK", "0")))
        except _lib.DcbError:
            _dist = False
    return _dist or None


def device_tables(g):
    """dcb_translate_tables of a GeneTables (built once per object), or None when the kernels cannot take this chain."""
    if not hasattr(g, "_device_tables"):
        g._device_tables = None
        nv, nj = len(g.v_regions), len(g.j_regions)
        if all(len(x) == nv for x in (g.v_names, g.v_translate_position, g.v_translate_residue, g.v_cdr1, g.v_cdr2)) and \
                all(len(x) == nj for x in (g.j_names, g.j_translate_position, g.j_translate_residue)):
            try:
                g._device_tables = _lib.TranslateTables(
                    g.v_regions, [n.split("*")[0] for n in g.v_names], g.v_translate_position, g.v_translate_residue, g.v_cdr1,
                    g.v_cdr2, g.j_regions, [n.split("*")[0] for n in g.j_names], g.j_translate_position, g.j_translate_residue)
            except (_lib.DcbError, UnicodeEncodeError):
                pass
    return g._device_tables


_U32 = 0xFFFFFFFF


def _parse_uints(buf, s, e):
    """int() of the fields buf[s:e] when every field is optional spaces then 1..15 digits; None otherwise."""
    n = len(s)
    width = e - s
    if n and (int(width.min()) < 1 or int(width.max()) > 16):
        return None
    val, seen = np.zeros(n, dtype=np.int64), np.zeros(n, dtype=bool)
    for k in range(int(width.max()) if n else 0):
        live = k < width
        c = buf[np.where(live, s + k, 0)].astype(np.int64)
        dig = live & (c >= 48) & (c <= 57)
        space = live & (c == 32)
        if (space & seen).any() or (live & ~dig & ~space).any():
            return None
        val = np.where(dig, val * 10 + (c - 48), val)
        seen |= dig
    return val if seen.all() else None


def _columns_from_freq(raw):
    """Columns of dcb_translate from .freq text (seven ',' separated fields per line), split as the host does:
    decombinator_id = ",".join(fields[:5]) (fields keep their leading space), insert = fields[4][1:], int() of the rest.
    None when the text is not plainly of that shape (the host path then reads it)."""
    buf = np.frombuffer(raw, dtype=np.uint8)
    if len(buf) == 0:
        return dict(text=buf, n=0)
    if (buf >= 0x80).any() or (buf == 13).any():        # decoding / universal newlines: the host's business
        return None
    ends = np.flatnonzero(buf == 10)
    if buf[-1] != 10:
        ends = np.append(ends, len(buf))
    n = len(ends)
    starts = np.empty(n, dtype=np.int64)
    starts[0] = 0
    starts[1:] = ends[:-1] + 1
    commas = np.flatnonzero(buf == 44)
    per_line = np.diff(np.searchsorted(commas, ends), prepend=0)
    if len(commas) != 6 * n or (per_line != 6).any():
        return None
    c = commas.reshape(n, 6)
    fs = [starts] + [c[:, k] + 1 for k in range(6)]
    fe = [c[:, k] for k in range(6)] + [ends]
    nums = {}
    for k in (0, 1, 2, 3, 5, 6):
        nums[k] = _parse_uints(buf, fs[k], fe[k])
        if nums[k] is None:
            return None
    ins_off = fs[4] + 1
    return dict(text=buf, n=n, v=nums[0], j=nums[1], vdel=nums[2], jdel=nums[3], freq=nums[5], cluster=nums[6],
                id_off=starts, id_len=c[:, 4] - starts, ins_off=ins_off, ins_len=np.maximum(fe[4] - ins_off, 0))


def _columns_from_rows(data):
    """Columns of dcb_translate from collapsinator's rows ([v, j, vdel, jdel, insert] as str, count and cluster size as
    int): decombinator_id = ", ".join(row[:5]).  None for rows of any other shape (the host path then takes them)."""
    if not isinstance(data, list):
        return None
    n = len(data)
    if n == 0:
        return dict(text=np.zeros(0, dtype=np.uint8), n=0)
    if any(len(r) != 7 for r in data):
        return None
    cols = list(zip(*data))
    if not all(type(x) is str for k in range(5) for x in cols[k]) or not all(type(x) is int for k in (5, 6) for x in cols[k]):
        return None
    try:
        nums = [np.fromiter(map(int, cols[k]), dtype=np.int64, count=n) for k in range(4)]
        freq = np.fromiter(cols[5], dtype=np.int64, count=n)
        cluster = np.fromiter(cols[6], dtype=np.int64, count=n)
        ids = [", ".join(r[:5]) for r in data]
        text = "\n".join(ids).encode("ascii")
    except (ValueError, OverflowError, UnicodeEncodeError):        # the host path raises (or copes) as it always did
        return None
    if any((x < 0).any() for x in nums):
        return None
    id_len = np.fromiter(map(len, ids), dtype=np.int64, count=n)
    id_off = np.zeros(n, dtype=np.int64)
    np.cumsum(id_len[:-1] + 1, out=id_off[1:])
    ins_len = np.fromiter(map(len, cols[4]), dtype=np.int64, count=n)
    return dict(text=np.frombuffer(text, dtype=np.uint8), n=n, v=nums[0], j=nums[1], vdel=nums[2], jdel=nums[3], freq=freq,
                cluster=cluster, id_off=id_off, id_len=id_len, ins_off=id_off + id_len - ins_len, ins_len=ins_len)


class TsvText:
    """The .tsv of a translate call as text: `header` + `body` (the kernels' lines, page-locked) -- what
    DataFrame.to_csv(sep="\\t", index=False) of the call's DataFrame writes."""

    def __init__(self, body, nobarcoding):
        self.header = ("\t".join(out_headers) + "\n").encode()
        self.body = body
        self.nobarcoding = nobarcoding

    def write(self, fh):
        fh.write(self.header)
        if len(self.body):
            fh.write(memoryview(self.body.a) if hasattr(self.body, "a") else self.body)

    def tobytes(self):
        return self.header + bytes(self.body)

    def frame(self):
        """The DataFrame of the host path: str columns, duplicate_count int64, av_UMI_cluster_size int64 (or "")."""
        import pandas as pd
        lines = bytes(self.body).decode("ascii").split("\n")[:-1]
        if not lines:
            return pd.DataFrame([], columns=out_headers)
        cols = dict(zip(out_headers, (list(c) for c in zip(*(line.split("\t") for line in lines)))))
        cols["duplicate_count"] = list(map(int, cols["duplicate_count"]))
        if not self.nobarcoding:
            cols["av_UMI_cluster_size"] = list(map(int, cols["av_UMI_cluster_size"]))
        return pd.DataFrame(cols, columns=out_headers)


def _translate_device(inputargs, g, data):
    """-> (TsvText, v, j, productive) or None when the host path must take the call."""
    d = _device()
    if d is None:
        return None
    tables = device_tables(g)
    if tables is None:
        return None
    if inputargs["command"] == "translate":
        opener = gzip.open if inputargs["infile"].endswith(".gz") else open
        with opener(inputargs["infile"], "rb") as fh:
            cols = _columns_from_freq(fh.read())
    else:
        cols = _columns_from_rows(data)
    if cols is None:
        return None
    nbc = bool(inputargs["nobarcoding"])
    if cols["n"] == 0:
        z = np.zeros(0, dtype=np.int64)
        return TsvText(b"", nbc), z, z, np.zeros(0, dtype=bool)
    clip = lambda a: np.minimum(a, _U32)
    body, productive, _ = _lib.translate_rows(d, tables, cols["text"], clip(cols["v"]), clip(cols["j"]), clip(cols["vdel"]),
                                              clip(cols["jdel"]), cols["id_off"], cols["id_len"], cols["ins_off"], cols["ins_len"],
                                              cols["freq"], cols["cluster"], inputargs["nonproductivefilter"], nbc)
    if body is None:
        return None
    return TsvText(body, nbc), cols["v"], cols["j"], productive


def _translate_host(inputargs, g, data):
    """The row loop of the reference's CDR3translator (translate.py:430-540) -> (DataFrame, v, j, productive)."""
    import pandas as pd
    from_file = inputargs["command"] == "translate"
    if from_file:
        opener = gzip.open if inputargs["infile"].endswith(".gz") else open
        infile = opener(inputargs["infile"], "rt")
    else:
        infile = data
    rows, vs, js, prod = [], [], [], []
    for line in infile:
        counts["line_count"] += 1
        if from_file:
            tcr = line.rstrip().split(",")
            tcr[5] = int(tcr[5])
            tcr[6] = int(tcr[6])
        else:
            tcr = line
        dcr = tcr[:5]
        v, j = int(tcr[0]), int(tcr[1])
        if inputargs["nobarcoding"]:
            frequency, cluster = 1, ""
        else:
            if not isinstance(tcr[5], int):
                print("TCR frequency could not be detected. If using non-barcoded data,"
                      " please include the additional '-nbc' argument when running"
                      " CDR3translator.")
                sys.exit()
            frequency = tcr[5]
            cluster = tcr[6] if isinstance(tcr[6], (int, float)) else ""
        fields = get_cdr3(dcr, out_headers, inputargs)
        fields["sequence_id"] = str(counts["line_count"])
        fields["duplicate_count"] = frequency
        fields["av_UMI_cluster_size"] = cluster
        productive = fields["productive"] == "T"
        if productive or not inputargs["nonproductivefilter"]:
            rows.append([fields[h] for h in out_headers])
        vs.append(v)
        js.append(j)
        prod.append(productive)
    if from_file:
        infile.close()
    out_df = pd.DataFrame(rows, columns=out_headers)
    print("CDR3 data written to dataframe")
    return out_df, vs, js, prod


def translate_tsv(inputargs: dict, data=None):
    """cdr3translator's work with the .tsv as text where a device is usable: -> TsvText, or the host path's
    DataFrame when no device is usable or a row is outside the kernels' envelope.  Writes the summary like
    cdr3translator.  Either result goes to io.write_out_translated."""
    global counts
    counts = coll.Counter()
    print("Running CDR3Translator version", __version__)
    ch = _resolve_chain(inputargs)
    inputargs["chain"] = ch          # the corrected value is what import_gene_information reads
    import_gene_information(inputargs)
    g = _genes

    if inputargs["command"] == "translate":
        findfile(inputargs["infile"])
    counts["line_count"] = 0
    print("Translating", chainnams[ch], "chain CDR3s from", inputargs["infile"])
    filename_id = os.path.basename(inputargs["infile"]).split(".")[0]
    count_functionality = inputargs["tags"] == "extended" and inputargs["species"] == "human"

    res = _translate_device(inputargs, g, data)
    if res is not None:
        print("CDR3 data translated on the GPU")
    else:
        res = _translate_host(inputargs, g, data)
        counts = coll.Counter()                  # recounted from the columns below, as for the device path
    out, v, j, productive = res
    v, j, productive = np.asarray(v, dtype=np.int64), np.asarray(j, dtype=np.int64), np.asarray(productive, dtype=bool)
    counts["line_count"] = len(productive)
    n_prod = int(productive.sum())
    if n_prod:
        counts["prod_recomb"] = n_prod
    if len(productive) - n_prod:
        counts["NP_count"] = len(productive) - n_prod
    if count_functionality:
        for tagp, sel in (("P", productive), ("NP", ~productive)):
            for gene, idx, func in (("V", v, g.v_functionality), ("J", j, g.j_functionality)):
                idx = np.where(idx < 0, idx + len(func), idx)          # Python indexing of the host loop
                for k, c in enumerate(np.bincount(idx[sel], minlength=len(func))):
                    if c:
                        counts[tagp + "_" + gene + "-" + func[k]] += int(c)

    if not inputargs["suppresssummary"]:
        logpath = inputargs["outpath"] + f"Logs{os.sep}"
        if not os.path.exists(logpath):
            os.makedirs(logpath)
        date = strftime("%Y_%m_%d")
        summaryname, fh = _summary_file(logpath, logpath + date + "_dcr_" + filename_id + f"_{chainnams[ch]}" + "_CDR3_Translation_Summary")
        inout_name = "_".join(f"{filename_id}".split("_")[:-1]) + f"_{chainnams[ch]}"
        text = ("Property,Value\nDirectory," + os.getcwd() + "\nInputFile," + inout_name + "\nOutputFile," + inout_name
                + "\nDateFinished," + date + "\nTimeFinished," + strftime("%H:%M:%S") + "\n\nInputArguments:,\n")
        for key in ("species", "chain", "tags", "dontgzip"):
            text += key + "," + str(inputargs[key]) + "\n"
        text += ("\nNumberUniqueDCRsInput," + str(counts["line_count"]) + "\nNumberUniqueDCRsProductive," + str(counts["prod_recomb"])
                 + "\nNumberUniqueDCRsNonProductive," + str(counts["NP_count"]))
        if count_functionality:
            text += "\n\nFunctionalityOfGermlineGenesUsed,"
            for p in ("P", "NP"):
                for gene in ("V", "J"):
                    for f in ("F", "ORF", "P"):
                        target = p + "_" + gene + "-" + f
                        text += "\n" + target + "," + str(counts[target])
        print(text, file=fh)
        fh.close()
        sort_permissions(summaryname)
    return out


def cdr3translator(inputargs: dict, data=None) -> "pandas.DataFrame":
    """Function wrapper for CDR3translator (translate.py:388-621)."""
    out = translate_tsv(inputargs, data)
    return out.frame() if isinstance(out, TsvText) else out
