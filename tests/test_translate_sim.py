"""csrc/translate_core.cuh compiled for the host (tests/sim/sim_translate.cpp) against translate.get_cdr3, field for field,
on every chain with .translate files; plus the host-side pieces of the device path (table checks, the .freq column
parse, the DataFrame rebuilt from .tsv text) and the no-GPU behaviour of dcb_translate.  CPU only."""
import ctypes
import io as pyio
import os
import random
import subprocess

import numpy as np
import pandas as pd
import pytest

from decombinator_b200 import _lib, translate

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "sim", "sim_translate.cpp")
SO = os.path.join(ROOT, "tests", "sim", "libtranslatesim.so")
CHAINS = [("human", "extended", "a"), ("human", "extended", "b"), ("human", "original", "a"), ("human", "original", "b"),
          ("mouse", "original", "a"), ("mouse", "original", "b")]
IUPAC = "ACGTURYSWKMBDHVN"

_sim = None


def sim():
    global _sim
    if _sim is None:
        dep = [SRC, os.path.join(ROOT, "decombinator_b200", "csrc", "translate_core.cuh")]
        if not os.path.exists(SO) or any(os.path.getmtime(d) > os.path.getmtime(SO) for d in dep):
            subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-x", "c++", SRC, "-o", SO])
        _sim = ctypes.CDLL(SO)
        _sim.sim_translate_row.restype = ctypes.c_long
        _sim.sim_translate_row.argtypes = [ctypes.c_void_p] + [ctypes.c_uint32] * 4 + [ctypes.c_char_p, ctypes.c_int, ctypes.c_char_p,
                                           ctypes.c_int] + [ctypes.c_int64] * 3 + [ctypes.c_int, ctypes.c_char_p, ctypes.c_long,
                                           ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int)]
    return _sim


def chain_args(species, tags, chain):
    return {"species": species, "tags": tags, "chain": chain, "tagfastadir": None, "command": None}


def tables(args):
    translate.import_gene_information(args)
    g = translate._genes
    t = translate.device_tables(g)
    assert t is not None
    return g, t.blob()


def sim_row(blob, v, j, vdel, jdel, ins, seq_id=7, freq=3, cluster=2, nbc=False):
    dcr = [str(v), str(j), str(vdel), str(jdel), ins]
    did = ", ".join(dcr).encode("latin-1")
    buf = ctypes.create_string_buffer(8192)
    flags, prod = ctypes.c_int(), ctypes.c_int()
    ib = ins.encode("latin-1")
    n = sim().sim_translate_row(blob.ctypes.data, v, j, vdel, jdel, ib, len(ib), did, len(did), seq_id, freq, cluster, int(nbc), buf,
                                8192, ctypes.byref(flags), ctypes.byref(prod))
    assert n >= 0
    return (buf.raw[:n].decode("latin-1") if n else None), flags.value, bool(prod.value)


def host_line(args, v, j, vdel, jdel, ins, seq_id=7, freq=3, cluster=2, nbc=False):
    """The .tsv line the host path writes for one in-memory row, or the exception class get_cdr3 raises."""
    try:
        f = translate.get_cdr3([str(v), str(j), str(vdel), str(jdel), ins], translate.out_headers, args)
    except Exception as e:       # noqa: BLE001 -- the class is what is compared
        return type(e)
    f["sequence_id"] = str(seq_id)
    f["duplicate_count"] = 1 if nbc else freq
    f["av_UMI_cluster_size"] = "" if nbc else cluster
    return "\t".join(str(f[h]) for h in translate.out_headers) + "\n"


def rows_for(g, rng):
    """(v, j, vdel, jdel, insert) grid of one chain."""
    nv, nj = len(g.v_regions), len(g.j_regions)
    rows = []
    for v in range(nv):                                   # every V x J
        for j in range(nj):
            ins = "".join(rng.choice("ACGT") for _ in range(rng.randint(0, 20)))
            rows.append((v, j, rng.randint(0, 15), rng.randint(0, 15), ins))
    for v in range(nv):                                   # vdel from 0 to beyond the region
        j = rng.randrange(nj)
        for vdel in range(0, len(g.v_regions[v]) + 4, 1 if v < 3 else 7):
            rows.append((v, j, vdel, rng.randint(0, 5), "".join(rng.choice("ACGT") for _ in range(rng.randint(0, 20)))))
    for j in range(nj):                                   # jdel likewise
        v = rng.randrange(nv)
        for jdel in range(0, len(g.j_regions[j]) + 4):
            rows.append((v, j, rng.randint(0, 5), jdel, "".join(rng.choice("ACGT") for _ in range(rng.randint(0, 20)))))
    alphabet = IUPAC + IUPAC.lower()
    for k in range(3000):                                 # inserts of 0..20 in all frames, IUPAC, lower case, U
        v, j = rng.randrange(nv), rng.randrange(nj)
        n = k % 21
        rows.append((v, j, rng.randint(0, 15), rng.randint(0, 15), "".join(rng.choice(alphabet) for _ in range(n))))
    for k in range(300):                                  # productive-looking rows: keep the frame of the V part
        v, j = rng.randrange(nv), rng.randrange(nj)
        rows.append((v, j, 0, 0, "".join(rng.choice("ACGT") for _ in range(3 * rng.randint(0, 6) + (k % 3)))))
    return rows


@pytest.mark.parametrize("species,tags,chain", CHAINS)
def test_core_matches_get_cdr3(species, tags, chain):
    args = chain_args(species, tags, chain)
    g, blob = tables(args)
    rng = random.Random(hash((species, tags, chain)) & 0xFFFF)
    n_prod = n_flag = 0
    for v, j, vdel, jdel, ins in rows_for(g, rng):
        for nbc in (False, True) if v == 0 else (False,):
            want = host_line(args, v, j, vdel, jdel, ins, nbc=nbc)
            got, flags, prod = sim_row(blob, v, j, vdel, jdel, ins, nbc=nbc)
            if isinstance(want, type):
                assert flags != 0, (v, j, vdel, jdel, ins, want)
                n_flag += 1
                continue
            assert flags == 0, (v, j, vdel, jdel, ins, flags)
            assert got.split("\t") == want.split("\t"), (v, j, vdel, jdel, ins)
            assert prod == (want.split("\t")[10] == "T")
            n_prod += prod
    assert n_prod > 100 and n_flag > 0


def test_position_zero_and_y_residue_genes_are_covered():
    args = chain_args("human", "extended", "b")
    g, blob = tables(args)
    assert 0 in g.v_translate_position and "Y" in g.v_translate_residue
    rng = random.Random(5)
    for v in [i for i, p in enumerate(g.v_translate_position) if p == 0] + [i for i, r in enumerate(g.v_translate_residue) if r == "Y"]:
        for j in range(len(g.j_regions)):
            for _ in range(20):
                ins = "".join(rng.choice("ACGT") for _ in range(rng.randint(0, 20)))
                vdel, jdel = rng.randint(0, 15), rng.randint(0, 15)
                want = host_line(args, v, j, vdel, jdel, ins)
                got, flags, _ = sim_row(blob, v, j, vdel, jdel, ins)
                if isinstance(want, type):
                    assert flags
                else:
                    assert got == want


def test_rows_the_host_rejects_are_flagged():
    args = chain_args("human", "extended", "b")
    g, blob = tables(args)
    nv, nj = len(g.v_regions), len(g.j_regions)
    assert host_line(args, nv, 0, 0, 0, "ACG") is IndexError and sim_row(blob, nv, 0, 0, 0, "ACG")[1] == _lib.TR_GENE
    assert host_line(args, 0, nj, 0, 0, "ACG") is IndexError and sim_row(blob, 0, nj, 0, 0, "ACG")[1] == _lib.TR_GENE
    assert host_line(args, 0, 0, 0, 0, "AC!GTA") is ValueError and sim_row(blob, 0, 0, 0, 0, "AC!GTA")[1] == _lib.TR_SYMBOL
    assert host_line(args, 0, 0, 0, 0, "ACXGTA") is ValueError and sim_row(blob, 0, 0, 0, 0, "ACXGTA")[1] == _lib.TR_SYMBOL
    assert host_line(args, 1, 0, 10 ** 4, 10 ** 4, "") is IndexError and sim_row(blob, 1, 0, 10 ** 4, 10 ** 4, "")[1] == _lib.TR_CINDEX
    assert sim_row(blob, 0, 0, 0, 0, "A" * 1100)[1] & _lib.TR_LONG
    # the device path leaves rows to_csv would quote to the host: a quote in decombinator_id
    assert sim_row(blob, 0, 0, 0, 0, 'AC"G')[1] & _lib.TR_QUOTE


@pytest.mark.parametrize("motif", ["FG.", "FG.GG", "F[GA]G", "fg.g", "F*GG", "FG\\G"])
def test_unsupported_motifs_are_refused(motif):
    args = chain_args("human", "extended", "b")
    translate.import_gene_information(args)
    g = translate._genes
    motifs = list(g.j_translate_residue)
    motifs[0] = motif
    with pytest.raises(_lib.DcbError) as e:
        _lib.TranslateTables(g.v_regions, g.v_names, g.v_translate_position, g.v_translate_residue, g.v_cdr1, g.v_cdr2,
                             g.j_regions, g.j_names, g.j_translate_position, motifs)
    assert e.value.rc == -4


def test_translate_fails_with_enogpu_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    g, _ = tables(chain_args("human", "extended", "b"))
    t = translate.device_tables(g)
    text = np.frombuffer(b"15, 10, 4, 1, CTACC", dtype=np.uint8)
    one = lambda x: np.array([x])
    with pytest.raises(_lib.DcbError, match=r"\(-2\).*no CUDA device"):
        _lib.translate_rows(None, t, text, one(15), one(10), one(4), one(1), one(0), one(19), one(14), one(5), one(1), one(1), False, False)
    with pytest.raises(_lib.DcbError, match="no CUDA device"):
        _lib.Dist()


def _freq_text(rows):
    return "".join(", ".join(map(str, r)) + "\n" for r in rows).encode()


def test_freq_columns_follow_the_host_split(golden_dir):
    raw = open(os.path.join(golden_dir, "dcr_TINY_1_beta.freq"), "rb").read()
    cols = translate._columns_from_freq(raw)
    lines = raw.decode().splitlines()
    assert cols["n"] == len(lines)
    for i, line in enumerate(lines):
        f = line.rstrip().split(",")
        ident = raw[cols["id_off"][i]:cols["id_off"][i] + cols["id_len"][i]].decode()
        ins = raw[cols["ins_off"][i]:cols["ins_off"][i] + cols["ins_len"][i]].decode()
        assert ident == ",".join(f[:5]) and ins == f[4][1:]
        assert [cols[k][i] for k in ("v", "j", "vdel", "jdel", "freq", "cluster")] == [int(f[k]) for k in (0, 1, 2, 3, 5, 6)]
    assert translate._columns_from_freq(raw.rstrip(b"\n"))["n"] == len(lines)          # no newline at the end
    # anything but plain digits, seven fields, ASCII and '\n' line ends goes to the host path
    for bad in (b"1, 2, 3, 4, AC, 5, 6, 7\n", b"1, 2, 3, 4, AC, 5\n", b"1, -2, 3, 4, AC, 5, 6\n", b"1, 2, 3, 4, AC, 5, 6 \n",
                b"1, 2, 3, 4, AC, 5, 6\r\n", b"1, 2, 3, 4, \xc3\xa9, 5, 6\n", b"1, 2, 3, 4, AC, 5, 6\n\n", b"1, 2 3, 3, 4, AC, 5, 6\n",
                b"1, 2, 3, 4, AC, 5, 1_0\n", b"1, 2, 3, 4, AC, 5, " + b"9" * 17 + b"\n"):
        assert translate._columns_from_freq(bad) is None, bad
    empty = translate._columns_from_freq(b"")
    assert empty["n"] == 0


def test_row_columns_take_only_collapse_shaped_rows():
    rows = [["15", "10", "4", "1", "CTACC", 1, 2], ["3", "2", "0", "0", "", 5, 1]]
    cols = translate._columns_from_rows(rows)
    text = cols["text"].tobytes().decode()
    assert [text[o:o + n] for o, n in zip(cols["id_off"], cols["id_len"])] == ["15, 10, 4, 1, CTACC", "3, 2, 0, 0, "]
    assert [text[o:o + n] for o, n in zip(cols["ins_off"], cols["ins_len"])] == ["CTACC", ""]
    for bad in ([["15", "10", "4", "1", "CTACC", 1]], [["15", "10", "4", "1", "CTACC", 1, 2.0]], [["15", "10", "4", "1", "CTACC", True, 2]],
                [[15, "10", "4", "1", "CTACC", 1, 2]], [["x", "10", "4", "1", "CTACC", 1, 2]], [["-1", "10", "4", "1", "CTACC", 1, 2]],
                [["1", "10", "4", "1", "CTAéC", 1, 2]], (r for r in rows)):
        assert translate._columns_from_rows(bad) is None


@pytest.mark.parametrize("nbc", [False, True])
def test_frame_from_text_equals_the_host_frame(golden_dir, tmp_path, nbc):
    """TsvText.frame() of the host path's own .tsv text rebuilds the host DataFrame, dtypes included."""
    rows = []
    for line in open(os.path.join(golden_dir, "dcr_TINY_1_beta.freq")):
        f = line.rstrip("\n").split(", ")
        rows.append(f[:5] + [int(f[5]), int(f[6])])
    args = dict(chain_args("human", "extended", "b"), infile="TINY_1.fq", suppresssummary=True, nobarcoding=nbc,
                nonproductivefilter=False, outpath=str(tmp_path) + os.sep, dontgzip=True)
    translate._dist = False                     # the host path, whatever this machine has
    try:
        df = translate.cdr3translator(args, data=rows)
    finally:
        translate._dist = None
    text = df.to_csv(sep="\t", index=False).encode()
    body = text.split(b"\n", 1)[1]
    got = translate.TsvText(body, nbc)
    assert got.tobytes() == text
    pd.testing.assert_frame_equal(got.frame(), df)
    empty = pd.DataFrame([], columns=translate.out_headers)
    pd.testing.assert_frame_equal(translate.TsvText(b"", nbc).frame(), empty)
    out = pyio.BytesIO()
    got.write(out)
    assert out.getvalue() == text
