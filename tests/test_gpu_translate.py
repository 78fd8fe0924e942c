"""The translate stage on the device (dcb_translate, csrc/translate.cu) against the host path (get_cdr3 and the row loop,
DataFrame.to_csv): goldens, synthetic grids, fall-backs to the host, a million rows, and the command line without
pandas.  Needs a GPU (-m gpu)."""
import contextlib
import gzip
import os
import random
import re
import shutil
import subprocess
import sys

import numpy as np
import pandas as pd
import pytest

from decombinator_b200 import io, translate

from test_translate_sim import CHAINS, chain_args, rows_for, sim_row, tables

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@contextlib.contextmanager
def host_path():
    saved = translate._dist
    translate._dist = False
    try:
        yield
    finally:
        translate._dist = saved


def _args(infile, chain, outdir, command, **kw):
    a = io.create_args_dict(infile=str(infile), chain=chain, bc_read="R2", dontgzip=True, outpath=str(outdir) + os.sep,
                            tagfastadir="Decombinator-Tags-FASTAs", command=command)
    a.update(kw)
    return a


def device_tsv(args, data=None):
    out = translate.translate_tsv(dict(args), data)
    assert isinstance(out, translate.TsvText), "the call took the host path"
    return out


def host_text(args, data=None):
    with host_path():
        df = translate.cdr3translator(dict(args), data)
    return df.to_csv(sep="\t", index=False).encode(), df


def _summary(outdir):
    logs = sorted(os.listdir(os.path.join(outdir, "Logs")))
    text = open(os.path.join(outdir, "Logs", logs[-1])).read()
    return re.sub(r"(Directory|DateFinished|TimeFinished),.*", r"\1,", text)


def _golden_rows(golden_dir, name):
    rows = []
    for line in open(os.path.join(golden_dir, "dcr_TINY_1_%s.freq" % name)):
        f = line.rstrip("\n").split(", ")
        rows.append(f[:5] + [int(f[5]), int(f[6])])
    return rows


@pytest.mark.parametrize("chain,name", [("a", "alpha"), ("b", "beta")])
def test_goldens_through_the_device(golden_dir, tmp_path, chain, name):
    want = open(os.path.join(golden_dir, "dcr_TINY_1_%s.tsv" % name), "rb").read()
    freq = tmp_path / ("dcr_TINY_1_%s.freq" % name)
    shutil.copy(os.path.join(golden_dir, freq.name), freq)
    for command, data, infile in (("translate", None, freq), (None, _golden_rows(golden_dir, name), os.path.join(golden_dir, "TINY_1.fq"))):
        dev_dir, host_dir = tmp_path / ("dev_%s" % command), tmp_path / ("host_%s" % command)
        dev_dir.mkdir()
        host_dir.mkdir()
        args = _args(infile, chain, dev_dir, command)
        tsv = device_tsv(args, data)
        assert tsv.tobytes() == want
        io.write_out_translated(tsv, args)
        out_name = "dcr_TINY_1_%s.tsv" % name if command else "dcr_TINY_1_%s.tsv" % name
        assert (dev_dir / out_name).read_bytes() == want
        host_args = _args(infile, chain, host_dir, command)
        text, df = host_text(host_args, data)
        assert text == want
        pd.testing.assert_frame_equal(translate.cdr3translator(_args(infile, chain, dev_dir, command, suppresssummary=True), data), df)
        assert _summary(dev_dir) == _summary(host_dir)


def _grid_rows(species, tags, chain, seed=11):
    """The CPU grid of test_translate_sim, kept to the rows inside the kernels' envelope, as collapse rows."""
    args = chain_args(species, tags, chain)
    g, blob = tables(args)
    rng = random.Random(seed)
    rows = []
    for k, (v, j, vdel, jdel, ins) in enumerate(rows_for(g, rng)):
        if sim_row(blob, v, j, vdel, jdel, ins)[1] == 0:
            rows.append([str(v), str(j), str(vdel), str(jdel), ins, 1 + k % 7, 1 + k % 3])
    return rows


@pytest.mark.parametrize("species,tags,chain", CHAINS)
def test_synthetic_grids(tmp_path, species, tags, chain):
    rows = _grid_rows(species, tags, chain)
    assert len(rows) > 1000
    for kw in ({}, {"nonproductivefilter": True}, {"nobarcoding": True}):
        args = _args("dcr_grid_%s.freq" % chain, chain, tmp_path, None, species=species, tags=tags, suppresssummary=True, **kw)
        got = device_tsv(args, rows).tobytes()
        want, df = host_text(args, rows)
        assert got == want, kw
        pd.testing.assert_frame_equal(translate.cdr3translator(dict(args), rows), df)
    # the same rows as a gzipped .freq through the translate command
    path = tmp_path / ("grid_%s_%s.freq.gz" % (species, chain))
    with gzip.open(path, "wt") as fh:
        fh.writelines(", ".join(map(str, r)) + "\n" for r in rows)
    args = _args(path, chain, tmp_path, "translate", species=species, tags=tags, suppresssummary=True)
    assert device_tsv(args).tobytes() == host_text(args)[0]


def test_zero_rows(tmp_path):
    empty = tmp_path / "dcr_empty_beta.freq"
    empty.write_bytes(b"")
    for command, data, infile in (("translate", None, empty), (None, [], "dcr_empty_beta.freq")):
        args = _args(infile, "b", tmp_path, command, suppresssummary=True)
        assert device_tsv(args, data).tobytes() == host_text(args, data)[0]
        pd.testing.assert_frame_equal(translate.cdr3translator(dict(args), data), host_text(args, data)[1])


def test_rows_outside_the_envelope_take_the_host_path(golden_dir, tmp_path):
    rows = _golden_rows(golden_dir, "beta")
    # a quote in decombinator_id: to_csv quotes the field; the call goes to the host and writes the same bytes
    freq = tmp_path / "dcr_q_beta.freq"
    lines = open(os.path.join(golden_dir, "dcr_TINY_1_beta.freq")).read().splitlines(True)
    f = lines[3].split(", ")
    lines[3] = ", ".join(f[:4]) + ',"' + ", ".join(f[4:])
    freq.write_text("".join(lines))
    args = _args(freq, "b", tmp_path, "translate", suppresssummary=True)
    out = translate.translate_tsv(dict(args))
    assert isinstance(out, pd.DataFrame)
    assert out.to_csv(sep="\t", index=False).encode() == host_text(args)[0]
    assert b'"' in host_text(args)[0]
    # rows the host raises on: the same exception class on both
    for bad, exc in (([rows[0][:1] + ["99"] + rows[0][2:]], IndexError), ([rows[0][:4] + ["ACGXTT"] + rows[0][5:]], ValueError),
                     ([["1", "0", "9999", "9999", ""] + rows[0][5:]], IndexError), ([["x"] + rows[0][1:]], ValueError)):
        args = _args("dcr_bad_beta.freq", "b", tmp_path, None, suppresssummary=True)
        with pytest.raises(exc):
            translate.translate_tsv(dict(args), rows + bad)
        with pytest.raises(exc), host_path():
            translate.cdr3translator(dict(args), rows + bad)


def synthetic_rows(g, n, seed):
    """Seeded unique-DCR-like rows: random V / J of the chain, deletions 0..15, inserts of 0..30 bases with rare N."""
    rng = np.random.default_rng(seed)
    v = rng.integers(0, len(g.v_regions), n)
    j = rng.integers(0, len(g.j_regions), n)
    vdel, jdel = rng.integers(0, 16, n), rng.integers(0, 16, n)
    ln = rng.integers(0, 31, n)
    sym = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, int(ln.sum()))]
    sym[rng.random(len(sym)) < 0.002] = ord("N")
    text = sym.tobytes().decode()
    ends = np.cumsum(ln)
    starts = ends - ln
    ins = [text[a:b] for a, b in zip(starts.tolist(), ends.tolist())]
    freq = rng.integers(1, 50, n).tolist()
    clus = rng.integers(1, 9, n).tolist()
    return [[str(a), str(b), str(c), str(d), e, f, h] for a, b, c, d, e, f, h in
            zip(v.tolist(), j.tolist(), vdel.tolist(), jdel.tolist(), ins, freq, clus)]


def test_a_million_rows_equal_the_host_text(tmp_path):
    args = _args("dcr_big_beta.freq", "b", tmp_path, None, suppresssummary=True)
    translate.import_gene_information(chain_args("human", "extended", "b"))
    rows = synthetic_rows(translate._genes, 1_000_000, 20261020)
    got = device_tsv(args, rows).tobytes()
    want, _ = host_text(args, rows)
    assert got == want


_CLI = """
import runpy, sys
sys.argv = ["decombinator"] + sys.argv[1:]
runpy.run_module("decombinator_b200", run_name="__main__")
assert "pandas" not in sys.modules, "pandas was imported"
"""


@pytest.mark.parametrize("chain,name", [("a", "alpha"), ("b", "beta")])
def test_cli_writes_the_golden_tsv_without_pandas(golden_dir, tmp_path, chain, name):
    want = open(os.path.join(golden_dir, "dcr_TINY_1_%s.tsv" % name), "rb").read()
    for f in ("TINY_1.fq", "TINY_2.fq", "dcr_TINY_1_%s.freq" % name):
        shutil.copy(os.path.join(golden_dir, f), tmp_path / f)
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    o1, o2 = tmp_path / "o1", tmp_path / "o2"
    o1.mkdir()
    o2.mkdir()
    runs = ((["translate", "-in", str(tmp_path / ("dcr_TINY_1_%s.freq" % name)), "-c", chain, "-dz", "-op", str(o1) + os.sep], o1),
            (["pipeline", "-in", str(tmp_path / "TINY_1.fq"), "-c", chain, "-br", "R2", "-bl", "42", "-dc", "-dz", "-ol", "M13",
              "-op", str(o2) + os.sep], o2))
    for argv, out in runs:
        res = subprocess.run([sys.executable, "-c", _CLI] + argv, cwd=tmp_path, env=env, capture_output=True, text=True)
        assert res.returncode == 0, res.stdout + res.stderr
        assert "on the GPU" in res.stdout
        assert (out / ("dcr_TINY_1_%s.tsv" % name)).read_bytes() == want
