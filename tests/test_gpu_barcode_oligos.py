"""dcb_barcodes for the single-spacer ligation-oligo designs I8_single, NEBIO and TAKARA (collapse.py:367-479): the kernel row by
row against the host path (get_barcode_positions / set_barcode / check_umi_quality), the counters and kept rows of
_filter_rows with and without the device path over every input form, the recorded reference runs of these designs through
the columnar hand-overs, and whole `pipeline` runs at 200 k read pairs with and without the device path."""
import collections as coll
import os
import random

import numpy as np
import pytest

import oligo_layouts
import synth_pairs
from decombinator_b200 import _lib, collapse, decombine, io, pipeline

pytestmark = pytest.mark.gpu

HOST_ONLY = {"m13": 0, "i8": 1}          # the designs the device took before: the rest go through the host path
SPACER = {"I8_single": "ATCACGAC", "NEBIO": "TACGGG", "TAKARA": "GTACGGG"}
WINDOW = {"I8_single": (0, 18), "NEBIO": (18, 28), "TAKARA": (0, 19)}
# where each design's layout puts the spacer, and the positions at both edges of its window and one beyond each edge
HOME = {"I8_single": 6, "NEBIO": 18, "TAKARA": 12}
EDGES = {"I8_single": (0, 10, 11), "NEBIO": (17, 18, 22, 23), "TAKARA": (0, 12, 13)}


@pytest.fixture(scope="module")
def dist():
    d = _lib.Dist(0)
    yield d
    d.close()


@pytest.fixture(autouse=True)
def real_gpu_context():
    collapse._dist = None   # whatever an earlier (CPU) test installed: the product path builds its own dcb_dist
    yield


def _host_barcode(bc, q, args, qp):
    """The host path for one row: -> (status, n1len as the kernel reports it, barcode or None)."""
    c = coll.Counter()
    saved = collapse.counts
    collapse.counts = coll.Counter()
    try:
        locs = collapse.get_barcode_positions(bc, args, c)
        if not locs:
            for key, st in (("getbarcode_fail_N", _lib.BC_FAIL_N), ("getbarcode_fail_nospacerfound", _lib.BC_FAIL_NOSPACER),
                            ("getbarcode_fail_not2spacersfound", _lib.BC_FAIL_NOT2), ("getbarcode_fail_n1tooshort", _lib.BC_FAIL_N1SHORT),
                            ("getbarcode_fail_n1toolong", _lib.BC_FAIL_N1LONG), ("getbarcode_fail_n2pastend", _lib.BC_FAIL_N2END)):
                if c[key]:
                    return st, 0, None
            raise AssertionError(c)
        barcode, bq = collapse.set_barcode([None] * 8 + [bc, q], locs, args)
        bad = collapse.check_umi_quality(bq, qp)
        n1 = 0 if args["oligo"] in ("NEBIO", "TAKARA") else locs[1] - locs[0]
        return (_lib.BC_FAIL_QUALITY if bad else _lib.BC_OK), n1, barcode
    finally:
        collapse.counts = saved


def _rand(rng, n):
    return "".join(rng.choice("ACGT") for _ in range(n))


def _region(rng, oligo, i):
    """One barcode region of the design (42 bases as a rule) with the edge cases the kernel has branches for."""
    sp = SPACER[oligo]
    lo, hi = WINDOW[oligo]
    r = rng.random()
    if oligo == "I8_single":               # N1 of 0..11 bases, N2 whole or cut short
        n1 = rng.choice((6, 6, 6, 6, 5, 4, 7, 8, 0, 1, 2, 3, 9, 10, 11))
        s = _rand(rng, n1) + sp + _rand(rng, rng.choice((28, 28, 28, 46, 5, 3, 0)))
    else:
        at = HOME[oligo] if r < 0.6 else rng.choice(EDGES[oligo])
        s = _rand(rng, at) + sp + _rand(rng, 42)
    s = list(s)[:rng.choice((42, 42, 42, 42, 30, 60))]
    k = rng.random()
    if k < 0.12:                           # substitutions in the spacer or beside it
        for _ in range(rng.randrange(1, 3)):
            p = min(len(s) - 1, max(0, lo + rng.randrange(-2, hi - lo + 2)))
            s[p] = rng.choice("ACGT")
    elif k < 0.18:                         # a second copy of the spacer inside the window
        p = rng.randrange(lo, max(lo + 1, hi - len(sp) + 1))
        s[p:p + len(sp)] = list(sp)
    elif k < 0.24:                         # an N, inside or outside the barcode
        s[rng.randrange(len(s))] = "N"
    elif k < 0.27:                         # lower case and IUPAC symbols
        s[rng.randrange(len(s))] = rng.choice("acgtnRYKMSW")
    elif k < 0.30 and s:
        del s[rng.randrange(len(s))]
    elif k < 0.33:
        s.insert(rng.randrange(len(s) + 1), rng.choice("ACGT"))
    s = "".join(s)
    if i % 97 == 0:                        # regions of 0, 1, 11, 12, 24 and 251 bases
        s = (s + _rand(rng, 260))[:rng.choice((0, 1, 11, 12, 24, 251))]
    q = "".join(rng.choice("IIIIIIIIIIFFF:5,#!") for _ in range(len(s)))
    if i % 53 == 0:
        q = q[:-1] if q else "I"           # a ragged quality string
    return s, q


def _handed_back_ok(oligo, bc, q):
    lo, hi = WINDOW[oligo]
    return (len(bc) > 250 or len(q) != len(bc) or bool(set(bc) - set("ACGTN")) or SPACER[oligo] not in bc[lo:hi]
            or (oligo == "TAKARA" and len(bc) < 12))


def _decode(code):
    return "".join("ACGTNSL"[(int(code) >> (3 * k)) & 7] for k in range(int(code) >> 58))


@pytest.mark.parametrize("oligo", ["I8_single", "NEBIO", "TAKARA"])
@pytest.mark.parametrize("allow_ns", [False, True])
def test_single_spacer_barcode_kernel_equals_the_host_path(dist, oligo, allow_ns):
    """Every row the kernel decides carries the host path's status, N1 length, barcode and quality verdict; every row it
    hands back has no exact spacer hit in the window, odd symbols, a ragged quality string, more than 250 bases, or (TAKARA)
    fewer than the barcode's 12."""
    rng = random.Random({"I8_single": 31, "NEBIO": 32, "TAKARA": 33}[oligo] + 10 * allow_ns)
    bcs, quals = zip(*[_region(rng, oligo, i) for i in range(6000)])
    sp, (lo, hi) = SPACER[oligo], WINDOW[oligo]
    # the spacer alone at every edge of its window, two copies in it, and the short regions, on a clean row each
    extra = [_rand(rng, at) + sp + _rand(rng, 42 - at - len(sp)) for at in EDGES[oligo] for _ in range(20)]
    extra += [_rand(rng, lo) + sp + sp + _rand(rng, 20) for _ in range(20)]
    extra += [(_rand(rng, HOME[oligo]) + sp + _rand(rng, 260))[:n] for n in (0, 1, 11, 12, 24, 251) for _ in range(5)]
    extra += [(_rand(rng, lo) + sp + _rand(rng, 30))[:n] for n in range(lo + len(sp), lo + len(sp) + 8) for _ in range(5)]
    bcs, quals = list(bcs) + extra, list(quals) + ["I" * len(x) for x in extra]
    args = {"oligo": oligo, "allowNs": allow_ns, "sampling_analysis": False}
    width = _lib.BC_LENGTH[oligo.lower()]
    seen = coll.Counter()
    for qp in ([20, 1, 30], [30, 0, 35.5], [2, 5, 0]):
        status, n1, code = dist.barcodes(bcs, quals, _lib.OLIGOS_ON_DEVICE[oligo.lower()], allow_ns, *qp)
        decided = 0
        for i, (bc, q) in enumerate(zip(bcs, quals)):
            if status[i] == _lib.BC_HOST:
                assert _handed_back_ok(oligo, bc, q), (i, bc, q)
                continue
            decided += 1
            st, hn1, barcode = _host_barcode(bc, q, args, qp)
            seen[int(st)] += 1
            assert status[i] == st, (i, bc, q, status[i], st)
            if st in (_lib.BC_OK, _lib.BC_FAIL_QUALITY):
                assert n1[i] == hn1, (i, bc)
                got = _decode(code[i])
                assert len(got) == width and got == barcode, (i, bc, got, barcode)
        assert decided > 0.6 * len(bcs), decided
    assert seen[_lib.BC_OK] and seen[_lib.BC_FAIL_QUALITY] and (allow_ns or seen[_lib.BC_FAIL_N]), seen
    if oligo != "NEBIO":                   # (NEBIO's 10-base window cannot hold two copies of its 6-base spacer)
        assert seen[_lib.BC_FAIL_NOSPACER], seen
    if oligo == "I8_single":
        assert seen[_lib.BC_FAIL_N1SHORT] and seen[_lib.BC_FAIL_N1LONG] and seen[_lib.BC_FAIL_N2END], seen


def test_an_unknown_design_is_refused(dist):
    with pytest.raises(_lib.DcbError):
        dist.barcodes(["A" * 42], ["I" * 42], 5, False, 20, 1, 30)


def _fastq(tmp_path, oligo, seed, n, pool, sub2, species="human", tagset="extended", chain="b"):
    layout, n1_at = oligo_layouts.LAYOUTS[oligo]
    f1, f2 = str(tmp_path / "s_1.fq"), str(tmp_path / "s_2.fq")
    synth_pairs.write_pairs(f1, f2, species, tagset, chain, n, pool, 250, 0.004, sub2, seed,
                            r2_layout=lambda b: layout(b)[:250], n1_at=n1_at)
    return f1


def _args(f1, oligo, tmp_path, species="human", tagset="extended", chain="b", **kw):
    a = io.create_args_dict(infile=f1, chain=chain, bc_read="R2", dontgzip=True, dontcount=True, suppresssummary=True, dontcheck=True,
                            outpath=str(tmp_path) + os.sep, species=species, tags=tagset, oligo=oligo, command="pipeline")
    a.update(kw)
    return a


def _int_counts():
    return {k: v for k, v in sorted(collapse.counts.items()) if not k.startswith("time_") and isinstance(v, int)}


def _filter(data, args, from_file=False):
    collapse.counts = coll.Counter()
    qp = [args["minbcQ"], args["bcQbelowmin"], args["avgQthreshold"]]
    kept, dcrs, n = collapse._filter_rows(data, args, qp, True, from_file)
    return kept, dcrs, n, _int_counts()


@pytest.mark.parametrize("oligo", ["I8_single", "NEBIO", "TAKARA"])
def test_filter_rows_with_and_without_the_device(tmp_path, monkeypatch, oligo):
    """The kept rows, the DCR counter and collapse.counts of _filter_rows are the same with the barcodes located on the
    device as on the host, for rows as lists, as decombine.RowsColumns and as the N12Columns of an .n12 file."""
    f1 = _fastq(tmp_path, oligo, 20261100, 6000, 400, 0.02)
    args = _args(f1, oligo, tmp_path)
    rows = decombine.decombinator(dict(args))
    cols = decombine.decombinator(dict(args, rows_as_columns=True))
    assert isinstance(cols, decombine.RowsColumns)
    path = str(tmp_path / "rows.n12")
    with open(path, "w") as fh:
        fh.write("".join(", ".join(r[:10]) + "\n" for r in rows))
    n12 = collapse.N12Columns.from_file(path, open)
    assert n12 is not None
    fast_list = _filter([list(r) for r in rows], args)
    fast_cols = _filter(cols, args)
    fast_n12 = _filter(n12, args)
    assert fast_list[3]["getbarcode_pass_exactmatch"] > 0.5 * len(rows)
    monkeypatch.setattr(_lib, "OLIGOS_ON_DEVICE", HOST_ONLY)
    host_list = _filter([list(r) for r in rows], args)
    host_cols = _filter(cols, args)
    with open(path) as fh:
        host_file = _filter(fh, args, from_file=True)
    assert fast_list == host_list
    assert fast_cols == host_cols == host_list
    assert fast_n12 == host_file == host_list


class _Spy:
    """Records the designs and statuses of the dcb_barcodes calls of the product path."""

    def __init__(self, monkeypatch):
        self.calls = []
        real = _lib.Dist.barcodes_arrays

        def spy(d, *a):
            out = real(d, *a)
            self.calls.append((a[6], out[0].copy()))
            return out
        monkeypatch.setattr(_lib.Dist, "barcodes_arrays", spy)

    def check(self, oligo):
        assert self.calls and all(c[0] == _lib.OLIGOS_ON_DEVICE[oligo.lower()] for c in self.calls)
        status = np.concatenate([c[1] for c in self.calls])
        assert float((status == _lib.BC_HOST).mean()) < 0.1
        self.calls.clear()


# the recorded cases 2-4 of collapse_cases_oligos.json.gz (oracle/make_golden_collapse_oligos.py):
# oligo, species, tags, chain, n reads, pool, sub1, sub2
RECORDED = {2: ("I8_single", "human", "extended", "b", 900, 80, 0.004, 0.01),
            3: ("NEBIO", "human", "extended", "a", 800, 60, 0.004, 0.01),
            4: ("TAKARA", "mouse", "original", "b", 800, 60, 0.004, 0.01)}


@pytest.mark.parametrize("index", [2, 3, 4])
def test_recorded_reference_runs_through_the_columnar_paths(golden_dir, tmp_path, monkeypatch, index):
    import gzip
    import json
    with gzip.open(os.path.join(golden_dir, "collapse_cases_oligos.json.gz"), "rt") as fh:
        case = json.load(fh)["cases"][index]
    oligo, species, tagset, chain, n, pool, sub1, sub2 = RECORDED[index]
    assert case["args"]["oligo"] == oligo
    layout, n1_at = oligo_layouts.LAYOUTS[oligo]
    f1, f2 = str(tmp_path / "s_1.fq"), str(tmp_path / "s_2.fq")
    synth_pairs.write_pairs(f1, f2, species, tagset, chain, n, pool, 250, sub1, sub2, 20260400 + index,
                            r2_layout=lambda b: layout(b)[:250], n1_at=n1_at)
    spy = _Spy(monkeypatch)
    a = _args(f1, oligo, tmp_path, species, tagset, chain, rows_as_columns=True)
    data = decombine.decombinator(a)
    assert isinstance(data, decombine.RowsColumns)
    n12 = "".join(", ".join(r[:10]) + "\n" for r in case["rows"])
    assert bytes(data.text).decode() == n12
    want_counts = case["counts_read_in_data"]

    def counts_after_read_in():
        return {k: v for k, v in _int_counts().items() if not k.startswith("number_output_")}
    args = dict(case["args"], infile=f1, outpath=str(tmp_path) + os.sep)
    freq = collapse.collapsinator(dict(args), data=data)
    assert freq == case["freq"]
    assert counts_after_read_in() == want_counts
    spy.check(oligo)
    path = str(tmp_path / "rows.n12")
    with open(path, "w") as fh:
        fh.write(n12)
    freq2 = collapse.collapsinator(dict(args, command="collapse", infile=path, dontcheckinput=True))
    assert freq2 == case["freq"]
    assert counts_after_read_in() == want_counts
    spy.check(oligo)


def _pipeline(tmp_path, f1, oligo, name):
    out = tmp_path / name
    out.mkdir()
    args = _args(f1, oligo, tmp_path, outpath=str(out) + os.sep)
    pipeline.run(dict(args))
    counts = _int_counts()
    files = {}
    for suffix in (".n12", ".freq"):
        with open(io.intermediate_filename(args, suffix)) as fh:
            files[suffix] = fh.read()
    return files, counts


@pytest.mark.parametrize("oligo", ["I8_single", "NEBIO", "TAKARA"])
def test_pipeline_at_size_with_and_without_the_device(tmp_path, monkeypatch, oligo):
    """200 k read pairs, 0.5 % substitutions in read 2: the same .n12, .freq and collapse counters either way."""
    f1 = _fastq(tmp_path, oligo, 20261200, 200_000, 10_000, 0.005)
    spy = _Spy(monkeypatch)
    native = []
    real_native = collapse._group_rows_native

    def native_spy(kept, frac):
        got = real_native(kept, frac)
        native.append((kept, frac, got))
        return got
    monkeypatch.setattr(collapse, "_group_rows_native", native_spy)
    fast, fast_counts = _pipeline(tmp_path, f1, oligo, "device")
    spy.check(oligo)
    assert len(native) == 1 and native[0][2] is not None
    kept, frac, groups = native[0]
    assert {len(k[1]) for k in kept} == {_lib.BC_LENGTH[oligo.lower()]}
    assert fast_counts["getbarcode_pass_exactmatch"] > 0.8 * fast_counts["readdata_input_dcrs"]
    monkeypatch.setattr(_lib, "OLIGOS_ON_DEVICE", HOST_ONLY)
    host, host_counts = _pipeline(tmp_path, f1, oligo, "host")
    assert fast[".n12"] == host[".n12"]
    assert fast[".freq"] == host[".freq"] and fast[".freq"]
    assert fast_counts == host_counts
    if oligo == "NEBIO":                   # 17-symbol barcodes: dcb_group against the Python state machines on the same rows
        monkeypatch.setenv("DCB_GROUP_NATIVE", "0")
        py = collapse._group_rows(kept, frac)
        assert sorted(py[0], key=lambda g: g[0]) == sorted(groups[0], key=lambda g: g[0]) and py[1:] == groups[1:]
