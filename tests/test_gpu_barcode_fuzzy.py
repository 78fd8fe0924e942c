"""dcb_barcodes_fuzzy: the reference's fuzzy spacer searches on the device.  The kernel row by row against the host path
(get_barcode_positions / set_barcode / check_umi_quality with `regex`) for all five designs, both -N settings and three
quality filters; the switch off against dcb_barcodes byte for byte; _filter_rows with the fuzzy searches on the device
against the host path for list rows, decombine.RowsColumns and N12Columns; the recorded reference runs and the
pipeline digests with the fuzzy searches on and with DCB_BC_FUZZY=0."""
import collections as coll
import ctypes
import os
import random

import numpy as np
import pytest

import collapse_checks
import oligo_layouts
import synth_pairs
import test_barcode_sim as bs
from decombinator_b200 import _lib, collapse, decombine, io

pytestmark = pytest.mark.gpu

OLIGOS = bs.OLIGOS


@pytest.fixture(scope="module")
def dist():
    d = _lib.Dist(0)
    yield d
    d.close()


@pytest.fixture(autouse=True)
def real_gpu_context():
    collapse._dist = None   # whatever an earlier (CPU) test installed: the product path builds its own dcb_dist
    yield


def _regions(oligo, seed, n=6000):
    """Regions of the design with substitutions, deletions and insertions in and around the spacers, N, odd symbols,
    ragged quality strings, short and overlong regions."""
    rng = random.Random(seed)
    sp1, sp2 = bs.DESIGN[oligo][:2]
    e1, e2 = bs.edits1(sp1), bs.edits1(sp2) if sp2 else None
    bcs, quals = [], []
    for i in range(n):
        r = rng.random()
        v1 = rng.choice(e1) if r < 0.45 else sp1
        v2 = rng.choice(e2) if e2 and (r > 0.35 and r < 0.7) else None
        at = None if rng.random() < 0.7 else rng.choice(bs.offsets(oligo, v1))
        bc = list(bs.region(rng, oligo, sp1=v1, sp2=v2, at1=at, n1=rng.choice((4, 5, 6, 6, 6, 6, 7, 8, 3, 9)),
                            length=rng.choice((42, 42, 42, 60, 30))))
        for _ in range(rng.choice((0, 0, 0, 1, 2))):          # more edits anywhere in the first 40 bases
            p, kind = rng.randrange(0, min(40, len(bc))), rng.randrange(4)
            if kind == 0:
                bc[p] = rng.choice("ACGT")
            elif kind == 1:
                del bc[p]
            elif kind == 2:
                bc.insert(p, rng.choice("ACGT"))
            else:
                bc[p] = "N"
        if rng.random() < 0.02:
            bc[rng.randrange(len(bc))] = rng.choice("acgtRY")
        bc = "".join(bc)
        if i % 97 == 0:
            bc = (bc + bs._rand(rng, 260))[:rng.choice((0, 1, 11, 12, 16, 24, 251))]
        q = bs._quals(rng, len(bc))
        if i % 53 == 0:
            q = q[:-1] if q else "I"
        bcs.append(bc)
        quals.append(q)
    return bcs, quals


@pytest.mark.parametrize("oligo", OLIGOS)
@pytest.mark.parametrize("allow_ns", [False, True])
def test_fuzzy_kernel_equals_the_host_path(dist, oligo, allow_ns):
    """Every row the kernel decides carries the host path's status, N1 length, barcode, quality verdict and match
    counters; it hands back only odd symbols, ragged quality strings, regions over 250 and short fixed-barcode regions."""
    bcs, quals = _regions(oligo, 40 + OLIGOS.index(oligo) + 10 * allow_ns)
    seen = coll.Counter()
    for qp in bs.QP:
        status, n1, code, match = dist.barcodes(bcs, quals, _lib.OLIGOS_ON_DEVICE[oligo.lower()], allow_ns, *qp, True)
        for i, (bc, q) in enumerate(zip(bcs, quals)):
            st = int(status[i])
            if st == _lib.BC_HOST:
                assert bs.handed_back_ok(oligo, bc, q), (i, bc, q)
                continue
            barcode = None
            if st in (_lib.BC_OK, _lib.BC_FAIL_QUALITY):
                c = int(code[i])
                barcode = "".join("ACGTNSL"[(c >> (3 * k)) & 7] for k in range(c >> 58))
            got = (st, int(n1[i]), barcode, bs.match_class(oligo, st, int(n1[i]), int(match[i])))
            want = bs.host_row(oligo, bc, q, allow_ns, qp)
            assert got == want, (i, bc, q, qp, got, want)
            seen[st] += 1
            seen["fuzzy"] += int(match[i])
    assert seen["fuzzy"] > 0.1 * len(bcs) and seen[_lib.BC_OK] and seen[_lib.BC_FAIL_QUALITY] and seen[_lib.BC_FAIL_NOSPACER], seen


@pytest.mark.parametrize("oligo", OLIGOS)
def test_switch_off_is_dcb_barcodes(dist, oligo):
    bcs, quals = _regions(oligo, 60 + OLIGOS.index(oligo), 4000)
    status, n1, code = dist.barcodes(bcs, quals, _lib.OLIGOS_ON_DEVICE[oligo.lower()], False, 20, 1, 30)
    bbuf = np.frombuffer("".join(bcs).encode() + b"\0", dtype=np.uint8)
    qbuf = np.frombuffer("".join(quals).encode() + b"\0", dtype=np.uint8)
    bl = np.array([len(x) for x in bcs], dtype=np.uint32)
    ql = np.array([len(x) for x in quals], dtype=np.uint32)
    bo = np.concatenate([[0], np.cumsum(bl[:-1], dtype=np.uint64)]).astype(np.uint64)
    qo = np.concatenate([[0], np.cumsum(ql[:-1], dtype=np.uint64)]).astype(np.uint64)
    n = len(bcs)
    st2, n12, cd2, m2 = np.full(n, 99, np.uint8), np.full(n, 99, np.uint8), np.full(n, 99, np.uint64), np.full(n, 99, np.uint8)
    prm = _lib.CBcParams(_lib.OLIGOS_ON_DEVICE[oligo.lower()], 0, 20, 1, 30.0)
    rc = _lib.lib().dcb_barcodes_fuzzy(dist._h, bbuf.ctypes.data, bo.ctypes.data, bl.ctypes.data, qbuf.ctypes.data, qo.ctypes.data,
                                       ql.ctypes.data, n, ctypes.byref(prm), 0, st2.ctypes.data, n12.ctypes.data, cd2.ctypes.data,
                                       m2.ctypes.data)
    assert rc == 0
    assert status.tobytes() == st2.tobytes() and n1.tobytes() == n12.tobytes() and code.tobytes() == cd2.tobytes()
    assert not m2.any()
    assert (status == _lib.BC_HOST).sum() > (dist.barcodes(bcs, quals, _lib.OLIGOS_ON_DEVICE[oligo.lower()], False, 20, 1, 30,
                                                           True)[0] == _lib.BC_HOST).sum()


def _with_indels(layout, seed):
    """Read 2 of a design with one base inserted or deleted in the first 40 bases of 4 % of the reads (length kept)."""
    rng = random.Random(seed)

    def f(b):
        b = layout(b) if layout else b
        L = len(b)
        if rng.random() < 0.04:
            p = rng.randrange(40)
            b = (b[:p] + b[p + 1:] + "A") if rng.random() < 0.5 else (b[:p] + rng.choice("ACGT") + b[p:])
        return b[:L]
    return f


class _HostCount:
    """The rows the product path's barcode kernel hands back."""

    def __init__(self, monkeypatch):
        self.host = 0
        real = _lib.Dist.barcodes_arrays

        def spy(d, *a):
            out = real(d, *a)
            self.host += int((out[0] == _lib.BC_HOST).sum())
            return out
        monkeypatch.setattr(_lib.Dist, "barcodes_arrays", spy)


def _filter(data, args, from_file=False):
    collapse.counts = coll.Counter()
    qp = [args["minbcQ"], args["bcQbelowmin"], args["avgQthreshold"]]
    kept, dcrs, n = collapse._filter_rows(data, args, qp, True, from_file)
    return kept, dcrs, n, {k: v for k, v in sorted(collapse.counts.items()) if not k.startswith("time_") and isinstance(v, int)}


@pytest.mark.parametrize("oligo", OLIGOS)
def test_filter_rows_fuzzy_on_the_device_equals_the_host(tmp_path, monkeypatch, oligo):
    """2 % substitutions and 4 % indels in read 2: the kept rows, DCR counter and collapse.counts of _filter_rows with the
    fuzzy searches on the device equal those without a device path, for list rows, RowsColumns and N12Columns; and the
    device hands back fewer rows than with DCB_BC_FUZZY=0."""
    layout, n1_at = oligo_layouts.LAYOUTS.get(oligo, (None, 22))
    f1, f2 = str(tmp_path / "s_1.fq"), str(tmp_path / "s_2.fq")
    synth_pairs.write_pairs(f1, f2, "human", "extended", "b", 8000, 500, 250, 0.004, 0.02, 20261300 + OLIGOS.index(oligo),
                            r2_layout=_with_indels(layout, 5), n1_at=n1_at)
    args = io.create_args_dict(infile=f1, chain="b", bc_read="R2", dontgzip=True, dontcount=True, suppresssummary=True, dontcheck=True,
                               outpath=str(tmp_path) + os.sep, species="human", tags="extended", oligo=oligo, command="pipeline")
    rows = decombine.decombinator(dict(args))
    cols = decombine.decombinator(dict(args, rows_as_columns=True))
    assert isinstance(cols, decombine.RowsColumns)
    path = str(tmp_path / "rows.n12")
    with open(path, "w") as fh:
        fh.write("".join(", ".join(r[:10]) + "\n" for r in rows))
    n12 = collapse.N12Columns.from_file(path, open)
    spy = _HostCount(monkeypatch)
    fuzzy = [_filter([list(r) for r in rows], args), _filter(cols, args), _filter(n12, args)]
    host_on = spy.host
    assert fuzzy[0][3]["getbarcode_pass_regexmatch"] > 0.005 * len(rows), fuzzy[0][3]
    monkeypatch.setenv("DCB_BC_FUZZY", "0")
    spy.host = 0
    exact = [_filter([list(r) for r in rows], args), _filter(cols, args), _filter(n12, args)]
    assert spy.host > host_on
    monkeypatch.delenv("DCB_BC_FUZZY")
    monkeypatch.setattr(_lib, "OLIGOS_ON_DEVICE", {})
    host = _filter([list(r) for r in rows], args)
    with open(path) as fh:
        host_file = _filter(fh, args, from_file=True)
    assert host_file == host
    for got in fuzzy + exact:
        assert got == host


def test_recorded_runs_and_digests_with_and_without_the_fuzzy_searches(golden_dir, tmp_path, monkeypatch):
    """The recorded collapse runs of the reference (all five designs), the golden .freq of the TINY fixture and the
    120 k / 60 k pipeline digests, with the fuzzy searches on the device and with DCB_BC_FUZZY=0; fewer rows handed back
    with them on."""
    import gzip
    import json
    from test_gpu_pipeline_scale import _digest_cases, _sha
    spy = _HostCount(monkeypatch)
    handed = {}
    for mode in ("1", "0"):
        monkeypatch.setenv("DCB_BC_FUZZY", mode)
        spy.host = 0
        for name in ("collapse_cases.json.gz", "collapse_cases_oligos.json.gz"):
            with gzip.open(os.path.join(golden_dir, name), "rt") as fh:
                for case in json.load(fh)["cases"]:
                    collapse_checks.check_case(case)
        for chain, name in (("a", "alpha"), ("b", "beta")):
            out = tmp_path / (mode + name)
            out.mkdir()
            collapse_checks.check_tiny_freq(golden_dir, out, chain, name)
        for index, case in enumerate(_digest_cases(golden_dir)):
            species, tagset, chain, n, pool, L, sub1, sub2, seed, oligo = case["spec"]
            f1, f2 = str(tmp_path / ("d%s%d_1.fq" % (mode, index))), str(tmp_path / ("d%s%d_2.fq" % (mode, index)))
            synth_pairs.write_pairs(f1, f2, species, tagset, chain, n, pool, L, sub1, sub2, seed)
            a = io.create_args_dict(infile=f1, chain=chain, bc_read="R2", dontgzip=True, dontcount=True, suppresssummary=True,
                                    dontcheck=True, outpath=str(tmp_path) + os.sep, species=species, tags=tagset, oligo=oligo,
                                    command="pipeline")
            a["rows_as_columns"] = True
            data = decombine.decombinator(a)
            assert _sha(bytes(data.text).decode()) == case["n12_sha256"]
            freq = collapse.collapsinator(dict(a), data=data)
            assert len(freq) == case["freq_rows"]
            assert _sha("".join(", ".join(map(str, r)) + "\n" for r in freq)) == case["freq_sha256"]
        handed[mode] = spy.host
    assert handed["1"] < handed["0"], handed
