"""csrc/barcode_core.cuh compiled for the host (tests/sim/sim_barcode.cpp) against the host path of collapse.py
(get_barcode_positions / set_barcode / check_umi_quality with the installed `regex`), row by row: status, N1 length,
barcode, quality verdict and the match counters, on every single and double edit of every design's spacers at every
offset of their windows, edit pairs whose cost exceeds the fuzzy searches' limit, second hits, the str.find quirk of
getSpacerPositions, N with and without -N, and a seeded random sweep.  CPU only."""
import collections as coll
import ctypes
import itertools
import os
import random
import subprocess

import numpy as np
import pytest

from decombinator_b200 import _lib, collapse

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "sim", "sim_barcode.cpp")
SO = os.path.join(ROOT, "tests", "sim", "libbarcodesim.so")
OLIGOS = ["M13", "I8", "I8_single", "NEBIO", "TAKARA"]
QP = ([20, 1, 30], [30, 0, 35.5], [2, 5, 0])
MATCH_KEYS = ("getbarcode_pass_exactmatch", "getbarcode_pass_regexmatch", "getbarcode_pass_fuzzymatch_rightlen",
              "getbarcode_pass_fuzzymatch_short", "getbarcode_pass_fuzzymatch_long", "getbarcode_pass_other")
FAIL_KEYS = (("getbarcode_fail_N", _lib.BC_FAIL_N), ("getbarcode_fail_nospacerfound", _lib.BC_FAIL_NOSPACER),
             ("getbarcode_fail_not2spacersfound", _lib.BC_FAIL_NOT2), ("getbarcode_fail_n1tooshort", _lib.BC_FAIL_N1SHORT),
             ("getbarcode_fail_n1toolong", _lib.BC_FAIL_N1LONG), ("getbarcode_fail_n2pastend", _lib.BC_FAIL_N2END))

_sim = None


def sim():
    global _sim
    if _sim is None:
        dep = [SRC, os.path.join(ROOT, "decombinator_b200", "csrc", "barcode_core.cuh"), os.path.join(ROOT, "include", "dcb.h")]
        if not os.path.exists(SO) or any(os.path.getmtime(d) > os.path.getmtime(SO) for d in dep):
            subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-x", "c++", SRC, "-o", SO])
        _sim = ctypes.CDLL(SO)
        _sim.sim_barcode_row.argtypes = [ctypes.c_int] * 4 + [ctypes.c_double, ctypes.c_int, ctypes.c_char_p, ctypes.c_int,
                                         ctypes.c_char_p, ctypes.c_int] + [ctypes.c_void_p] * 4
        _sim.sim_one_edit.argtypes = [ctypes.c_int, ctypes.c_char_p, ctypes.c_char_p, ctypes.c_int]
    return _sim


def device_row(oligo, bc, q, allow_ns, qp, fuzzy=True):
    """-> (status, n1len, barcode or None, match) of the core."""
    st, n1, code, match = ctypes.c_uint8(), ctypes.c_uint8(), ctypes.c_uint64(), ctypes.c_uint8()
    b, qq = bc.encode("ascii"), q.encode("ascii")
    rc = sim().sim_barcode_row(_lib.OLIGOS_ON_DEVICE[oligo.lower()], int(allow_ns), qp[0], qp[1], float(qp[2]), int(fuzzy), b, len(b),
                               qq, len(qq), ctypes.byref(st), ctypes.byref(n1), ctypes.byref(code), ctypes.byref(match))
    assert rc == 0
    barcode = None
    if st.value in (_lib.BC_OK, _lib.BC_FAIL_QUALITY):
        c = code.value
        barcode = "".join("ACGTNSL"[(c >> (3 * k)) & 7] for k in range(c >> 58))
    return st.value, n1.value, barcode, match.value


def match_class(oligo, status, n1, match):
    """The match counters _count_device_barcodes derives from a placed row's n1len and match byte."""
    if status not in (_lib.BC_OK, _lib.BC_FAIL_QUALITY):
        return ()
    n = 6 if oligo in ("NEBIO", "TAKARA") else n1
    out = ["getbarcode_pass_regexmatch" if match else "getbarcode_pass_exactmatch"]
    if match:
        out += ["getbarcode_pass_fuzzymatch_rightlen"] if n == 6 else ["getbarcode_pass_fuzzymatch_short"] if n in (4, 5) else \
            ["getbarcode_pass_fuzzymatch_long"] if n >= 7 else []
    elif n == 6:
        out.append("getbarcode_pass_other")
    return tuple(sorted(out))


def host_row(oligo, bc, q, allow_ns, qp):
    """-> (status, n1len, barcode or None, match counters) of the host path."""
    c = coll.Counter()
    saved = collapse.counts
    collapse.counts = coll.Counter()
    args = {"oligo": oligo, "allowNs": allow_ns}
    try:
        locs = collapse.get_barcode_positions(bc, args, c)
        if not locs:
            fails = [st for key, st in FAIL_KEYS if c[key]]
            assert len(fails) == 1, c
            return fails[0], 0, None, ()
        barcode, bq = collapse.set_barcode([None] * 8 + [bc, q], locs, args)
        bad = collapse.check_umi_quality(bq, qp)
        n1 = 0 if oligo in ("NEBIO", "TAKARA") else locs[1] - locs[0]
        return (_lib.BC_FAIL_QUALITY if bad else _lib.BC_OK), n1, barcode, tuple(sorted(k for k in MATCH_KEYS if c[k]))
    finally:
        collapse.counts = saved


def handed_back_ok(oligo, bc, q):
    """The rows the device leaves to the host even with the fuzzy searches on."""
    return (len(bc) > 250 or len(q) != len(bc) or bool(set(bc) - set("ACGTN"))
            or (oligo in ("NEBIO", "TAKARA") and len(bc) < _lib.BC_LENGTH[oligo.lower()]))


def check(oligo, rows, allow_ns=False, qps=QP[:1]):
    """Every row through both; -> Counter of the statuses seen."""
    seen = coll.Counter()
    for bc, q in rows:
        for qp in qps:
            st, n1, barcode, match = device_row(oligo, bc, q, allow_ns, qp)
            if st == _lib.BC_HOST:
                assert handed_back_ok(oligo, bc, q), (oligo, bc, q)
                seen[st] += 1
                continue
            want = host_row(oligo, bc, q, allow_ns, qp)
            got = (st, n1, barcode, match_class(oligo, st, n1, match))
            assert got == want, (oligo, bc, q, allow_ns, qp, got, want)
            seen[st] += 1
            seen["fuzzy"] += match
    return seen


def _rand(rng, n):
    return "".join(rng.choice("ACGT") for _ in range(n))


def _quals(rng, n):
    return "".join(rng.choice("IIIIIIIIIIFFF:5,#!") for _ in range(n))


# each design: spacer 1, spacer 2 (or None), where the layout puts spacer 1, the window of spacer 1
DESIGN = {"M13": ("GTCGTGACTGGGAAAACCCTGG", "GTCGTGAT", 0, (0, 32)), "I8": ("GTCGTGAT", "GTCGTGAT", 0, (0, 18)),
          "I8_single": ("ATCACGAC", None, 6, (0, 18)), "NEBIO": ("TACGGG", None, 18, (18, 28)),
          "TAKARA": ("GTACGGG", None, 12, (0, 19))}


def region(rng, oligo, sp1=None, sp2=None, at1=None, n1=6, length=42):
    """A barcode region of the design with (variants of) its spacers: spacer 1 at `at1` (default: where the layout puts
    it), for two spacers N1 of `n1` bases and then spacer 2, the rest random, cut or padded to `length`."""
    s1, s2, home, _ = DESIGN[oligo]
    sp1 = s1 if sp1 is None else sp1
    at1 = home if at1 is None else at1
    s = _rand(rng, at1) + sp1
    if s2 is not None:
        s += _rand(rng, n1) + (s2 if sp2 is None else sp2)
    return (s + _rand(rng, max(0, length - len(s))))[:length]


def edits1(sp):
    """Every single substitution, deletion and insertion (of each base, at every position, ends included)."""
    out = set()
    for i in range(len(sp)):
        for b in "ACGT":
            if b != sp[i]:
                out.add(sp[:i] + b + sp[i + 1:])
        out.add(sp[:i] + sp[i + 1:])
    for i in range(len(sp) + 1):
        for b in "ACGT":
            out.add(sp[:i] + b + sp[i:])
    out.discard(sp)
    return sorted(out)


def subs2(sp):
    out = set()
    for i, j in itertools.combinations(range(len(sp)), 2):
        for a in "ACGT":
            for b in "ACGT":
                if a != sp[i] and b != sp[j]:
                    out.add(sp[:i] + a + sp[i + 1:j] + b + sp[j + 1:])
    return sorted(out)


def edits2(rng, sp, n):
    """n random variants of two edits of which at least one is an indel (a substitution and an indel, or two indels)."""
    out = []
    for _ in range(n):
        v = sp
        kinds = rng.choice((("s", "i"), ("s", "d"), ("i", "i"), ("d", "d"), ("i", "d")))
        for kind in kinds:
            p = rng.randrange(len(v) + (kind == "i"))
            if kind == "s":
                v = v[:p] + rng.choice([b for b in "ACGT" if b != v[p]]) + v[p + 1:]
            elif kind == "d":
                v = v[:p] + v[p + 1:]
            else:
                v = v[:p] + rng.choice("ACGT") + v[p:]
        out.append(v)
    return out


def offsets(oligo, variant):
    """Every start of a variant of spacer 1 in its window, and two beyond each edge (where it lies across lo or hi)."""
    lo, hi = DESIGN[oligo][3]
    return range(max(0, lo - 2), hi - len(variant) + 3)


def test_one_edit_primitives():
    """The one-edit tests of the {2i+2d+1s<=2} stage against brute force, for every spacer: a deletion at any position, an
    insertion only between two spacer bases.  (Within the stage an insertion before the first or after the last base
    cannot show: it leaves the spacer itself in the range, and the exact stage would have found it.)"""
    for sp in sorted({v for d in DESIGN.values() for v in d[:2] if v}):
        L = len(sp)
        for t in {sp[:i] + sp[i + 1:] for i in range(L)} | {v for v in subs2(sp)[::7]}:
            if len(t) == L - 1:
                assert sim().sim_one_edit(0, t.encode(), sp.encode(), L) == 1, (sp, t)
        for i in range(L + 1):
            for b in "ACGT":
                t = sp[:i] + b + sp[i:]
                inner = any(t[:j] + t[j + 1:] == sp for j in range(1, L))
                assert sim().sim_one_edit(1, t.encode(), sp.encode(), L) == int(inner), (sp, t)
        rng = random.Random(L)
        for _ in range(2000):
            t = "".join(rng.choice(sp[rng.randrange(L)] + "ACGT") for _ in range(L - 1))
            want = any(sp[:j] + sp[j + 1:] == t for j in range(L))
            assert sim().sim_one_edit(0, t.encode(), sp.encode(), L) == int(want), (sp, t)
            t = sp[:rng.randrange(L)] + "".join(rng.choice("ACGT") for _ in range(2))
            t = (t + sp[len(t) - 1:])[:L + 1]
            want = any(t[:j] + t[j + 1:] == sp for j in range(1, L))
            assert sim().sim_one_edit(1, t.encode(), sp.encode(), L) == int(want), (sp, t)


@pytest.mark.parametrize("oligo", OLIGOS)
def test_spacer1_single_edits_at_every_offset(oligo):
    rng = random.Random(10 * OLIGOS.index(oligo) + 1)
    sp1 = DESIGN[oligo][0]
    rows = []
    for v in edits1(sp1) + [sp1]:
        for at in offsets(oligo, v):
            bc = region(rng, oligo, sp1=v, at1=at, length=rng.choice((42, 60)))
            rows.append((bc, _quals(rng, len(bc))))
    seen = check(oligo, rows)
    assert seen["fuzzy"] > 0.2 * len(rows) and seen[_lib.BC_FAIL_NOSPACER], seen


@pytest.mark.parametrize("oligo", OLIGOS)
def test_spacer1_double_edits(oligo):
    """Every pair of substitutions at the layout's place and at a random offset; two edits with an indel (above the fuzzy
    searches' cost limit at that spot, yet another window may take them as substitutions)."""
    rng = random.Random(10 * OLIGOS.index(oligo) + 2)
    sp1 = DESIGN[oligo][0]
    rows = []
    for v in subs2(sp1):
        for at in (None, rng.choice(offsets(oligo, v))):
            bc = region(rng, oligo, sp1=v, at1=at)
            rows.append((bc, _quals(rng, len(bc))))
    for v in edits2(rng, sp1, 1500):
        bc = region(rng, oligo, sp1=v, at1=rng.choice(offsets(oligo, v)))
        rows.append((bc, _quals(rng, len(bc))))
    seen = check(oligo, rows)
    assert seen["fuzzy"] and seen[_lib.BC_FAIL_NOSPACER], seen


@pytest.mark.parametrize("oligo", ["M13", "I8"])
def test_spacer2_edits_at_every_n1(oligo):
    """Spacer 2's single edits behind every N1 length from 0 to 11, its double edits behind N1 of 6, and spacer 1 and 2
    edited together."""
    rng = random.Random(10 * OLIGOS.index(oligo) + 3)
    sp1, sp2 = DESIGN[oligo][:2]
    rows = []
    for v in edits1(sp2) + [sp2]:
        for n1 in range(12):
            bc = region(rng, oligo, sp2=v, n1=n1)
            rows.append((bc, _quals(rng, len(bc))))
    for v in subs2(sp2) + edits2(rng, sp2, 400):
        bc = region(rng, oligo, sp2=v)
        rows.append((bc, _quals(rng, len(bc))))
    e1, e2 = edits1(sp1), edits1(sp2)
    for _ in range(3000):
        bc = region(rng, oligo, sp1=rng.choice(e1), sp2=rng.choice(e2), n1=rng.choice((4, 5, 6, 6, 6, 7, 8)))
        rows.append((bc, _quals(rng, len(bc))))
    seen = check(oligo, rows)
    for st in (_lib.BC_OK, _lib.BC_FAIL_NOT2, _lib.BC_FAIL_N1SHORT, _lib.BC_FAIL_N1LONG):
        assert seen[st], seen


def test_second_fuzzy_hits_and_the_find_quirk():
    """Two fuzzy copies of a spacer in its range (one hit too many), an exact copy beside a fuzzy one, and M13 regions whose
    spacer 1 is matched as 21 or 23 bases, so str.find looks for spacer 2 from there rather than from 22 (where regex
    searched it): spacer 2 starting at 21, 22 or 23, with and without a later copy of its matched text."""
    rng = random.Random(4)
    rows = []
    for oligo in ("I8", "I8_single", "TAKARA", "M13"):
        sp1 = DESIGN[oligo][0]
        e = edits1(sp1)
        lo, hi = DESIGN[oligo][3]
        for _ in range(300):
            a, b = rng.choice(e), rng.choice(e + [sp1])
            bc = (_rand(rng, rng.randrange(0, 3)) + a + _rand(rng, rng.randrange(0, 3)) + b + _rand(rng, 42))[:42]
            rows.append((oligo, bc))
    m13, i8 = DESIGN["M13"][:2]
    longer = [v for v in edits1(m13) if len(v) == 23]
    shorter = [v for v in edits1(m13) if len(v) == 21]
    for v in longer + shorter:
        for at2 in (20, 21, 22, 23, 24):
            for text2 in [i8] + rng.sample(edits1(i8), 4):
                s = v + _rand(rng, 10)
                s = (s[:at2] + text2 + _rand(rng, 20))
                rows.append(("M13", s[:42]))
                s2 = (s[:at2 + len(text2) + 6] + text2 + _rand(rng, 20))           # a later copy of the matched text
                rows.append(("M13", s2[:48]))
    by = coll.defaultdict(list)
    for oligo, bc in rows:
        by[oligo].append((bc, _quals(rng, len(bc))))
    total = coll.Counter()
    for oligo, rs in by.items():
        total += check(oligo, rs)
    assert total["fuzzy"] and total[_lib.BC_FAIL_NOSPACER] and total[_lib.BC_FAIL_N1SHORT], total


@pytest.mark.parametrize("allow_ns", [False, True])
def test_n_in_and_around_the_spacers(allow_ns):
    """N is one more mismatching symbol for the fuzzy searches; without -N it rejects the row before any search."""
    rng = random.Random(5 + allow_ns)
    for oligo in OLIGOS:
        sp1, sp2 = DESIGN[oligo][:2]
        rows = []
        for _ in range(600):
            bc = list(region(rng, oligo, sp1=rng.choice(edits1(sp1) + [sp1]), sp2=None if sp2 is None else rng.choice(edits1(sp2) + [sp2])))
            for _ in range(rng.randrange(1, 3)):
                bc[rng.randrange(0, 40)] = "N"
            bc = "".join(bc)
            rows.append((bc, _quals(rng, len(bc))))
        seen = check(oligo, rows, allow_ns=allow_ns, qps=QP)
        assert seen[_lib.BC_FAIL_N] if not allow_ns else seen[_lib.BC_OK], seen


def test_known_answers_and_handed_back_rows():
    """The reference's known answers; symbols outside ACGTN, ragged quality strings, regions over 250 and TAKARA regions
    under 12 stay with the host; with the fuzzy stages off a row no exact search places is handed back."""
    rng = random.Random(6)
    for oligo, bc in (("M13", "GTCGTGACTGGGAAAACCCTGGTTTCCGGTCGTGATAAAGTG"), ("I8", "GTCGTGATTTTCCGGTCGTGATAAAGTG"),
                      ("I8_single", "GAAGCTATCACGACATCACTAC"), ("NEBIO", "CGGGCTTGGTATCGGCCGATCTACGGG"),
                      ("TAKARA", "CTCGTTAGGTTCGTACGGGGATTGCA"), ("M13", "GTCGTGACTGGGAAAACCCTGGTTNCCGGTCGTGATAAAGTG")):
        check(oligo, [(bc, "I" * len(bc))], qps=QP)
    for oligo in OLIGOS:
        bc = region(rng, oligo)
        for odd, q in ((bc[:5] + "R" + bc[6:], "I" * 42), (bc[:5] + "a" + bc[6:], "I" * 42), (bc, "I" * 41),
                       ((bc * 7)[:251], "I" * 251)):
            assert device_row(oligo, odd, q, False, QP[0])[0] == _lib.BC_HOST
        fuzzy1 = region(rng, oligo, sp1=edits1(DESIGN[oligo][0])[3])
        st, _, _, _ = device_row(oligo, fuzzy1, "I" * 42, False, QP[0], fuzzy=False)
        assert st == _lib.BC_HOST
        assert device_row(oligo, fuzzy1, "I" * 42, False, QP[0])[0] != _lib.BC_HOST
    # regions shorter than the fixed barcode: decided when no stage finds the spacer, handed back when one does
    short = [("TAKARA", "GTACGGGACGTACG"[:n]) for n in range(12)] + [("TAKARA", "ACGTAGTACGGA"[:n]) for n in range(12)]
    short += [("NEBIO", "CGGGCTTGGTATCGGCCGATCTACGGG"[:n]) for n in range(17)]
    got = coll.Counter()
    for oligo, bc in short:
        got[device_row(oligo, bc, "I" * len(bc), False, QP[0])[0]] += 1
        check(oligo, [(bc, "I" * len(bc))])
    assert got[_lib.BC_HOST] and got[_lib.BC_FAIL_NOSPACER], got


@pytest.mark.parametrize("oligo", OLIGOS)
def test_random_sweep(oligo):
    """Regions of the design with up to four random edits anywhere in their first 40 bases, of 12 to 60 bases."""
    rng = random.Random(7 + OLIGOS.index(oligo))
    rows = []
    for _ in range(4000):
        bc = list(region(rng, oligo, n1=rng.choice((4, 5, 6, 6, 6, 7, 8)), length=60))
        for _ in range(rng.randrange(0, 5)):
            p, kind = rng.randrange(0, 40), rng.randrange(3)
            if kind == 0:
                bc[p] = rng.choice("ACGT")
            elif kind == 1:
                del bc[p]
            else:
                bc.insert(p, rng.choice("ACGT"))
        bc = "".join(bc)[:rng.choice((12, 20, 30, 42, 42, 42, 60))]
        rows.append((bc, _quals(rng, len(bc))))
    check(oligo, rows, qps=QP)


def test_counters_of_a_batch():
    """_count_device_barcodes over the core's per-row outputs gives the counters the host path counts, row for row summed."""
    rng = random.Random(8)
    for oligo in OLIGOS:
        sp1, sp2 = DESIGN[oligo][:2]
        rows = [region(rng, oligo, sp1=rng.choice(edits1(sp1) + [sp1] * 20),
                       sp2=None if sp2 is None else rng.choice(edits1(sp2) + [sp2] * 10), n1=rng.choice((4, 5, 6, 6, 7, 8)))
                for _ in range(1500)]
        out = [device_row(oligo, bc, "I" * len(bc), False, QP[0]) for bc in rows]
        status = np.array([o[0] for o in out], dtype=np.uint8)
        n1 = np.array([o[1] for o in out], dtype=np.uint8)
        match = np.array([o[3] for o in out], dtype=np.uint8)
        saved = collapse.counts
        try:
            collapse.counts = coll.Counter()
            collapse._count_device_barcodes(status, n1, oligo.lower(), match)
            dev = collapse.counts
            collapse.counts = host = coll.Counter()
            for bc in rows:
                if collapse.get_barcode_positions(bc, {"oligo": oligo, "allowNs": False}, host):
                    pass
                else:
                    host["readdata_fail_no_bclocs"] += 1
                    continue
                locs = collapse.get_barcode_positions(bc, {"oligo": oligo, "allowNs": False}, coll.Counter())
                _, bq = collapse.set_barcode([None] * 8 + [bc, "I" * len(bc)], locs, {"oligo": oligo})
                if collapse.check_umi_quality(bq, QP[0]):
                    host["readdata_fail_low_barcode_quality"] += 1
        finally:
            collapse.counts = saved
        assert dev == host, (oligo, dev, host)
        assert dev["getbarcode_pass_regexmatch"] > 0, dev
