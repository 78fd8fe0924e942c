"""Decombine against the oracle on read shapes outside the envelope the fast kernels were tuned for: slots wider than 20
words (reads of 321 to 4096 nt, where the generic exact-tag kernel and a narrowed general kernel run and no half-tag
kernel), 4-word slots (batches of reads of at most 64 nt), the reference fixtures cut the way decombine_batch cuts a file,
reads dense in tags or in non-ACGT symbols, and a device-side exception list that overflows.  Every record field and every
counter is compared with the oracle; every GPU case also asserts which exact-tag / half-tag kernel it ran.

The reads are built on the host from seeded generators; the checks that they are what they claim to be (tag positions,
keyword occurrence counts, numbers of Ns) run without a GPU."""
import collections
import os

import numpy as np
import pytest

import decombine_oracle as O
from decombinator_b200 import _lib, decombine, fastq, tags
from helpers import assert_records_equal, record_to_list, synth_batch
from test_device_logic_sim import sweep_reads

NT = os.cpu_count() or 4
ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)

# 20 words is the widest slot of the flat, specialised and half-tag kernels (320 nt); 32 words = 512 nt; 4096 nt = the
# longest read (DCB_MAX_READ_LEN)
LONG_LENGTHS = [321, 336, 384, 448, 512, 513, 640, 1000, 1024, 1025, 2047, 2048, 3000, 4095, 4096]
# one seed geometry + union index (human extended b, human original a), two seed geometries (human original b), 12-nt J
# tags (mouse original g)
LONG_CHAINS = [("human", "extended", "b"), ("human", "original", "a"), ("human", "original", "b"), ("mouse", "original", "g")]
ALL_CHAINS = [(sp, ts, ch) for sp in ("human", "mouse") for ts in ("original", "extended") for ch in "abgd"]


def _ctx(info, **kw):
    vt, jt = info.tables()
    return _lib.Context(vt, jt, device=0, **kw)


def _rand(rng, k):
    return ACGT[rng.integers(0, 4, k)].tobytes().decode()


def _store(oriented, orientation):
    """Reads as they are analysed -> reads as they are stored: `reverse` stores the reverse complement, `both` every
    other read each way."""
    if orientation == "forward":
        return list(oriented)
    if orientation == "reverse":
        return [O.revcomp(r) for r in oriented]
    return [O.revcomp(r) if i % 2 == 0 else r for i, r in enumerate(oriented)]


def _arrays(reads):
    bufs = [r.encode("latin-1") for r in reads]
    ln = np.array([len(b) for b in bufs], dtype=np.uint32)
    off = np.zeros(len(bufs), dtype=np.uint64)
    if len(bufs) > 1:
        off[1:] = np.cumsum(ln[:-1], dtype=np.uint64)
    return np.frombuffer(b"".join(bufs) + b"\0" * 8, dtype=np.uint8).copy(), off, ln


def _synth_oriented(info, n, L, sub=0.0, nrate=0.0, junk=0.0, seed=1):
    """n synthetic reads of L nt in the frame they are analysed in (the generator emits the reverse strand): the
    rearrangement ends 20-60 nt + the constant region before the read's end, left of it random bases."""
    r1, _, _ = synth_batch(info, n, L, sub, nrate, junk, seed=seed)
    return [O.revcomp(bytes(r1[i * L:(i + 1) * L]).decode()) for i in range(n)]


def _want(key, reads, orientation, allow_ns=False, lenthreshold=130):
    orc = O.Oracle(O.TagSet(*key), allowNs=allow_ns, lenthreshold=lenthreshold)
    res = orc.decombine_reads(reads, orientation, nthreads=NT)
    return res, orc.counts.copy()


def _check(ctx, packed, want, orientation, what):
    res, cnt = ctx.decombine(packed)
    assert_records_equal(res, want[0], orientation, what)
    assert np.array_equal(cnt, want[1]), (what, dict(zip(O.COUNTER_NAMES, zip(cnt.tolist(), want[1].tolist()))))
    return res, cnt


def _same_records(a, b, what):
    """Two dcb_result arrays: same status, and the same fields on every decombined read."""
    assert np.array_equal(a["status"], b["status"]), what
    m = a["status"] != 0
    for f in ("v", "j", "vdel", "jdel", "ins_start", "ins_end", "v_seq_start", "j_seq_end", "frame"):
        assert np.array_equal(a[f][m], b[f][m]), (what, f)


# ---------------------------------------------------------------------------------------------------------------------
# read construction (host side)
# ---------------------------------------------------------------------------------------------------------------------
def molecule_reads(info, seed):
    """Rearrangements (200-nt synthetic molecules, 1 % substitutions, 0.2 % N) put at chosen offsets into random flanks,
    in the analysed frame: at the first bases; at 48 consecutive offsets around each of several 256 k-base boundaries (so
    the tags inside take every residue modulo the seed strides 8, 12 and 5 on both sides of the boundary); beyond 320,
    2048 and 4000; and cut off by the read's end (the constant region, then the J tag).  -> [(oriented read, offset)]."""
    rng = np.random.default_rng(seed)
    mols = _synth_oriented(info, 1200, 200, 0.01, 0.002, 0.0, seed=seed)
    out = []
    k = 0

    def put(p, L):
        nonlocal k
        m = mols[k % len(mols)]
        k += 1
        s = _rand(rng, p) + m + _rand(rng, max(0, L - p - len(m)))
        out.append((s[:L], p))
    for p in range(4):
        put(p, LONG_LENGTHS[(p * 5) % len(LONG_LENGTHS)])
    for b in (256, 512, 768, 1024, 2048, 3072, 3840):
        for d in range(-24, 24):
            # the V tag sits about 90-140 nt into a molecule: these offsets put it around the boundary
            put(b - 110 + d, 4096 if b >= 1024 else 1025)
    for p in (321, 330, 476, 500, 2049, 2100, 3500, 3896):
        put(p, 4096)
    for L in (513, 1024, 4096):                          # cut by the read's end: the constant region, then the J tag
        for c in range(0, 120, 4):
            put(L - 200 + c, L)
    return out


def tag_reads(info, L, pvs, seed):
    """One V tag at each start pv and one J tag behind it (30-38 nt on) or cut off by the read's end, random bases
    elsewhere, in the analysed frame (sweep_reads at chosen positions)."""
    rng = np.random.default_rng(seed)
    vs, js = list(info.v_seqs), list(info.j_seqs)
    out = []
    for i, pv in enumerate(pvs):
        vtag, jtag = vs[i % len(vs)], js[(i * 7 + pv) % len(js)]
        for pj in (pv + len(vtag) + 30 + (pv % 9), L - len(jtag) + 1 + (pv % 5)):
            body = bytearray(_rand(rng, L).encode())
            body[pv:pv + len(vtag)] = vtag.encode()
            body[pj:min(L, pj + len(jtag))] = jtag.encode()[:L - pj]
            out.append(bytes(body[:L]).decode())
    return out


def boundary_positions():
    return [b + d for b in (256, 512, 1024, 2048, 3840) for d in range(-12, 13)]


def long_batch(info, orientation, seed):
    """The ragged long-read batch of one chain: synthetic reads of every length of LONG_LENGTHS (1 % substitutions, 0.2 %
    N, 5 % junk), the placed molecules and the placed tags, stored for `orientation`."""
    oriented = []
    for L in LONG_LENGTHS:
        oriented += _synth_oriented(info, 60, L, 0.01, 0.002, 0.05, seed=seed + L)
    oriented += [s for s, _ in molecule_reads(info, seed)]
    oriented += tag_reads(info, 4096, [0, 1, 2, 3] + boundary_positions() + [4000, 4040], seed + 1)
    return _store(oriented, orientation)


def dense_reads(info, n, L, seed):
    """Tag-dense reads of L nt in the analysed frame: back-to-back V and J tags as they are, the same with one
    substitution in every tag, and half tags (one half of a tag, random bases for the other: half-tag keyword
    occurrences, no full tag) in front of a real rearrangement, whose tags come after more than DCB_HITS_CAP occurrences."""
    rng = np.random.default_rng(seed)
    vs, js = list(info.v_seqs), list(info.j_seqs)
    mols = _synth_oriented(info, n, 200, 0.0, 0.0, 0.0, seed=seed)

    def tagrun(k, sub):
        parts = []
        while sum(len(p) for p in parts) < k:
            t = bytearray(_pick(rng, vs, js).encode())
            if sub == 2:
                h = len(t) // 2
                if rng.random() < 0.5:
                    t[h:] = _rand(rng, len(t) - h).encode()
                else:
                    t[:h] = _rand(rng, h).encode()
            elif sub:
                q = int(rng.integers(0, len(t)))
                t[q] = ACGT[(list(ACGT).index(t[q]) + 1 + int(rng.integers(0, 3))) % 4]
            parts.append(bytes(t).decode())
        return "".join(parts)[:k]
    out = []
    for i in range(n):
        kind = i % 3
        if kind < 2:
            out.append(tagrun(L, kind == 1))
        else:
            m = mols[i]
            out.append(tagrun(L - len(m), 2) + m)
    return out


def _pick(rng, vs, js):
    return vs[int(rng.integers(0, len(vs)))] if rng.random() < 0.7 else js[int(rng.integers(0, len(js)))]


def keyword_occurrences(orc, read):
    """Occurrences of the keywords of the six sets (V, V half 1, V half 2, J, ...) in one analysed read, per set."""
    return [len(orc.findall(w, read, cap=4096)) for w in range(6)]


def tag_spans(orc, info, read):
    """(start, end) of the full V and J tags found in one analysed read."""
    spans = []
    for w, seqs in ((0, info.v_seqs), (3, info.j_seqs)):
        for kw, st in orc.findall(w, read):
            spans.append((st, st + len(seqs[kw])))
    return spans


def n_dense_reads(info, key, L, seed):
    """Reads of L nt with many non-ACGT symbols, in the analysed frame, as (kind, read) pairs: N at 0.5, 2 and 10 % per
    base; exactly 4 and 5 Ns inside the tags only, and outside them only; groups of 32 reads whose first read is all N (so
    each group's run of the exception list is longer than 32 entries) with Ns in the other reads' tags and inserts."""
    rng = np.random.default_rng(seed)
    orc = O.Oracle(O.TagSet(*key))
    out = []
    for j, rate in enumerate((0.005, 0.02, 0.1)):
        out += [("rate%g" % rate, r) for r in _synth_oriented(info, 320, L, 0.005, rate, 0.02, seed=seed + j)]
    clean = _synth_oriented(info, 1600, L, 0.0, 0.0, 0.0, seed=seed + 7)
    placed = 0
    for i, r in enumerate(clean):
        spans = tag_spans(orc, info, r)
        if len(spans) != 2:
            continue
        inside = sorted({p for a, b in spans for p in range(a, b)})
        outside = [p for p in range(L) if p not in set(inside)]
        k = 4 + (placed % 2)
        where = inside if (placed // 2) % 2 == 0 else outside
        if len(where) < k:
            continue
        s = bytearray(r.encode())
        for p in rng.choice(where, size=k, replace=False):
            s[int(p)] = ord("N")
        out.append(("%dN_%s" % (k, "in" if where is inside else "out"), bytes(s).decode()))
        placed += 1
        if placed == 640:
            break
    # 32-read groups led by an all-N read: the batch built so far is padded to a whole group first
    while len(out) % 32:
        out.append(("pad", _rand(rng, L)))
    grouped = _synth_oriented(info, 32 * 12, L, 0.0, 0.0, 0.0, seed=seed + 9)
    for g in range(12):
        out.append(("allN", "N" * L))
        for r in grouped[32 * g + 1:32 * g + 32]:
            s = bytearray(r.encode())
            spans = tag_spans(orc, info, r)
            if spans and g % 2 == 0:                     # an N inside a tag, on an A of the analysed frame where one exists
                a, b = spans[int(rng.integers(0, len(spans)))]
                p = next((q for q in range(a, b) if s[q] == ord("A")), a)
                s[p] = ord("N")
            elif spans:                                  # an N between the tags (the insert side)
                a, b = min(spans)[1], max(spans)[0]
                if b > a:
                    s[int(rng.integers(a, b))] = ord("N")
            out.append(("grouped", bytes(s).decode()))
    return out


def mixed_symbol_reads(info, L, seed):
    """Stored reads with U (a real base on the reverse strand: kind 3), N and lower case mixed in."""
    r1, _, _ = synth_batch(info, 640, L, 0.01, 0.002, 0.02, seed=seed)
    rng = np.random.default_rng(seed)
    out = []
    for i in range(640):
        s = bytearray(r1[i * L:(i + 1) * L].tobytes())
        for p in rng.integers(0, L, int(rng.integers(1, 9))):
            s[int(p)] = b"UUNnaucgt"[int(rng.integers(0, 9))]
        out.append(bytes(s).decode())
    return out


def short_reads(info, seed):
    """Batches whose longest read is 33 to 64 nt (4-word slots), analysed frame: synthetic reads, and rearrangements
    written out from the germline regions (V tag to the V end less 0-20 deleted bases, two inserted bases, J region from
    0-16 deleted bases to the J tag's end), those that fit in 64 nt."""
    out = []
    for L in (33, 40, 48, 64):
        out += _synth_oriented(info, 200, L, 0.01, 0.002, 0.05, seed=seed + L)
    for k, (vtag, vreg) in enumerate(zip(info.v_seqs, info.v_regions)):
        jreg, jtag = info.j_regions[k % len(info.j_regions)], info.j_seqs[k % len(info.j_seqs)]
        p, q = vreg.find(vtag), jreg.find(jtag)
        if p < 0 or q < 0:
            continue
        for vdel in (0, 4, 8, 12, 16, 20):
            for jdel in (0, 4, 8, 12, 16):
                s = vreg[p:len(vreg) - vdel] + "GA" + jreg[jdel:q + len(jtag)]
                if len(s) <= 64:
                    out.append(s)
    return out


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the constructed reads are what the GPU tests say they are
# ---------------------------------------------------------------------------------------------------------------------
def test_long_read_construction():
    info = tags.load("human", "extended", "b")
    placed = molecule_reads(info, 3)
    assert all(len(s) <= 4096 and set(s) <= set("ACGTN") for s, _ in placed)
    offs = [p for _, p in placed]
    assert min(offs) == 0 and max(offs) > 4000
    orc = O.Oracle(O.TagSet("human", "extended", "b"))
    deep = [s for s, p in placed if p > 2048 and len(s) == 4096]
    want = orc.decombine_reads(deep, "forward")
    assert want["ok"].sum() > 0.3 * len(deep) and want["v_seq_start"][want["ok"] == 1].min() > 2048
    reads = tag_reads(info, 4096, boundary_positions(), 1)
    found = [st for r in reads for kw, st in orc.findall(0, r)]
    for b in (256, 512, 1024, 2048, 3840):     # V tags at every residue modulo 8, 12 and 5 around the boundary
        near = {p for p in found if abs(p - b) <= 12}
        for s in (8, 12, 5):
            assert {p % s for p in near} == set(range(s))
    batch = long_batch(info, "reverse", 5)
    assert max(len(r) for r in batch) == 4096 and min(len(r) for r in batch) == 321
    assert {len(r) for r in batch} >= set(LONG_LENGTHS)


def test_dense_read_construction():
    """Every tag-dense read has more keyword occurrences than the general kernel's hit list holds (DCB_HITS_CAP = 16) and
    fewer per set than the oracle keeps (MAX_HITS = 2048)."""
    info = tags.load("human", "extended", "b")
    orc = O.Oracle(O.TagSet("human", "extended", "b"))
    for r in dense_reads(info, 60, 4096, 4):
        occ = keyword_occurrences(orc, r)
        assert sum(occ) > 16 and max(occ) < 2048, occ
    mixed = dense_reads(info, 30, 4096, 4)[2::3]          # half tags in front of a real rearrangement: the oracle finds it
    want = orc.decombine_reads(mixed, "forward")
    assert want["ok"].sum() > 0.6 * len(mixed)


def test_n_dense_construction():
    key = ("human", "extended", "b")
    info = tags.load(*key)
    orc = O.Oracle(O.TagSet(*key))
    reads = n_dense_reads(info, key, 250, 8)
    kinds = collections.Counter(k for k, _ in reads)
    assert kinds["4N_in"] > 100 and kinds["5N_in"] > 100 and kinds["4N_out"] > 100 and kinds["5N_out"] > 100
    for k, r in reads:
        if k[1:] == "N_in" or k[1:] == "N_out":
            assert r.count("N") == int(k[0])
            # inside: one of the two full tags is broken; outside: both are still found
            assert (len(tag_spans(orc, info, r)) < 2) == k.endswith("in"), k
        if k == "allN":
            assert r == "N" * 250
    first_all_n = [i for i, (k, _) in enumerate(reads) if k == "allN"]
    assert len(first_all_n) == 12 and all(i % 32 == 0 for i in first_all_n)
    assert 0.08 < np.mean([r.count("N") / 250 for k, r in reads if k == "rate0.1"]) < 0.12


def test_short_read_construction():
    info = tags.load("human", "extended", "b")
    reads = short_reads(info, 2)
    assert 33 <= max(len(r) for r in reads) <= 64
    want = O.Oracle(O.TagSet("human", "extended", "b")).decombine_reads(reads, "forward")
    assert want["ok"].sum() > 0.3 * len(reads)             # rearrangements that fit in 64 nt


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("orientation", ["reverse", "forward", "both"])
@pytest.mark.parametrize("key", LONG_CHAINS, ids=lambda k: "-".join(k))
def test_long_reads_match_oracle(key, orientation):
    """Ragged batches of 200-4096 nt (sweep_reads at 512, 1024 and 4096 nt too) and uniform batches at every length of
    LONG_LENGTHS, through the shipped path, the general kernel alone and the bit-filter exact kernels: the generic
    exact-tag kernel runs, no half-tag kernel."""
    info = tags.load(*key)
    seed = 100 + LONG_CHAINS.index(key)
    both = orientation == "both"
    rc = orientation != "forward"
    batches = [("ragged", long_batch(info, orientation, seed))]
    if orientation == "reverse":
        batches += [("sweep%d" % L, sweep_reads(info, L)) for L in (512, 1024, 4096)]
    batches += [("uniform%d" % L, _store(_synth_oriented(info, 64, L, 0.01, 0.002, 0.05, seed=seed + 7 * L), orientation))
                for L in LONG_LENGTHS]
    wants = [(name, reads, _want(key, reads, orientation)) for name, reads in batches]
    assert wants[0][2][0]["ok"].sum() > 0.2 * len(wants[0][1])
    for fg in (0, 1, 2):
        ctx = _ctx(info, both_frames=both, force_general=fg)
        for name, reads, want in wants:
            packed = _lib.pack_strings(reads, revcomp=rc)
            _check(ctx, packed, want, orientation, "%s fg=%d" % (name, fg))
            assert ctx.exact_kernel_name() == "dcb_exact_kernel" and ctx.halftag_kernel_name() == "", name
            packed.free()
        ctx.close()


@pytest.mark.gpu
def test_tag_dense_long_reads_overflow_the_hit_list():
    """4096 nt of back-to-back tags (exact, one substitution each, and substituted decoys in front of a real
    rearrangement): more keyword occurrences than DCB_HITS_CAP, so the general kernel drops its hit list and scans."""
    key = ("human", "extended", "b")
    info = tags.load(*key)
    oriented = dense_reads(info, 600, 4096, 12) + dense_reads(info, 300, 1000, 13)
    orc = O.Oracle(O.TagSet(*key))
    assert all(sum(keyword_occurrences(orc, r)) > 16 for r in oriented[:60])
    reads = _store(oriented, "reverse")
    want = _want(key, reads, "reverse")
    assert want[0]["ok"][2::3].sum() > 0.3 * len(reads) / 3
    packed = _lib.pack_strings(reads, revcomp=True)
    for fg in (0, 1, 2, 3):
        ctx = _ctx(info, force_general=fg)
        _check(ctx, packed, want, "reverse", "dense fg=%d" % fg)
        assert ctx.exact_kernel_name() == "dcb_exact_kernel"
        ctx.close()
    packed.free()


@pytest.mark.gpu
@pytest.mark.parametrize("key", ALL_CHAINS, ids=lambda k: "-".join(k))
def test_every_chain_at_4096_nt_both_frames(key):
    """The narrowest general-kernel blocks (tables + two frames of 4096 nt): every shipped chain must fit and match."""
    info = tags.load(*key)
    n, L = 2000, 4096
    reads = _store(_synth_oriented(info, n, L, 0.01, 0.002, 0.05, seed=31), "both")
    want = _want(key, reads, "both")
    packed = _lib.pack_strings(reads, revcomp=True)
    for fg in (0, 1):
        ctx = _ctx(info, both_frames=True, force_general=fg)
        _check(ctx, packed, want, "both", "4096 both fg=%d" % fg)
        assert ctx.exact_kernel_name() == "dcb_exact_kernel" and ctx.halftag_kernel_name() == ""
        ctx.close()
    packed.free()


@pytest.mark.gpu
@pytest.mark.parametrize("key", LONG_CHAINS, ids=lambda k: "-".join(k))
def test_four_word_slots(key):
    """Batches whose longest read is 33-64 nt: 4-word slots, which only the generic kernels serve."""
    info = tags.load(*key)
    oriented = short_reads(info, 41)
    for orientation in ("reverse", "forward", "both"):
        reads = _store(oriented, orientation)
        want = _want(key, reads, orientation)
        packed = _lib.pack_strings(reads, revcomp=orientation != "forward")
        assert packed.slot_words == 4
        for fg in (0, 1, 2, 3):
            ctx = _ctx(info, both_frames=orientation == "both", force_general=fg)
            _check(ctx, packed, want, orientation, "%s fg=%d" % (orientation, fg))
            assert ctx.exact_kernel_name() == "dcb_exact_kernel" and ctx.halftag_kernel_name() == ""
            ctx.close()
        packed.free()


@pytest.mark.gpu
def test_fixtures_through_the_fast_kernels(dcr_cases):
    """Each one-frame fixture group cut as decombine_batch cuts a file: reads of up to 320 nt in a batch of their own (the
    flat or specialised exact-tag kernel, then the half-tag kernel), the longer ones in another; together they give the
    recorded results and totals."""
    names = dcr_cases["counters"]
    ran = 0
    for gi, g in enumerate(dcr_cases["groups"]):
        if g["orientation"] == "both":
            continue
        info = tags.load(g["species"], g["tags"], g["chain"])
        lens = np.array([len(r) for r in g["reads"]])
        parts = [np.nonzero(lens <= 320)[0], np.nonzero(lens > 320)[0]]
        assert len(parts[0]) and len(parts[1]), gi
        for fg in (0, 3):
            ctx = _ctx(info, allow_ns=g["allowNs"], lenthreshold=g["lenthreshold"], force_general=fg)
            got = [None] * len(g["reads"])
            total = np.zeros(len(names), dtype=np.uint64)
            for pi, part in enumerate(parts):
                reads = [g["reads"][i] for i in part]
                packed = _lib.pack_strings(reads, revcomp=(g["orientation"] != "forward"))
                res, cnt = ctx.decombine(packed)
                if pi == 0:
                    assert packed.slot_words <= 20
                    assert ctx.exact_kernel_name() in ("dcb_exact_kernel_flat", "dcb_exact_kernel_spec"), (gi, ctx.exact_kernel_name())
                    if fg == 0:
                        assert ctx.halftag_kernel_name() == "dcb_halftag_kernel", gi
                for i, r, rec in zip(part, reads, res):
                    got[i] = record_to_list(r, rec, g["orientation"])
                total += cnt
                packed.free()
            bad = [i for i, (a, b) in enumerate(zip(got, g["results"])) if a != b]
            assert not bad, (gi, fg, bad[:5])
            assert {n: int(c) for n, c in zip(names, total)} == g["totals"], (gi, fg)
            ctx.close()
        ran += 1
    assert ran >= 5


def _batch_of(reads):
    b = fastq.ReadBatch()
    b.buf, b.off, b.len = _arrays(reads)
    return b


@pytest.mark.gpu
@pytest.mark.parametrize("n_long", [0, 1, 499, 500, 501, 1000], ids=["none", "one", "49.9%", "50%", "50.1%", "all"])
def test_decombine_batch_split(n_long, monkeypatch):
    """decombine_batch analyses the reads of up to 320 nt apart from the longer ones when at least half are short: the
    scattered records are the oracle's and those of one wide batch, the counters it adds up are the oracle's."""
    key = ("human", "extended", "b")
    info = tags.load(*key)
    n = 1000
    rng = np.random.default_rng(n_long)
    short = _synth_oriented(info, n, 250, 0.01, 0.002, 0.05, seed=61)
    long_ = [s for L in (400, 700, 1500, 4096) for s in _synth_oriented(info, 250, L, 0.01, 0.002, 0.05, seed=62 + L)]
    where = np.zeros(n, dtype=bool)
    where[rng.choice(n, n_long, replace=False)] = True
    reads = _store([long_[i] if where[i] else short[i] for i in range(n)], "reverse")
    want = _want(key, reads, "reverse")
    ctx = _ctx(info)
    monkeypatch.setattr(decombine, "_context", lambda inputargs, both: ctx)
    monkeypatch.setattr(decombine, "counts", collections.Counter())
    res = decombine.decombine_batch(_batch_of(reads), {"orientation": "reverse", "allowNs": False, "lenthreshold": 130})
    assert_records_equal(res, want[0], "reverse", "decombine_batch n_long=%d" % n_long)
    assert {k: decombine.counts[k] for k in O.COUNTER_NAMES} == dict(zip(O.COUNTER_NAMES, (int(c) for c in want[1])))
    packed = _lib.pack_strings(reads, revcomp=True)
    wide, _ = ctx.decombine(packed)
    _same_records(res, wide, "wide batch")
    packed.free(); ctx.close()


N_DENSE = [(("human", "extended", "b"), 250), (("human", "extended", "b"), 320), (("human", "original", "b"), 250),
           (("human", "original", "a"), 320)]


@pytest.mark.gpu
@pytest.mark.parametrize("key,L", N_DENSE, ids=lambda v: "-".join(v) if isinstance(v, tuple) else str(v))
def test_n_dense_reads(key, L):
    """Reads dense in N (and U, lower case): the flat kernel's exception probe and its hand-overs (more than four entries,
    none fetched, a group's run cut at entry 32), the half-tag kernel's invalid-base column and the general kernel's
    invalid-base masks in both frames.  allow_ns on and off, force_general 0-3, one frame and both, packed on the host and
    on the device."""
    info = tags.load(*key)
    oriented = [r for _, r in n_dense_reads(info, key, L, 17)]
    for orientation in ("reverse", "both"):
        reads = _store(oriented, orientation) + mixed_symbol_reads(info, L, 19)
        buf, off, ln = _arrays(reads)
        packed = _lib.pack_arrays(buf, off, ln, revcomp=True)
        assert packed.n_exc > 0.01 * len(reads) * L
        for allow_ns in (False, True):
            want = _want(key, reads, orientation, allow_ns=allow_ns)
            for fg in (0, 1, 2, 3):
                ctx = _ctx(info, both_frames=orientation == "both", allow_ns=allow_ns, force_general=fg)
                what = "%s allow_ns=%s fg=%d" % (orientation, allow_ns, fg)
                res, cnt = _check(ctx, packed, want, orientation, what)
                if fg in (0, 3):
                    assert ctx.exact_kernel_name() == ("dcb_exact_kernel_flat" if key[1] == "extended" else
                                                       ctx.exact_kernel_name() if key[2] == "a" else "dcb_exact_kernel_spec"), what
                if fg == 0 and orientation == "reverse":
                    assert ctx.halftag_kernel_name() == "dcb_halftag_kernel", what
                got, gcnt = ctx.decombine_ascii(buf, off, ln, True)
                assert_records_equal(got, want[0], orientation, what + " ascii")
                assert np.array_equal(gcnt, want[1]), what + " ascii"
                ctx.close()
        packed.free()


@pytest.mark.gpu
@pytest.mark.parametrize("share", ["0", "1"])
def test_long_reads_through_decombine_ascii(share, monkeypatch):
    """Long ragged reads packed on the device (and by the host threads where they are clean), from page-locked and
    pageable text, in chunks of 1024 reads: records and counters equal the host-packed batch's and the oracle's."""
    monkeypatch.setenv("DCB_HOST_SHARE", share)
    monkeypatch.setenv("DCB_CHUNK_READS", "1024")
    key = ("human", "extended", "b")
    info = tags.load(*key)
    oriented = []
    for L in LONG_LENGTHS:
        oriented += _synth_oriented(info, 400, L, 0.01, 0.0, 0.05, seed=71 + L)
    rng = np.random.default_rng(5)
    oriented = [oriented[i] for i in rng.permutation(len(oriented))]
    dirty = _synth_oriented(info, 400, 2048, 0.01, 0.002, 0.05, seed=72)      # one part with Ns: device-packed chunks
    reads = _store(oriented[:3000] + dirty + oriented[3000:], "reverse")
    buf, off, ln = _arrays(reads)
    want = _want(key, reads, "reverse")
    for fg in (0, 1):
        ctx = _ctx(info, force_general=fg)
        packed = _lib.pack_arrays(buf, off, ln, revcomp=True)
        ref, rcnt = _check(ctx, packed, want, "reverse", "host-packed fg=%d" % fg)
        packed.free()
        text = _lib.PinnedBytes(buf)
        for what, b in (("page-locked", text.a), ("pageable", buf)):
            got, cnt = ctx.decombine_ascii(b, off, ln, True)
            assert np.array_equal(got, ref) and np.array_equal(cnt, rcnt), (what, fg)
            host, dev = ctx.last_pack_shares()
            assert dev >= 1 and (share == "1" or host == 0), (what, host, dev)
        text.free()
        ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("share", ["0", "1"])
def test_over_full_device_exception_list(share, monkeypatch):
    """100 k reads of 250 nt, 10 % of them all N: 2.5 M non-ACGT symbols against a device list of 2 n + 2^20 entries.
    Packing on the device fails with DcbError (the kernels that ran read nothing past the list), the same context then
    decombines a normal batch correctly, and decombine_batch falls back to host packing and matches the oracle."""
    monkeypatch.setenv("DCB_HOST_SHARE", share)
    key = ("human", "extended", "b")
    info = tags.load(*key)
    n, L = 100_000, 250
    r1, off, ln = synth_batch(info, n, L, 0.01, 0.001, 0.05, seed=81)
    r1 = r1.copy()
    rng = np.random.default_rng(81)
    for i in rng.choice(n, n // 10, replace=False):
        r1[i * L:(i + 1) * L] = ord("N")
    normal, noff, nln = synth_batch(info, 50_000, L, 0.01, 0.002, 0.05, seed=82)
    ctx = _ctx(info)
    packed = _lib.pack_arrays(normal, noff, nln, revcomp=True)
    ref, rcnt = ctx.decombine(packed)
    packed.free()
    orc = O.Oracle(O.TagSet(*key))
    want = orc.decombine_arrays(r1, off, ln, "reverse", nthreads=NT)
    text = _lib.PinnedBytes(r1)
    for what, b in (("page-locked", text.a), ("pageable", r1)):
        with pytest.raises(_lib.DcbError, match="exceed the list capacity"):
            ctx.decombine_ascii(b, off, ln, True)
        with pytest.raises(_lib.DcbError, match="exceed the list capacity"):
            ctx.pack_device(b, off, ln, True)
        got, cnt = ctx.decombine_ascii(normal, noff, nln, True)             # the context is still sound
        assert np.array_equal(got, ref) and np.array_equal(cnt, rcnt), what
        batch = fastq.ReadBatch()
        batch.buf, batch.off, batch.len = b, off, ln
        monkeypatch.setattr(decombine, "_context", lambda inputargs, both: ctx)
        monkeypatch.setattr(decombine, "counts", collections.Counter())
        res = decombine.decombine_batch(batch, {"orientation": "reverse", "allowNs": False, "lenthreshold": 130})
        assert_records_equal(res, want, "reverse", what)
        assert {k: decombine.counts[k] for k in O.COUNTER_NAMES} == dict(zip(O.COUNTER_NAMES, (int(c) for c in orc.counts)))
    text.free()
    ctx.close()
