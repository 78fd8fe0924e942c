"""Parity tests proper: the CUDA kernels, called through the C ABI (libdcb.so), against
  * fixtures recorded from the unmodified reference (tests/golden/dcr_cases.json.gz),
  * the reference's own golden .n12 files,
  * the oracle on seeded synthetic reads,
and, at BASELINE.json's full batch size, through size-independent properties.  Bit-exact everywhere."""
import hashlib
import os

import numpy as np
import pytest

import decombine_oracle as O
from decombinator_b200 import _lib, tags
from helpers import assert_records_equal, record_to_list, synth_batch

pytestmark = pytest.mark.gpu


def _ctx(info, **kw):
    vt, jt = info.tables()
    return _lib.Context(vt, jt, device=0, **kw)


# force_general: 0 = the shipped path (flat kernel -> half-tag kernel -> general kernel where the chain has one seed
# geometry and half tags of >= 10 bases, else the bit-filter exact kernels -> general kernel), 1 = general kernel only,
# 2 = bit-filter exact kernels only, 3 = the shipped path without the half-tag kernel
@pytest.mark.parametrize("force_general", [0, 1, 2, 3])
def test_cuda_matches_reference_fixtures(dcr_cases, force_general):
    names = dcr_cases["counters"]
    for gi, g in enumerate(dcr_cases["groups"]):
        info = tags.load(g["species"], g["tags"], g["chain"])
        ctx = _ctx(info, both_frames=(g["orientation"] == "both"), allow_ns=g["allowNs"], lenthreshold=g["lenthreshold"],
                   force_general=force_general)
        packed = _lib.pack_strings(g["reads"], revcomp=(g["orientation"] != "forward"))
        res, cnt = ctx.decombine(packed)
        got = [record_to_list(r, rec, g["orientation"]) for r, rec in zip(g["reads"], res)]
        bad = [i for i, (a, b) in enumerate(zip(got, g["results"])) if a != b]
        assert not bad, (gi, bad[:5], [g["reads"][i] for i in bad[:2]])
        assert {n: int(c) for n, c in zip(names, cnt)} == g["totals"], gi
        packed.free(); ctx.close()


# (species, tag set, chain, orientation, read length, substitution, N and junk rates); test_gpu_halftag_capacity.py runs
# them again on libraries built with the half-tag kernel's work lists shrunk
SYNTHETIC_SHAPES = [
    ("human", "extended", "b", "reverse", 250, 0.0, 0.0, 0.0),       # BASELINE configs[1] shape
    ("human", "extended", "b", "reverse", 250, 0.01, 0.001, 0.05),   # configs[2] shape (beta half)
    ("human", "extended", "a", "reverse", 250, 0.01, 0.001, 0.05),   # configs[2] shape (alpha half)
    ("human", "extended", "a", "both", 150, 0.01, 0.001, 0.05),
    ("human", "extended", "b", "reverse", 300, 0.005, 0.0005, 0.05),  # 20-word slots: the flat kernel's two hit words
    ("human", "extended", "a", "both", 310, 0.0, 0.0, 0.02),
    ("human", "original", "b", "forward", 300, 0.02, 0.002, 0.05),
    ("human", "original", "a", "reverse", 100, 0.01, 0.0, 0.0),
    ("mouse", "original", "g", "reverse", 250, 0.005, 0.0, 0.02),    # configs[4] shape
    ("mouse", "original", "d", "both", 250, 0.005, 0.001, 0.02),
    ("mouse", "original", "a", "reverse", 250, 0.01, 0.001, 0.02),
    ("human", "original", "a", "reverse", 250, 0.01, 0.002, 0.02),   # flat kernel + N + 6-base J halves: the J scan over the invalid-base column
]


@pytest.mark.parametrize("species,tagset,chain,orientation,L,sub,nrate,junk", SYNTHETIC_SHAPES)
def test_cuda_matches_oracle_on_synthetic(species, tagset, chain, orientation, L, sub, nrate, junk):
    info = tags.load(species, tagset, chain)
    n = 200000
    r1, off, ln = synth_batch(info, n, L, sub, nrate, junk, seed=20260002)
    if orientation == "forward":  # the generator emits reverse-strand reads
        packed_rc = _lib.pack_arrays(r1, off, ln, revcomp=True)
        r1 = np.frombuffer("".join(packed_rc.unpack(i) for i in range(2000)).encode(), dtype=np.uint8).copy()
        n = 2000
        off, ln = off[:n], ln[:n]
        packed_rc.free()
    orc = O.Oracle(O.TagSet(species, tagset, chain))
    want = orc.decombine_arrays(r1, off, ln, orientation, nthreads=os.cpu_count() or 4)
    packed = _lib.pack_arrays(r1, off, ln, revcomp=(orientation != "forward"))
    for force_general in (0, 1, 2, 3):
        ctx = _ctx(info, both_frames=(orientation == "both"), force_general=force_general)
        res, cnt = ctx.decombine(packed)
        assert_records_equal(res, want, orientation, "force_general=%s" % force_general)
        assert np.array_equal(cnt, orc.counts), dict(zip(O.COUNTER_NAMES, zip(cnt, orc.counts)))
        if force_general == 0 and tagset == "extended" and orientation != "both":
            # the half-tag kernel takes what the flat kernel queues; next to nothing is left for the general kernel
            assert ctx.halftag_kernel_name() == "dcb_halftag_kernel"
            assert ctx.last_general() <= 0.02 * n, (ctx.last_deferred(), ctx.last_general())
            if sub > 0:
                assert ctx.last_deferred() > 0.05 * n
        ctx.close()
    packed.free()


ALL_CHAINS = [(sp, ts, ch) for sp in ("human", "mouse") for ts in ("original", "extended") for ch in "abgd"]


@pytest.mark.parametrize("nrate", [0.0, 0.001])
@pytest.mark.parametrize("species,tagset,chain", ALL_CHAINS)
def test_halftag_kernel_serves_every_shipped_chain(species, tagset, chain, nrate):
    """Every shipped tag set / chain, 250-nt reads with 1 % substitutions (and 0.1 % N): the half-tag kernel is picked (its
    tables and columns fit an SM for each of them), it takes most of what the exact-tag kernel queues -- for the 12-nt J
    tags through the 6-mer scan, dcr_core.cuh half_jshort_at; reads with non-ACGT symbols too, which the bit-filter
    exact kernels hand over unsearched -- and the records and counters are the oracle's."""
    info = tags.load(species, tagset, chain)
    n = 40000
    r1, off, ln = synth_batch(info, n, 250, 0.01, nrate, 0.02, seed=20260006)
    orc = O.Oracle(O.TagSet(species, tagset, chain))
    want = orc.decombine_arrays(r1, off, ln, "reverse", nthreads=os.cpu_count() or 4)
    packed = _lib.pack_arrays(r1, off, ln, revcomp=True)
    ctx = _ctx(info)
    res, cnt = ctx.decombine(packed)
    assert_records_equal(res, want, "reverse", "%s %s %s" % (species, tagset, chain))
    assert np.array_equal(cnt, orc.counts), dict(zip(O.COUNTER_NAMES, zip(cnt, orc.counts)))
    assert ctx.halftag_kernel_name() == "dcb_halftag_kernel"
    assert ctx.last_deferred() > 0.05 * n and ctx.last_general() <= 0.35 * ctx.last_deferred(), (ctx.last_deferred(), ctx.last_general())
    res2, cnt2 = ctx.decombine(packed)                 # work lists filled by atomics: the order must not matter
    assert np.array_equal(res2, res) and np.array_equal(cnt2, cnt)
    packed.free(); ctx.close()


def test_mixed_alpha_beta_stream_config3():
    """BASELINE configs[2]: one mixed file (even reads alpha, odd reads beta) analysed once per chain."""
    ia, ib = tags.load("human", "extended", "a"), tags.load("human", "extended", "b")
    n, L = 100000, 250
    sets = [(ia.v_regions, ia.j_regions), (ib.v_regions, ib.j_regions)]
    r1, off, ln = synth_batch(ia, n, L, 0.01, 0.001, 0.0, seed=20260003, sets=sets)
    packed = _lib.pack_arrays(r1, off, ln, revcomp=True)
    for chain, info in (("a", ia), ("b", ib)):
        orc = O.Oracle(O.TagSet("human", "extended", chain))
        want = orc.decombine_arrays(r1, off, ln, "reverse", nthreads=os.cpu_count() or 4)
        for fg in (0, 3):
            ctx = _ctx(info, force_general=fg)
            res, cnt = ctx.decombine(packed)
            assert_records_equal(res, want, "reverse", chain)
            assert np.array_equal(cnt, orc.counts)
            if fg == 0:   # the other chain's reads have no tag of this chain: more than half the file is queued, none for the general kernel
                assert ctx.last_deferred() > 0.5 * n and ctx.last_general() < 0.02 * n
            ctx.close()
    packed.free()


def test_ragged_empty_and_extreme_inputs():
    info = tags.load("human", "extended", "b")
    r1, off, ln = synth_batch(info, 3000, 250, 0.01, 0.001, 0.05, seed=5)
    reads = [bytes(r1[i * 250:(i + 1) * 250]).decode() for i in range(3000)]
    rng = np.random.default_rng(1)
    ragged = []
    for i, r in enumerate(reads):
        a, b = sorted(rng.integers(0, 251, size=2))
        ragged.append(r[a:b] if i % 3 else r)
    ragged += ["", "A", "N" * 250, "ACGT" * 1000, "N", "acgt" * 30, reads[0] * 8, (reads[1] + reads[2]) * 2]
    orc = O.Oracle(O.TagSet("human", "extended", "b"))
    want = orc.decombine_reads(ragged, "both")
    packed = _lib.pack_strings(ragged, revcomp=True)
    assert packed.uniform_len == 0 and packed.max_len == 4000
    # ragged reads of up to 320 nt, one frame: the flat kernel and the half-tag kernel on reads of every length
    short = [r for r in ragged if len(r) <= 320]
    orc1 = O.Oracle(O.TagSet("human", "extended", "b"))
    want1 = orc1.decombine_reads(short, "reverse")
    p1 = _lib.pack_strings(short, revcomp=True)
    assert p1.uniform_len == 0
    for fg in (0, 1, 3):
        ctx = _ctx(info, force_general=fg)
        res, cnt = ctx.decombine(p1)
        assert_records_equal(res, want1, "reverse", "ragged one frame fg=%s" % fg)
        assert np.array_equal(cnt, orc1.counts)
        if fg == 0:
            assert ctx.halftag_kernel_name() == "dcb_halftag_kernel" and ctx.last_deferred() > 0
        ctx.close()
    p1.free()
    for fg in (0, 1, 2, 3):
        ctx = _ctx(info, both_frames=True, force_general=fg)
        res, cnt = ctx.decombine(packed)
        assert_records_equal(res, want, "both", "ragged fg=%s" % fg)
        assert np.array_equal(cnt, orc.counts)
        ctx.close()
    packed.free()
    # empty batch
    ctx = _ctx(info)
    p0 = _lib.pack_strings([], revcomp=True)
    res, cnt = ctx.decombine(p0)
    assert len(res) == 0 and not cnt.any()
    ctx.close()


def _revcomp(s):
    return s[::-1].translate(str.maketrans("ACGT", "TGCA"))


@pytest.mark.parametrize("L", [128, 250, 320])
def test_tag_dense_reads(L):
    """Reads made of back-to-back tags give every lane of a warp ~10 seed hits (and every hit word its 'several
    occurrences' state): the confirmation loop of the exact-tag kernels must find them all, results unchanged.
    L = 320 needs the flat kernel's second hit word."""
    info = tags.load("human", "extended", "b")
    rng = np.random.default_rng(7)
    vs, js = list(info.v_seqs), list(info.j_seqs)
    r1, off, ln = synth_batch(info, 4000, L, 0.0, 0.0, 0.0, seed=3)
    reads = [bytes(r1[i * L:(i + 1) * L]).decode() for i in range(4000)]
    for i in range(0, 4000, 2):          # every other read, and one solid block of them
        parts = [(vs if rng.random() < 0.8 else js)[rng.integers(0, 14)] for _ in range(L // 20 + 1)]
        reads[i] = _revcomp("".join(parts)[:L])
    for i in range(1000, 1200):
        reads[i] = _revcomp("".join(vs[(i + k) % len(vs)] for k in range(L // 20 + 1))[:L])
    orc = O.Oracle(O.TagSet("human", "extended", "b"))
    want = orc.decombine_reads(reads, "reverse")
    packed = _lib.pack_strings(reads, revcomp=True)
    for fg in (0, 2, 3):
        ctx = _ctx(info, force_general=fg)
        res, cnt = ctx.decombine(packed)
        assert_records_equal(res, want, "reverse", "dense fg=%s" % fg)
        assert np.array_equal(cnt, orc.counts)
        ctx.close()
    packed.free()


def _digest(res):
    return hashlib.sha256(np.ascontiguousarray(res).tobytes()).hexdigest()


def test_full_size_properties_config2():
    """BASELINE configs[1] at full size (10 M x 250 nt, human beta): properties that do not need the oracle on
    every read -- determinism, the two independent kernels agreeing, shard invariance (checksum of checksums),
    counter conservation -- plus the oracle on a 500 k-read window."""
    info = tags.load("human", "extended", "b")
    n, L = 10_000_000, 250
    r1, off, ln = synth_batch(info, n, L, 0.0, 0.0, 0.0, seed=20260002)
    packed = _lib.pack_arrays(r1, off, ln, revcomp=True)
    ctx = _ctx(info)
    res, cnt = ctx.decombine(packed)
    res2, cnt2 = ctx.decombine(packed)
    assert _digest(res) == _digest(res2) and np.array_equal(cnt, cnt2)          # deterministic
    for fg in (1, 2, 3):
        ctxg = _ctx(info, force_general=fg)
        resg, cntg = ctxg.decombine(packed)
        assert _digest(res) == _digest(resg) and np.array_equal(cnt, cntg)      # independent kernels agree
        ctxg.close()
    # shard invariance: 8 contiguous shards (what 8 GPUs would each see) concatenate to the whole
    parts, csum = [], np.zeros_like(cnt)
    for s in range(8):
        lo, hi = n * s // 8, n * (s + 1) // 8
        p = _lib.pack_arrays(r1[lo * L:hi * L], off[:hi - lo], ln[:hi - lo], revcomp=True)
        rs, cs = ctx.decombine(p)
        parts.append(rs); csum += cs
        p.free()
    assert _digest(np.concatenate(parts)) == _digest(res) and np.array_equal(csum, cnt)
    # conservation: every read is decombined or accounted for by exactly one terminal counter
    c = dict(zip(O.COUNTER_NAMES, (int(x) for x in cnt)))
    ok = int(res["status"].sum())
    filt = sum(c[k] for k in ("dcrfilter_intertagN", "dcrfilter_toolong_intertag", "dcrfilter_imposs_deletion",
                              "dcrfilter_tag_overlap"))
    assert 0.9 * n < ok < n
    # every read whose V was assigned and whose J was not is counted once in VJ_assignment_failed (decombine.py:583-585);
    # the J-side counters can only exceed it (several half-tag candidates of one read may each fail their deletion walk,
    # and a J half2 failure is counted as foundv2notv1, decombine.py:526)
    assert c["VJ_assignment_failed"] >= c["multiple_j_matches"] + c["foundj1notj2"] + c["no_j_assigned"]
    # the oracle on a window in the middle
    lo, w = 4_000_000, 500_000
    orc = O.Oracle(O.TagSet("human", "extended", "b"))
    want = orc.decombine_arrays(r1[lo * L:(lo + w) * L], off[:w], ln[:w], "reverse", nthreads=os.cpu_count() or 4)
    assert_records_equal(res[lo:lo + w], want, "reverse", "window")
    assert ok + filt <= n
    ctx.close(); packed.free()


@pytest.mark.parametrize("tagset,chain,L", [("extended", "b", 250), ("extended", "a", 150), ("original", "a", 128),
                                            ("original", "b", 250), ("extended", "b", 318)])
def test_tag_position_sweep(tagset, chain, L):
    """Every tag at every start position modulo the seed stride and at both read ends (see sweep_reads), through every
    exact-tag kernel and the general kernel."""
    from test_device_logic_sim import sweep_reads
    info = tags.load("human", tagset, chain)
    reads = sweep_reads(info, L)
    orc = O.Oracle(O.TagSet("human", tagset, chain))
    want = orc.decombine_reads(reads, "reverse")
    packed = _lib.pack_strings(reads, revcomp=True)
    for fg in (0, 1, 2, 3):
        ctx = _ctx(info, force_general=fg)
        res, cnt = ctx.decombine(packed)
        assert_records_equal(res, want, "reverse", "sweep fg=%s" % fg)
        assert np.array_equal(cnt, orc.counts)
        ctx.close()
    packed.free()
