"""The half-tag kernel at and beyond the capacities of its work lists.

dcb_halftag_kernel (csrc/decombine.cu) pools the work of a warp's 32 reads in shared-memory lists of fixed size -- the
probe hits (DCB_HALF_WCAP = 192), the prefix hits and the (occurrence, tag) pairs (DCB_HALF_WCAP2 = 126 each) -- and keeps
at most DCB_HALF_CAP = 12 candidates per read.  Work that does not fit passes its read on to the general kernel; the
12-nt J scan takes a few reads per round so that its lists do not overflow.  Reads with 1 % substitutions rarely come near
these limits, so the reads here are built to:

  * V-dense reads: V tags back to back, each with one substitution (in its first half or its second, some of them tags
    whose intact half is shared with other tags), so no full V tag matches and every tag gives half-keyword occurrences
    and candidates; some with Ns between the tags, some with a real V region, insert and J region behind the decoys;
  * J-dense reads for the chains with short J halves: a clean V region followed by J tags with one substitution each,
    which drives the 6-mer J scan over several rounds; some with Ns next to the decoys or in place of the substitution;
  * both alone and interleaved with ordinary reads (1 % substitutions) at 1:1, 1:4 and 1:16, in reads of 128, 192, 250
    and 320 nt (8, 12, 16 and 20-word slots: one instantiation and block width of the kernel each).

Part (a) runs them on the shipped library; part (b) runs them, the synthetic shapes of test_cuda_matches_oracle_on_synthetic
and the mixed-chain files of configs[2] and configs[4] on libraries built with the capacities shrunk (build.VARIANTS), in
which nearly every warp overflows every list, so that every pass-on branch runs on ordinary data.  Records and all 20
counters are compared with the oracle everywhere, and every batch is run twice: the lists are filled by atomics, so their
order differs from run to run, and the output must not."""
import os
import subprocess
import sys

import numpy as np
import pytest

import decombine_oracle as O
from decombinator_b200 import _lib, build, tags
from helpers import assert_records_equal, synth_batch
from test_gpu_parity import SYNTHETIC_SHAPES

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CAP = 12                                  # DCB_HALF_CAP of the shipped library
WIDTHS = (128, 192, 250, 320)
DENSE = {                                 # workload -> tag set, and the gene whose tags are laid back to back
    "vdense_hb": ("human", "extended", "b", "v"),
    "vdense_ha": ("human", "extended", "a", "v"),
    "jdense_mg": ("mouse", "original", "g", "j"),      # the four chains whose J halves are below the sampled index
    "jdense_md": ("mouse", "original", "d", "j"),
    "jdense_ha": ("human", "original", "a", "j"),
    "jdense_hb": ("human", "original", "b", "j"),
}
MIX = (1, 4, 16)                          # ordinary reads per dense read in the mixed segments
BLOCK = 256                               # dense reads per segment (8 warps' worth in the solid block)


def _revcomp(s):
    return s[::-1].translate(str.maketrans("ACGTN", "TGCAN"))


class _Gene:
    """One gene's tags, with what the read builder and the candidate count need."""

    def __init__(self, seqs, regions, split):
        self.seqs, self.regions, self.split = list(seqs), list(regions), split
        by_half = [{}, {}]
        for i, t in enumerate(self.seqs):
            by_half[0].setdefault(t[:split], []).append(i)
            by_half[1].setdefault(t[split:], []).append(i)
        # tags whose first (second) half keyword is shared with other tags: a substitution in the OTHER half leaves an
        # occurrence that stands for several (occurrence, tag) pairs at once
        self.shared = [[i for i, t in enumerate(self.seqs) if len(by_half[h][t[:split] if h == 0 else t[split:]]) > 1]
                       for h in (0, 1)]
        # the half-tag search makes a candidate of a keyword occurrence only for the tags as long as the first tag with
        # that keyword (the reference's length guard); the count below keeps to tags whose keywords are all of one length
        lens = {k: {len(self.seqs[i]) for i in v} for h in (0, 1) for k, v in by_half[h].items()}
        self.countable = [i for i, t in enumerate(self.seqs) if len(lens[t[:split]]) == 1 and len(lens[t[split:]]) == 1]

    def decoy(self, rng, n_sub=False):
        """A tag with one substitution (an N when n_sub) in its first or its second half."""
        second = bool(rng.integers(0, 2))
        pool = self.shared[0 if second else 1] if rng.random() < 0.4 else ()
        t = self.seqs[pool[rng.integers(0, len(pool))] if len(pool) else rng.integers(0, len(self.seqs))]
        p = int(rng.integers(self.split, len(t))) if second else int(rng.integers(0, self.split))
        c = "N" if n_sub else "ACGT"[("ACGT".index(t[p]) + 1 + int(rng.integers(0, 3))) % 4]
        return t[:p] + c + t[p + 1:]

    def exact(self, a):
        return any(t in a for t in self.seqs)

    def n_candidates(self, a):
        """(tag, start) windows the half-tag search makes candidates of: a half keyword of the tag occurs there, the
        window lies inside the read and is within Hamming distance 1 of the tag (an N matches nothing)."""
        found = set()
        for i in self.countable:
            t = self.seqs[i]
            for off, half in ((0, t[:self.split]), (self.split, t[self.split:])):
                k = a.find(half)
                while k >= 0:
                    s = k - off
                    if s >= 0 and s + len(t) <= len(a) and sum(x != y for x, y in zip(a[s:s + len(t)], t)) <= 1:
                        found.add((i, s))
                    k = a.find(half, k + 1)
        return len(found)


def _random(rng, n):
    return "".join("ACGT"[b] for b in rng.integers(0, 4, size=n))


def _mutate(rng, s, lo, hi):
    p = int(rng.integers(lo, hi))
    return s[:p] + "ACGT"[("ACGT".index(s[p]) + 1 + int(rng.integers(0, 3))) % 4] + s[p + 1:]


def _v_part(rng, v, sub):
    """A real V region from its tag on (the tag with one substitution when sub)."""
    i = int(rng.integers(0, len(v.seqs)))
    reg, t = v.regions[i], v.seqs[i]
    p = reg.find(t)
    part = reg[p:]
    return _mutate(rng, part, 0, len(t)) if sub else part


def _j_part(rng, j, sub):
    """A real J region up to 8 bases behind its tag (the tag with one substitution when sub)."""
    i = int(rng.integers(0, len(j.seqs)))
    reg, t = j.regions[i], j.seqs[i]
    p = reg.find(t)
    part = reg[:p + len(t) + 8]
    return _mutate(rng, part, p, p + len(t)) if sub else part


def _fill(rng, gene, n, n_sep, n_sub):
    """n bases of decoys laid back to back (an N between some of them when n_sep, an N as the substitution of some when
    n_sub); the last one is cut off at n."""
    s = ""
    while len(s) < n:
        s += gene.decoy(rng, n_sub=n_sub and rng.random() < 0.3)
        if n_sep and rng.random() < 0.5:
            s += "N"
    return s[:n]


def _dense_read(rng, v, j, gene, L):
    """One dense read in the analysed orientation."""
    kind = int(rng.integers(0, 6))
    n_sep, n_sub = kind == 1, kind == 2
    if gene == "v":
        tail = ""
        if kind >= 3:         # a real rearrangement behind the decoys: clean, with a J error, or with a V error
            tail = _v_part(rng, v, kind == 5) + _random(rng, int(rng.integers(0, 8))) + _j_part(rng, j, kind == 4)
        tail = tail[-L:]
        return _fill(rng, v, L - len(tail), n_sep, n_sub) + tail
    head = _v_part(rng, v, False) + _random(rng, int(rng.integers(0, 8)))
    if kind == 3:             # fewer decoys, then a real J region with one error
        head += _fill(rng, j, int(rng.integers(0, 4)) * len(j.seqs[0]), False, False) + _j_part(rng, j, True)
    head = head[:L]
    body = _fill(rng, j, L - len(head), n_sep, n_sub)
    return head + body


class Workload:
    """Reads as sequenced (the reverse complement of the analysed orientation, like the synthetic generator's), the tag
    set and orientation they are analysed with; for dense workloads which reads are dense, and n_over, how many of them
    the half-tag kernel cannot decide (a lower bound computed here)."""

    def __init__(self, key, species, tagset, chain, orientation, buf, off, ln, n_over=0, dense=None):
        self.key, self.species, self.tagset, self.chain, self.orientation = key, species, tagset, chain, orientation
        self.buf, self.off, self.ln, self.n_over, self.dense = buf, off, ln, n_over, dense

    @property
    def info(self):
        return tags.load(self.species, self.tagset, self.chain)

    def oracle(self):
        """-> (records, counters) of the oracle."""
        orc = O.Oracle(O.TagSet(self.species, self.tagset, self.chain))
        want = orc.decombine_arrays(self.buf, self.off, self.ln, self.orientation, nthreads=os.cpu_count() or 4)
        return want, orc.counts.copy()

    def packed(self):
        return _lib.pack_arrays(self.buf, self.off, self.ln, revcomp=(self.orientation != "forward"))


def _from_strings(reads):
    ln = np.array([len(r) for r in reads], dtype=np.uint32)
    off = np.zeros(len(reads), dtype=np.uint64)
    off[1:] = np.cumsum(ln[:-1], dtype=np.uint64)
    return np.frombuffer("".join(reads).encode() + b"\0", dtype=np.uint8), off, ln


def dense_workload(name, L):
    """A solid block of dense reads, then one segment per MIX ratio of dense reads interleaved with ordinary ones."""
    species, tagset, chain, gene = DENSE[name]
    info = tags.load(species, tagset, chain)
    v = _Gene(info.v_seqs, info.v_regions, info.v_half_split)
    j = _Gene(info.j_seqs, info.j_regions, info.j_half_split)
    rng = np.random.default_rng([WIDTHS.index(L), list(DENSE).index(name), 20261020])
    n_ord = sum(BLOCK * r for r in MIX)
    r1, _, _ = synth_batch(info, n_ord, L, 0.01, 0.001, 0.02, seed=20261020 + L)
    ordinary = iter(bytes(r1[i * L:(i + 1) * L]).decode() for i in range(n_ord))
    analysed, dense = [], []
    for r in (0,) + MIX:
        for _ in range(BLOCK):
            analysed.append(_dense_read(rng, v, j, gene, L))
            dense.append(True)
            for _ in range(r):
                analysed.append(_revcomp(next(ordinary)))
                dense.append(False)
    n_over = 0
    for a, d in zip(analysed, dense):
        if not d:
            continue
        # a lower bound of the reads that cannot be decided here: more than CAP candidates of the gene the half-tag
        # search looks for -- V when no full V tag occurs; J when one does and no full J tag (for the chains with short
        # J halves only then are J candidates collected)
        if not v.exact(a):
            n_over += v.n_candidates(a) > CAP
        elif not j.exact(a):
            n_over += j.n_candidates(a) > CAP
    reads = [_revcomp(a) for a in analysed]
    buf, off, ln = _from_strings(reads)
    return Workload("%s_%d" % (name, L), species, tagset, chain, "reverse", buf, off, ln, n_over, np.array(dense))


def synthetic_workload(i, n=50000):
    """test_cuda_matches_oracle_on_synthetic's shape i, at n reads (forward: 2000, as there)."""
    species, tagset, chain, orientation, L, sub, nrate, junk = SYNTHETIC_SHAPES[i]
    info = tags.load(species, tagset, chain)
    r1, off, ln = synth_batch(info, n, L, sub, nrate, junk, seed=20260002)
    if orientation == "forward":          # the generator emits reverse-strand reads
        p = _lib.pack_arrays(r1, off, ln, revcomp=True)
        r1, off, ln = _from_strings([p.unpack(k) for k in range(2000)])
        p.free()
    return Workload("syn%d" % i, species, tagset, chain, orientation, r1, off, ln)


def mixed_workload(cfg, chain, n=50000):
    """configs[2] (human alpha / beta, extended tags, 1 % substitutions) or configs[4] (mouse gamma / delta): one file,
    even reads of the first chain and odd reads of the second, analysed once per chain."""
    species, tagset, pair, sub = {2: ("human", "extended", "ab", 0.01), 4: ("mouse", "original", "gd", 0.005)}[cfg]
    infos = [tags.load(species, tagset, c) for c in pair]
    sets = [(x.v_regions, x.j_regions) for x in infos]
    r1, off, ln = synth_batch(infos[0], n, 250, sub, 0.001, 0.02, seed=20260003 + cfg, sets=sets)
    return Workload("cfg%d%s" % (cfg, chain), species, tagset, chain, "reverse", r1, off, ln)


def variant_keys():
    return (["syn%d" % i for i in range(len(SYNTHETIC_SHAPES))] + ["cfg2a", "cfg2b", "cfg4g", "cfg4d"]
            + ["%s_%d" % (name, L) for name in DENSE for L in WIDTHS])


def workload(key):
    if key.startswith("syn"):
        return synthetic_workload(int(key[3:]))
    if key.startswith("cfg"):
        return mixed_workload(int(key[3]), key[4])
    name, L = key.rsplit("_", 1)
    return dense_workload(name, int(L))


def run(w, force_general=0):
    """-> (records, counters, (deferred, general), half-tag kernel name); the batch is run twice on one context, and the
    second run must be identical to the first."""
    vt, jt = w.info.tables()
    ctx = _lib.Context(vt, jt, device=0, both_frames=(w.orientation == "both"), force_general=force_general)
    packed = w.packed()
    try:
        res, cnt = ctx.decombine(packed)
        stats = (ctx.last_deferred(), ctx.last_general())
        res2, cnt2 = ctx.decombine(packed)
        assert np.array_equal(res2, res) and np.array_equal(cnt2, cnt), "%s fg=%d: the second run differs" % (w.key, force_general)
        return res, cnt, stats, ctx.halftag_kernel_name()
    finally:
        ctx.close()
        packed.free()


def _check_oracle(w, res, cnt, want, counts, what):
    assert_records_equal(res, want, w.orientation, "%s %s" % (w.key, what))
    assert np.array_equal(cnt, counts), "%s %s: %s" % (w.key, what, {k: (int(a), int(b)) for k, a, b in zip(O.COUNTER_NAMES, cnt, counts) if a != b})


# ------------------------------------------------------------------------------------------------------------------------
# what the reads are built to be (no GPU)
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(DENSE))
def test_dense_reads_are_what_they_claim(name):
    """The dense reads lack a full tag of their dense gene, more than CAP candidate windows are common in them, and the
    oracle decombines some of them, so that records are compared and not only failure counters."""
    for L in WIDTHS:
        w = dense_workload(name, L)
        assert len(w.ln) == len(w.dense) and (w.ln == L).all()
        gene = DENSE[name][3]
        info = w.info
        g = _Gene(getattr(info, gene + "_seqs"), getattr(info, gene + "_regions"),
                  info.v_half_split if gene == "v" else info.j_half_split)
        reads = [bytes(w.buf[int(o):int(o) + L]).decode() for o in w.off]
        dense = [_revcomp(r) for r, d in zip(reads, w.dense) if d]
        assert len(dense) == BLOCK * (1 + len(MIX))
        # no full tag of the dense gene, except in V-dense reads with a clean real rearrangement behind the decoys
        assert sum(not g.exact(a) for a in dense) > 0.5 * len(dense), (name, L)
        want, _ = w.oracle()
        assert want["ok"][w.dense].sum() > 0.2 * len(dense), (name, L)
        # 13 tags of 20 nt take 260 nt: only the longer reads can hold more than CAP candidates
        if L == 320:
            assert w.n_over > 0.3 * len(dense), (name, L, w.n_over)


# ------------------------------------------------------------------------------------------------------------------------
# (a) the shipped capacities
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("L", WIDTHS)
@pytest.mark.parametrize("name", list(DENSE))
def test_dense_reads_at_shipped_capacities(name, L):
    w = dense_workload(name, L)
    want, counts = w.oracle()
    got = {}
    for fg in (0, 1, 3):
        res, cnt, (deferred, general), half = run(w, fg)
        _check_oracle(w, res, cnt, want, counts, "force_general=%d" % fg)
        if fg == 0:
            assert half == "dcb_halftag_kernel"
            # the construction reached the pass-on paths: every dense read with more than CAP candidates went on (and in
            # the shorter reads, the reads whose probe hits did not fit the warp's list)
            assert general >= w.n_over and general > 0, (deferred, general, w.n_over)
            assert general < deferred, (deferred, general)
        got[fg] = (res, cnt)
    for fg in (1, 3):
        assert np.array_equal(got[fg][0], got[0][0]) and np.array_equal(got[fg][1], got[0][1]), "force_general=%d vs 0" % fg


# ------------------------------------------------------------------------------------------------------------------------
# (b) the capacities shrunk
# ------------------------------------------------------------------------------------------------------------------------
_cache = {}


def _reference(key):
    """(workload, oracle records, oracle counters, shipped library's run), once per session."""
    if key not in _cache:
        w = workload(key)
        _cache[key] = (w,) + w.oracle() + (run(w),)
    return _cache[key]


def _worker(out):
    """Run in a process of its own that loaded a variant library (DCB_LIB): every variant workload, twice each."""
    arrays = {}
    for key in variant_keys():
        res, cnt, stats, half = run(workload(key))
        arrays[key + "_res"], arrays[key + "_cnt"] = res, cnt
        arrays[key + "_stats"] = np.array(stats + (half == "dcb_halftag_kernel",), dtype=np.uint64)
    np.savez(out, **arrays)


@pytest.mark.gpu
@pytest.mark.parametrize("variant", list(build.VARIANTS))
def test_shrunk_capacities(variant, tmp_path):
    path = build.variant_path(variant)
    assert os.path.exists(path), ("%s is missing; build it with `python -m decombinator_b200.build --variants` "
                                  "(__graft_entry__.build() builds it too)" % path)
    out = str(tmp_path / "runs.npz")
    env = dict(os.environ, DCB_LIB=path,
               PYTHONPATH=os.pathsep.join([ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")]
                                          + [p for p in os.environ.get("PYTHONPATH", "").split(os.pathsep) if p]))
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [
        "-c", "import sys, test_gpu_halftag_capacity as t; t._worker(sys.argv[1])", out]
    p = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=1800)
    assert p.returncode == 0, "%s worker failed:\n%s" % (variant, (p.stdout + p.stderr)[-4000:])
    got = np.load(out)
    table = []
    for key in variant_keys():
        w, want, counts, (res0, cnt0, (deferred0, general0), half0) = _reference(key)
        res, cnt, (deferred, general, half) = got[key + "_res"], got[key + "_cnt"], (int(x) for x in got[key + "_stats"])
        _check_oracle(w, res, cnt, want, counts, variant)
        assert np.array_equal(res, res0) and np.array_equal(cnt, cnt0), "%s %s: differs from the shipped library" % (w.key, variant)
        assert deferred == deferred0 and bool(half) == (half0 == "dcb_halftag_kernel"), (w.key, variant)
        if half and deferred:
            table.append((key, deferred, general0, general))
    report = "\n".join("%-14s queued %6d  passed on %6d -> %6d" % row for row in table)
    print(variant + "\n" + report)
    # more reads pass on than with the shipped capacities, yet the kernel still decides some -- except in the 100-nt reads
    # of human alpha (original tags): they hold a J region and hardly any V half keyword, the J scan waits for a V, and
    # not even the shrunk lists fill, so only as many pass on as with the shipped library
    short = "syn%d" % SYNTHETIC_SHAPES.index(("human", "original", "a", "reverse", 100, 0.01, 0.0, 0.0))
    bad = [row for row in table if not (row[2] <= row[3] if row[0] == short else row[2] < row[3]) or not row[3] < row[1]]
    assert not bad, "%s: queued / shipped / variant\n%s" % (variant, report)
