"""Device-side packing (csrc/pack_device.cuh) against the host packer dcb_pack_reads: bit-identical slot words, lengths,
flag words and exception list (decombine.py:182-184 revcomp through Bio.Seq's table, :965-977 slicing), and
dcb_decombine_ascii against dcb_decombine_batch on the host-packed batch.  GPU, through the C ABI."""
import numpy as np
import pytest

from decombinator_b200 import _lib, tags
from helpers import synth_batch

pytestmark = pytest.mark.gpu


def _ctx(info=None, **kw):
    info = info or tags.load("human", "extended", "b")
    vt, jt = info.tables()
    return _lib.Context(vt, jt, device=0, **kw)


def _same(a: "_lib.Packed", b: "_lib.Packed", what):
    assert (a.n_reads, a.slot_words, a.n_exc, a.uniform_len, a.max_len) == (b.n_reads, b.slot_words, b.n_exc, b.uniform_len, b.max_len), what
    xa, xb = a.arrays(), b.arrays()
    for k in xa:
        assert np.array_equal(xa[k], xb[k]), "%s: %s differs at %s" % (what, k, np.nonzero(xa[k] != xb[k])[0][:8])


def _concat(reads):
    bufs = [r.encode("latin-1") for r in reads]
    length = np.array([len(b) for b in bufs], dtype=np.uint32)
    off = np.zeros(len(bufs), dtype=np.uint64)
    if len(bufs) > 1:
        off[1:] = np.cumsum(length[:-1], dtype=np.uint64)
    return np.frombuffer(b"".join(bufs) + b"\0" * 8, dtype=np.uint8).copy(), off, length


SYMBOLS = "ACGTNacgtnUuRYKMSWBDHVrykm-.*X"


def _fuzzed_reads(n, seed, max_len=330):
    """Ragged reads over ACGT with sprinkled N / IUPAC / lower-case / U / junk symbols, empty and one-base reads included."""
    rng = np.random.default_rng(seed)
    reads = []
    for i in range(n):
        L = int(rng.integers(0, max_len + 1)) if i % 7 else int(rng.choice([0, 1, 7, 8, 9, 15, 16, 17, 63, 64, 65, 255, 256, 257, max_len]))
        s = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, L)].copy()
        if i % 3 == 0 and L:
            k = int(rng.integers(1, 6))
            pos = rng.integers(0, L, k)
            s[pos] = np.frombuffer(SYMBOLS.encode(), dtype=np.uint8)[rng.integers(0, len(SYMBOLS), k)]
        if i % 41 == 0:
            s[:] = ord("N")
        reads.append(s.tobytes().decode("latin-1"))
    return reads


@pytest.mark.parametrize("revcomp", [True, False])
def test_device_pack_equals_host_pack_ragged(revcomp):
    ctx = _ctx()
    for n, seed, max_len in ((1, 1, 40), (31, 2, 100), (33, 3, 330), (5000, 4, 330), (3000, 5, 1000), (70, 6, 4000)):
        reads = _fuzzed_reads(n, seed, max_len)
        buf, off, length = _concat(reads)
        host = _lib.pack_arrays(buf, off, length, revcomp)
        dev = ctx.pack_device(buf, off, length, revcomp)
        _same(dev, host, "ragged n=%d revcomp=%s" % (n, revcomp))
        for i in (0, n // 2, n - 1):
            assert dev.unpack(i) == host.unpack(i)
        host.free(); dev.free()
    ctx.close()


def test_device_pack_equals_host_pack_uniform_chunks():
    """3.3 M uniform reads (four chunks on two streams: the exception list continues across chunks), contiguous layout."""
    info = tags.load("human", "extended", "b")
    n, L = 3_300_000, 250
    r1, off, ln = synth_batch(info, n, L, 0.01, 0.002, 0.02, seed=9)
    r1[np.arange(0, n * L, 997)] = ord("n")          # lower case: kind 2
    r1[np.arange(5, n * L, 4999)] = ord("U")         # kind 3 on the reverse strand
    ctx = _ctx(info)
    for revcomp in (True, False):
        host = _lib.pack_arrays(r1, off, ln, revcomp)
        dev = ctx.pack_device(r1, None, None, revcomp, uniform_len=L)
        _same(dev, host, "uniform contiguous revcomp=%s" % revcomp)
        dev2 = ctx.pack_device(r1, off, ln, revcomp)
        _same(dev2, host, "uniform with offsets revcomp=%s" % revcomp)
        host.free(); dev.free(); dev2.free()
    ctx.close()


@pytest.mark.parametrize("chain,both", [("b", False), ("a", False), ("b", True)])
def test_decombine_ascii_equals_decombine_batch(chain, both):
    info = tags.load("human", "extended", chain)
    n, L = 2_200_000, 250
    r1, off, ln = synth_batch(info, n, L, 0.01, 0.001, 0.05, seed=20260003)
    ctx = _ctx(info, both_frames=both)
    packed = _lib.pack_arrays(r1, off, ln, True)
    want, wcnt = ctx.decombine(packed)
    got, cnt = ctx.decombine_ascii(r1, None, None, True, uniform_len=L)
    assert np.array_equal(got, want) and np.array_equal(cnt, wcnt)
    got2, cnt2 = ctx.decombine_ascii(r1, off, ln, True)
    assert np.array_equal(got2, want) and np.array_equal(cnt2, wcnt)
    packed.free(); ctx.close()


def test_decombine_ascii_ragged_and_empty():
    info = tags.load("human", "extended", "b")
    r1, off, ln = synth_batch(info, 4000, 250, 0.01, 0.001, 0.05, seed=5)
    reads = [bytes(r1[i * 250:(i + 1) * 250]).decode() for i in range(4000)]
    rng = np.random.default_rng(1)
    ragged = [r[sorted(rng.integers(0, 251, size=2))[0]:] if i % 3 else r for i, r in enumerate(reads)] + ["", "A", "N" * 250, "acgt" * 30]
    buf, off, length = _concat(ragged)
    for kw in ({}, {"both_frames": True}, {"allow_ns": True}):
        ctx = _ctx(info, **kw)
        packed = _lib.pack_arrays(buf, off, length, True)
        want, wcnt = ctx.decombine(packed)
        got, cnt = ctx.decombine_ascii(buf, off, length, True)
        assert np.array_equal(got, want) and np.array_equal(cnt, wcnt), kw
        packed.free(); ctx.close()
    ctx = _ctx(info)
    got, cnt = ctx.decombine_ascii(np.zeros(8, dtype=np.uint8), np.zeros(0, dtype=np.uint64), np.zeros(0, dtype=np.uint32), True)
    assert len(got) == 0 and not cnt.any()
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("share", ["0", "1"])
def test_decombine_ascii_host_share_changes_nothing(share, monkeypatch):
    """dcb_decombine_ascii shares the chunks of clean reads between the device packer and the host threads
    (DCB_HOST_SHARE: 0 the device packs every chunk; 1, the default, page-locked text shared from both ends and pageable
    text packed by the host threads): the records and counters are those of the host-packed batch whichever packs; a
    chunk with another symbol goes back to the device."""
    monkeypatch.setenv("DCB_HOST_SHARE", share)
    info = tags.load("human", "extended", "b")
    vt, jt = info.tables()
    ctx = _lib.Context(vt, jt, device=0)
    n, L = 2_300_000, 250                                   # three chunks of the page-locked path
    syn = _lib.Synth([(info.v_regions, info.j_regions)], 20260007, L, 0, 0.0, 0.0, 0.0)
    r1, _ = syn.reads(0, n)
    off = np.arange(n, dtype=np.uint64) * L
    ln = np.full(n, L, dtype=np.uint32)
    packed = _lib.pack_arrays(r1, off, ln, revcomp=True)
    want, wcnt = ctx.decombine(packed)
    packed.free()
    text = _lib.PinnedBytes(r1)
    for buf in (text.a, r1):                                # page-locked and pageable text
        got, cnt = ctx.decombine_ascii(buf, None, None, True, uniform_len=L)
        assert np.array_equal(got, want) and np.array_equal(cnt, wcnt)
        host, dev = ctx.last_pack_shares()
        assert host + dev >= 3
        if share == "0":
            assert host == 0
    text.free()
    # ragged reads, and an N in the second chunk: from there on the device packs
    r2, off2, ln2 = synth_batch(info, 1_200_000, 250, 0.0, 0.0, 0.0, seed=5)
    r2 = r2.copy()
    r2[int(off2[1_100_000]) + 17] = ord("N")
    packed = _lib.pack_arrays(r2, off2, ln2, revcomp=True)
    want, wcnt = ctx.decombine(packed)
    packed.free()
    got, cnt = ctx.decombine_ascii(r2, off2, ln2, True)
    assert np.array_equal(got, want) and np.array_equal(cnt, wcnt)
    ctx.close()


def test_decombine_ascii_host_share_rejects_other_values(monkeypatch):
    """DCB_HOST_SHARE takes 0 or 1: any other value fails the call instead of running one of those schemes unannounced."""
    monkeypatch.setenv("DCB_HOST_SHARE", "2")
    ctx = _ctx()
    with pytest.raises(_lib.DcbError, match="DCB_HOST_SHARE"):
        ctx.decombine_ascii(np.frombuffer(b"ACGT" * 64, dtype=np.uint8).copy(), None, None, True, uniform_len=256)
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("stage_mb", ["1024", "1"])
def test_decombine_ascii_two_ended_sharing(stage_mb, monkeypatch):
    """Page-locked text, one rank per host: the device takes chunks from the front while a worker packs chunks from the back
    (ascii_two_ended).  Small chunks so that a modest batch has many of them; uniform and ragged reads; a batch whose
    front half is full of Ns (device chunks with exception lists, clean host chunks behind them: the exception index must
    run on); an N near the end (the worker gives that chunk back and stops); a page-locked region that holds two chunks."""
    monkeypatch.setenv("DCB_HOST_SHARE", "1")
    monkeypatch.setenv("DCB_CHUNK_READS", "8192")
    monkeypatch.setenv("DCB_HOST_STAGE_MB", stage_mb)
    info = tags.load("human", "extended", "b")
    ctx = _ctx(info)
    L = 250

    def check(buf, off, ln, uniform):
        packed = _lib.pack_arrays(buf, off, ln, revcomp=True)
        want, wcnt = ctx.decombine(packed)
        packed.free()
        text = _lib.PinnedBytes(buf)
        for _ in range(2):
            if uniform:
                got, cnt = ctx.decombine_ascii(text.a, None, None, True, uniform_len=L)
            else:
                got, cnt = ctx.decombine_ascii(text.a, off, ln, True)
            assert np.array_equal(got, want) and np.array_equal(cnt, wcnt)
        shares = ctx.last_pack_shares()
        text.free()
        return shares

    n = 300_000
    clean, off, ln = synth_batch(info, n, L, 0.01, 0.0, 0.05, seed=11)
    host, dev = check(clean, off, ln, True)
    assert host + dev == (n + 8191) // 8192 and host >= 1 and dev >= 1
    if stage_mb == "1":
        assert host <= 2
    # Ns in the front half only
    dirty, _, _ = synth_batch(info, n, L, 0.01, 0.002, 0.05, seed=12)
    mixed = np.concatenate([dirty[:n // 2 * L], clean[n // 2 * L:]])
    host, dev = check(mixed, off, ln, True)
    assert dev >= n // 2 // 8192
    # one N in the third chunk from the end
    late = clean.copy()
    late[(n - 20_000) * L + 5] = ord("N")
    check(late, off, ln, True)
    # ragged reads
    rng = np.random.default_rng(3)
    ln2 = rng.integers(0, L + 1, size=n).astype(np.uint32)
    ln2[::7] = L
    check(clean, off, ln2, False)
    ctx.close()
