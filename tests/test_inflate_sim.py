"""csrc/inflate_core.cuh compiled for the host (tests/sim/sim_inflate.cpp) against zlib: whole streams at every level,
strategy and window size, the start finder's header test on every true block boundary, marker-mode decodes resolved
with the true window, the chaining rule over candidate lists with false starts, CRC-32 arithmetic, and (a second build
with AddressSanitizer) every truncation and single-byte change of a small stream ending in a status.  CPU only."""
import ctypes
import gzip
import os
import random
import subprocess
import zlib

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "sim", "sim_inflate.cpp")
CORE = os.path.join(ROOT, "decombinator_b200", "csrc", "inflate_core.cuh")
SO = os.path.join(ROOT, "tests", "sim", "libinflatesim.so")
ASAN = os.path.join(ROOT, "tests", "sim", "inflate_asan")

INF_END, INF_LANDED, INF_LIMIT = 0, 1, 2
u64p = ctypes.c_void_p

_sim = None


def _stale(out):
    return not os.path.exists(out) or any(os.path.getmtime(d) > os.path.getmtime(out) for d in (SRC, CORE))


def sim():
    global _sim
    if _sim is None:
        if _stale(SO):
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", SRC, "-o", SO])
        L = ctypes.CDLL(SO)
        L.sim_inflate.argtypes = [u64p, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_uint64, u64p, ctypes.c_uint32, ctypes.c_int,
                                  ctypes.c_int, u64p, ctypes.c_uint64, u64p, u64p, u64p, ctypes.c_uint32, u64p, ctypes.c_uint32, u64p]
        L.sim_dyn_ok.argtypes = [u64p, ctypes.c_uint64, ctypes.c_uint64]
        L.sim_find_all.argtypes = [u64p, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_uint64, u64p, ctypes.c_uint64]
        L.sim_find_all.restype = ctypes.c_uint64
        L.sim_resolve.argtypes = [u64p, ctypes.c_uint64, u64p, u64p]
        L.sim_chain.argtypes = [u64p, u64p, ctypes.c_uint32, u64p, ctypes.POINTER(ctypes.c_int)]
        L.sim_chain.restype = ctypes.c_uint32
        L.sim_crc32.argtypes = [ctypes.c_char_p, ctypes.c_uint64]
        L.sim_crc32.restype = ctypes.c_uint32
        L.sim_crc_combine.argtypes = [ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint64]
        L.sim_crc_combine.restype = ctypes.c_uint32
        _sim = L
    return _sim


def header_end(blob):
    """Bit offset of the first block of the gzip member at the start of blob (names, comments and extras skipped)."""
    flg, p = blob[3], 10
    if flg & 4:
        p += 2 + int.from_bytes(blob[10:12], "little")
    for bit in (8, 16):
        if flg & bit:
            p = blob.index(b"\0", p) + 1
    if flg & 2:
        p += 2
    return 8 * p


def inflate(blob, start, cap, marker=False, gzip_=True, cand=(), limit=2 ** 64 - 1, blocks_cap=0, mend_cap=64):
    """-> (status, landed, produced, end_bit, out array, member ends [(pos, crc, isize)], block headers [(bit, type)])"""
    src = np.frombuffer(blob, dtype=np.uint8)
    out = np.zeros(max(cap, 1), dtype=np.uint16 if marker else np.uint8)
    cand = np.array(sorted(cand), dtype=np.uint64)
    mp, mc, mi = np.zeros(mend_cap + 1, np.uint64), np.zeros(mend_cap + 1, np.uint32), np.zeros(mend_cap + 1, np.uint32)
    blocks = np.zeros(blocks_cap + 1, np.uint64)
    res = np.zeros(6, np.uint64)
    sim().sim_inflate(src.ctypes.data, len(src), start, limit, cand.ctypes.data, len(cand), int(gzip_), int(marker), out.ctypes.data, cap,
                      mp.ctypes.data, mc.ctypes.data, mi.ctypes.data, mend_cap, blocks.ctypes.data, blocks_cap, res.ctypes.data)
    status = int(np.int64(res[0]))
    nm, nb = int(res[4]), min(int(res[5]), blocks_cap)
    return (status, int(res[1]), int(res[2]), int(res[3]), out[:min(cap, int(res[2]))],
            [(int(mp[i]), int(mc[i]), int(mi[i])) for i in range(nm)], [(int(b) >> 2, int(b) & 3) for b in blocks[:nb]])


def compress(data, level=6, strategy=zlib.Z_DEFAULT_STRATEGY, wbits=15, flushes=()):
    c = zlib.compressobj(level, zlib.DEFLATED, 16 + wbits, 8, strategy)
    out, at = [], 0
    for pos, mode in flushes:
        out.append(c.compress(data[at:pos]))
        out.append(c.flush(mode))
        at = pos
    out.append(c.compress(data[at:]))
    out.append(c.flush())
    return b"".join(out)


_fastq = None


def fastq_text(n_reads=1500):
    global _fastq
    if _fastq is None:
        from decombinator_b200 import _lib, tags
        info = tags.load("human", "extended", "b")
        syn = _lib.Synth([(info.v_regions, info.j_regions)], 20261022, 250, 62, 0.01, 0.001, 0.02)
        r1, _ = syn.reads(0, n_reads, want_r2=False)
        rng = random.Random(5)
        a = r1.reshape(n_reads, 250)
        _fastq = b"".join(b"@SYN:%d 1:N:0\n%s\n+\n%s\n" % (i, a[i].tobytes(), bytes(rng.choice(b"#,:FFFF") for _ in range(250)))
                          for i in range(n_reads))
    return _fastq


def runs_text():
    """Long runs: matches of length 258 at distance 1 and at distance 32768, overlapping copies."""
    rng = random.Random(9)
    block = bytes(rng.randrange(256) for _ in range(32768))
    return b"A" * 70000 + block + block + b"xy" * 5000 + block[:1000] * 3


def random_bytes(n=120000):
    return np.random.default_rng(4).integers(0, 256, n, dtype=np.uint8).tobytes()


def true_blocks(blob):
    """Every block header of a stream decoded from its start: [(bit offset, BTYPE, output offset)]."""
    start = header_end(blob)
    st, _, produced, _, out, mends, blocks = inflate(blob, start, len(gzip.decompress(blob)) + 1, blocks_cap=100000)
    assert st == INF_END
    # output offset of each block: decode again, stopping at every block header in turn
    heads = [b for b, t in blocks]
    offs = []
    for b in heads:
        if b == start:
            offs.append(0)
            continue
        st2, _, p2, _, _, _, _ = inflate(blob, start, 0, cand=[b])
        assert st2 == INF_LANDED
        offs.append(p2)
    return [(b, t, o) for (b, t), o in zip(blocks, offs)]


LEVEL_CASES = [(lv, zlib.Z_DEFAULT_STRATEGY, 15) for lv in range(10)] + \
    [(6, s, 15) for s in (zlib.Z_FILTERED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE, zlib.Z_FIXED)] + \
    [(9, zlib.Z_DEFAULT_STRATEGY, w) for w in range(9, 15)] + [(1, zlib.Z_FILTERED, 9), (9, zlib.Z_RLE, 12)]


@pytest.mark.parametrize("level,strategy,wbits", LEVEL_CASES)
@pytest.mark.parametrize("kind", ["fastq", "random", "runs"])
def test_whole_stream_equals_zlib(kind, level, strategy, wbits):
    data = {"fastq": fastq_text, "random": random_bytes, "runs": runs_text}[kind]()
    blob = compress(data, level, strategy, wbits)
    st, _, produced, end_bit, out, mends, _ = inflate(blob, header_end(blob), len(data) + 7)
    assert st == INF_END and produced == len(data) and bytes(out) == data
    assert mends == [(len(data), zlib.crc32(data), len(data))]
    assert end_bit == 8 * len(blob)
    # a buffer too small: the exact size is still reported (counting continuation), the part written is right
    st, _, produced, _, out, _, _ = inflate(blob, header_end(blob), len(data) // 3)
    assert st == INF_END and produced == len(data) and bytes(out) == data[:len(data) // 3]


@pytest.mark.parametrize("mode", [zlib.Z_SYNC_FLUSH, zlib.Z_FULL_FLUSH])
def test_flush_points_and_members(mode):
    data = fastq_text()
    cuts = [(p, mode) for p in range(10000, len(data), 37000)]
    parts = [compress(data, 6, flushes=cuts), gzip.compress(b""), gzip.compress(data[:5000], 9), b"\0" * 64]
    blob = b"".join(parts)
    want = gzip.decompress(blob)
    st, _, produced, _, out, mends, _ = inflate(blob, header_end(blob), len(want))
    assert st == INF_END and bytes(out) == want
    assert [m[0] for m in mends] == [len(data), len(data), len(data) + 5000]
    assert [m[1] for m in mends] == [zlib.crc32(data), 0, zlib.crc32(data[:5000])]
    # a member header with every optional field
    named = b"\x1f\x8b\x08\x1e\0\0\0\0\0\xff" + b"\x03\x00abc" + b"name\0" + b"comment\0" + b"\xaa\xbb"
    body = zlib.compressobj(6, zlib.DEFLATED, -15)
    named += body.compress(data[:3000]) + body.flush() + zlib.crc32(data[:3000]).to_bytes(4, "little") + (3000).to_bytes(4, "little")
    st, _, _, _, out, mends, _ = inflate(named + blob, header_end(named), len(want) + 3000)
    assert st == INF_END and bytes(out) == data[:3000] + want and len(mends) == 4
    # a raw deflate stream stops at its final block
    st, _, produced, _, out, mends, _ = inflate(body_raw := zlib.compress(data[:9000])[2:-4], 0, 9000, gzip_=False)
    assert st == INF_END and bytes(out) == data[:9000] and mends == [] and body_raw


@pytest.mark.parametrize("level,strategy", [(1, zlib.Z_DEFAULT_STRATEGY), (6, zlib.Z_DEFAULT_STRATEGY), (9, zlib.Z_DEFAULT_STRATEGY),
                                            (6, zlib.Z_FILTERED), (6, zlib.Z_HUFFMAN_ONLY), (6, zlib.Z_RLE)])
@pytest.mark.parametrize("kind", ["fastq", "runs"])
def test_marker_mode_from_every_true_boundary(kind, level, strategy):
    data = (fastq_text() + runs_text()) if kind == "runs" else fastq_text() * 3
    blob = compress(data, level, strategy, flushes=[(len(data) // 2, zlib.Z_SYNC_FLUSH)])
    blocks = true_blocks(blob)
    dynamic = [b for b, t, _ in blocks if t == 2]
    assert len(dynamic) >= 3
    src = np.frombuffer(blob, dtype=np.uint8)
    for b in dynamic:
        assert sim().sim_dyn_ok(src.ctypes.data, len(src), b) == 1
    heads = [b for b, _, _ in blocks]
    for i, (b, t, off) in enumerate(blocks):
        if t != 2:
            continue
        st, landed, produced, end_bit, sym, _, _ = inflate(blob, b, len(data), marker=True, cand=heads)
        nxt = blocks[i + 1][2] if i + 1 < len(blocks) else len(data)
        if i + 1 < len(blocks):
            assert st == INF_LANDED and landed == i + 1 and end_bit == heads[i + 1]
        else:
            assert st == INF_END
        assert produced == nxt - off
        window = np.zeros(32768, np.uint8)
        w = np.frombuffer(data[max(0, off - 32768):off], np.uint8)
        window[32768 - len(w):] = w
        got = np.zeros(produced, np.uint8)
        sim().sim_resolve(sym.ctypes.data, produced, window.ctypes.data, got.ctypes.data)
        assert got.tobytes() == data[off:nxt]


@pytest.mark.parametrize("seed", range(4))
def test_chain_keeps_exactly_the_true_starts(seed):
    rng = random.Random(seed)
    data = fastq_text() * 4
    blob = compress(data, rng.choice([1, 6, 9]))
    blocks = true_blocks(blob)
    start = header_end(blob)
    true_dyn = [b for b, t, _ in blocks if t == 2 and b != start]
    src = np.frombuffer(blob, dtype=np.uint8)
    # false starts: offsets that pass the validator without being block headers where there are any, else random bits
    found = np.zeros(256, np.uint64)
    nf = sim().sim_find_all(src.ctypes.data, len(src), start + 1, 8 * len(blob), found.ctypes.data, 256)
    false = [int(x) for x in found[:min(nf, 256)] if int(x) not in set(b for b, _, _ in blocks)]
    false += rng.sample(range(start + 1, 8 * len(blob) - 64), 12)
    keep_true = rng.sample(true_dyn, max(1, len(true_dyn) * 2 // 3))
    cand = sorted(set([start] + keep_true + false))
    n = len(cand)
    status, landed = np.zeros(n, np.int32), np.zeros(n, np.uint32)
    outs = []
    for k, c in enumerate(cand):
        st, ld, produced, _, sym, _, _ = inflate(blob, c, 2 * len(data), marker=True, cand=cand, limit=c + 8 * len(blob))
        status[k], landed[k] = st, ld
        outs.append(sym)
    chain = np.zeros(n, np.uint32)
    bad = ctypes.c_int()
    m = sim().sim_chain(status.ctypes.data, landed.ctypes.data, n, chain.ctypes.data, ctypes.byref(bad))
    assert m > 0 and bad.value == 0
    kept = [cand[i] for i in chain[:m]]
    assert kept == sorted([start] + keep_true)
    # the kept chunks, resolved in chain order, are the stream
    text = bytearray()
    for i in chain[:m]:
        window = np.zeros(32768, np.uint8)
        w = np.frombuffer(bytes(text[-32768:]), np.uint8)
        window[32768 - len(w):] = w
        got = np.zeros(len(outs[i]), np.uint8)
        sim().sim_resolve(outs[i].ctypes.data, len(outs[i]), window.ctypes.data, got.ctypes.data)
        text += got.tobytes()
    assert bytes(text) == data


def test_chain_rule_by_table():
    def chain(status, landed):
        n = len(status)
        st, ld = np.array(status, np.int32), np.array(landed, np.uint32)
        out = np.zeros(n, np.uint32)
        bad = ctypes.c_int()
        m = sim().sim_chain(st.ctypes.data, ld.ctypes.data, n, out.ctypes.data, ctypes.byref(bad))
        return list(out[:m]), bad.value
    assert chain([INF_LANDED, INF_LANDED, INF_END, INF_END], [2, 3, 0, 0]) == ([0, 2], 0)
    assert chain([INF_LANDED, -1, INF_LANDED, INF_END], [2, 0, 3, 0]) == ([0, 2, 3], 0)     # a broken chunk off the chain
    assert chain([INF_LANDED, INF_END, INF_LIMIT], [2, 0, 0]) == ([], INF_LIMIT)            # a chain chunk at its bit limit
    assert chain([INF_END], [0]) == ([0], 0)


def test_crc_arithmetic():
    rng = np.random.default_rng(1)
    for n in (0, 1, 7, 4096, 100003):
        a = rng.integers(0, 256, n, dtype=np.uint8).tobytes()
        b = rng.integers(0, 256, 12345, dtype=np.uint8).tobytes()
        assert sim().sim_crc32(a, len(a)) == zlib.crc32(a)
        assert sim().sim_crc_combine(zlib.crc32(a), zlib.crc32(b), len(b)) == zlib.crc32(a + b)
        assert sim().sim_crc_combine(zlib.crc32(b), zlib.crc32(a), len(a)) == zlib.crc32(b + a)


def test_bad_input_ends_in_a_status():
    data = fastq_text()[:2500]
    blob = compress(data, 6)
    for cut in range(1, len(blob)):
        st = inflate(blob[:cut], header_end(blob), len(data))[0]
        assert st < 0, cut
    bad = bytearray(blob)
    bad[-8] ^= 1                                     # the trailer is the caller's to check: same bytes, other CRC
    st, _, _, _, out, mends, _ = inflate(bytes(bad), header_end(blob), len(data))
    assert st == INF_END and bytes(out) == data and mends[0][1] != zlib.crc32(data)
    stored = bytearray(compress(data, 0))
    stored[header_end(stored) // 8 + 3] ^= 0xff       # NLEN of the first stored block
    assert inflate(bytes(stored), header_end(stored), len(data))[0] == -4
    assert inflate(b"\x1f\x8b\x08\0\0\0\0\0\0\xff\x07", 80, 10)[0] == -5          # BTYPE 11


def test_every_truncation_and_byte_change_under_the_sanitizer(tmp_path):
    if _stale(ASAN):
        subprocess.check_call(["g++", "-O1", "-g", "-std=c++17", "-fsanitize=address,undefined", "-fno-sanitize-recover=all",
                               "-DSIM_MAIN", "-x", "c++", SRC, "-o", ASAN])
    data = fastq_text()[:700] + b"A" * 300
    for blob in (compress(data, 6), compress(data, 0), compress(data, 9, zlib.Z_FIXED)):
        path = tmp_path / "small.gz"
        path.write_bytes(blob)
        env = dict(os.environ, ASAN_OPTIONS="detect_leaks=0:abort_on_error=0", UBSAN_OPTIONS="halt_on_error=1")
        res = subprocess.run([ASAN, str(path), "600"], capture_output=True, text=True, env=env, timeout=600)
        assert res.returncode == 0, res.stderr[-3000:]
        counts = dict(tuple(map(int, line.split())) for line in res.stdout.strip().splitlines())
        assert sum(counts.values()) >= 256 * len(blob)
