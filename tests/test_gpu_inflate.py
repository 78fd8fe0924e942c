"""gzip input inflated on the GPU (csrc/inflate.cu through _lib.gpu_inflate and fastq.gunzip_file) against the gzip module:
single streams, members, BGZF, an output beyond 4 GiB, thousands of chunks in several segments, perturbed candidate starts,
damaged files (which must reach the host path and raise what they raise there), and decombine end to end on text, one
gzip stream and BGZF."""
import collections
import gzip
import os
import random
import subprocess
import sys
import zlib

import numpy as np
import pytest

from decombinator_b200 import _lib, fastq

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
from test_fastq_native import _bgzf  # noqa: E402


def _pairs(n, seed=20261022):
    from decombinator_b200 import tags
    info = tags.load("human", "extended", "b")
    syn = _lib.Synth([(info.v_regions, info.j_regions)], seed, 250, 62, 0.01, 0.001, 0.05)
    r1, r2 = syn.reads(0, n, want_r2=True)
    rng = np.random.default_rng(seed)
    q1 = rng.choice(np.frombuffer(b"#,:FFFF", np.uint8), size=(n, 250))
    a1, a2 = r1.reshape(n, 250), r2.reshape(n, 62)
    t1 = b"".join(b"@SYN:%d 1:N:0\n%s\n+\n%s\n" % (i, a1[i].tobytes(), q1[i].tobytes()) for i in range(n))
    t2 = b"".join(b"@SYN:%d 2:N:0\n%s\n+\n%s\n" % (i, a2[i].tobytes(), b"I" * 62) for i in range(n))
    return t1, t2


_text = None


def text():
    global _text
    if _text is None:
        _text = _pairs(40000)[0]
    return _text


def gpu(blob, **kw):
    return bytes(_lib.gpu_inflate(blob, **kw))


@pytest.mark.parametrize("level", [1, 6, 9])
def test_single_stream(level):
    blob = gzip.compress(text(), level)
    assert gpu(blob) == text()
    assert gpu(blob, chunk_bytes=16384, segment_bytes=65536) == text()


def test_members_padding_and_empty_members():
    t = text()
    blob = b"".join(gzip.compress(t[lo:lo + 700000], 6) for lo in range(0, len(t), 700000))
    blob = gzip.compress(b"") + blob + gzip.compress(b"") + gzip.compress(t[:100], 9) + b"\0" * 300
    want = gzip.decompress(blob)
    assert gpu(blob) == want
    assert gpu(blob, chunk_bytes=4096, segment_bytes=8192) == want
    assert gpu(gzip.compress(b"")) == b""


def test_bgzf_members():
    blob = _bgzf(text())
    blocks = fastq._bgzf_blocks(blob)
    assert gpu(blob, members=blocks) == text()
    assert gpu(blob, members=blocks, segment_bytes=100000) == text()


def test_thousands_of_chunks_in_several_segments():
    """Small blocks (memLevel 1: a block every 128 symbols) and 1 KiB chunks: thousands of candidates, 8 segments."""
    t = text()[:6_000_000]
    c = zlib.compressobj(6, zlib.DEFLATED, 31, 1)
    blob = c.compress(t) + c.flush()
    L = _lib.lib()
    import ctypes
    src = np.frombuffer(blob, np.uint8)
    h = ctypes.c_void_p()
    assert L.dcb_inflate_create(0, src.ctypes.data, len(src), 1024, 0, ctypes.byref(h)) == 0
    n = ctypes.c_uint64()
    assert L.dcb_inflate_find_starts(h, None, 0, ctypes.byref(n)) == 0
    starts = np.zeros(n.value, np.uint64)
    assert L.dcb_inflate_find_starts(h, starts.ctypes.data, n.value, ctypes.byref(n)) == 0
    L.dcb_inflate_destroy(h)
    assert int((starts != _lib.NO_START).sum()) > 1000
    assert gpu(blob, chunk_bytes=1024, segment_bytes=len(blob) // 8) == t


@pytest.mark.parametrize("seed", range(3))
def test_perturbed_starts(seed):
    """Candidate lists with false starts (off by a bit, random offsets), with true ones dropped: the output stays the same."""
    rng = random.Random(seed)
    blob = gzip.compress(text(), 6)
    nbits = 8 * len(blob)

    def hook(starts):
        s = [int(x) for x in starts[1:] if int(x) != _lib.NO_START]
        s = [x for x in s if rng.random() < 0.7]
        s += [x + rng.choice((-1, 1, 3)) for x in s if rng.random() < 0.3]
        s += rng.sample(range(int(starts[0]) + 1, nbits - 1), 200)
        return np.array([int(starts[0])] + sorted(set(x for x in s if int(starts[0]) < x < nbits)), dtype=np.uint64)
    assert gpu(blob, chunk_bytes=8192, segment_bytes=65536, starts_hook=hook) == text()


def test_bit_limit_on_fixed_blocks_goes_to_the_host():
    """Z_FIXED: the finder finds no dynamic header, chunk 0 reaches its bit limit; gunzip_file still returns the text."""
    c = zlib.compressobj(6, zlib.DEFLATED, 31, 8, zlib.Z_FIXED)
    blob = c.compress(text() * 2) + c.flush()
    assert len(blob) > 5 << 20
    with pytest.raises(_lib.DcbError) as e:
        gpu(blob, chunk_bytes=4096)
    assert e.value.rc == -5


def test_output_past_4_gib():
    """Runs compress about 1000:1: a 4.3 GB stream from a few MB; ISIZE wraps, the caller's buffer grows."""
    rng = random.Random(1)
    unit = b"".join(bytes([rng.randrange(256)]) * rng.randrange(50000, 150000) for _ in range(256))
    reps = (2 ** 32 + 10_000_000) // len(unit) + 1
    c = zlib.compressobj(6, zlib.DEFLATED, 31)
    parts, crc = [], 0
    for _ in range(reps):
        parts.append(c.compress(unit))
        crc = zlib.crc32(unit, crc)
    parts.append(c.flush())
    blob = b"".join(parts)
    out = _lib.gpu_inflate(blob)
    assert len(out) == reps * len(unit) > 2 ** 32
    assert zlib.crc32(out) == crc
    assert out[len(out) - len(unit):] == unit and out[:len(unit)] == unit


def _host_error(path):
    try:
        fastq._file_bytes(str(path), gzip.open)
    except Exception as e:          # noqa: BLE001
        return type(e)
    return None


def test_damaged_files_take_the_host_path(tmp_path):
    blob = gzip.compress(text()[:3_000_000], 6)
    cases = {}
    bad = bytearray(blob)
    bad[len(blob) // 2] ^= 0x10
    cases["flip"] = bytes(bad)
    cases["cut"] = blob[:-1000]
    cases["trailer"] = blob[:-8] + (zlib.crc32(b"x")).to_bytes(4, "little") + blob[-4:]
    cases["isize"] = blob[:-4] + b"\0\0\0\0"
    cases["garbage"] = blob + b"not gzip"
    for name, b in cases.items():
        with pytest.raises(_lib.DcbError) as e:
            gpu(b)
        assert e.value.rc == -5, name
        path = tmp_path / (name + ".gz")
        path.write_bytes(b)
        want = None
        try:
            with gzip.open(path, "rb") as fh:
                fh.read()
        except Exception as err:     # noqa: BLE001
            want = type(err)
        assert want is not None, name
        assert _host_error(path) is want, name
    bgzf = bytearray(_bgzf(text()[:500000]))
    bgzf[3000] ^= 0x55
    with pytest.raises(_lib.DcbError):
        gpu(bytes(bgzf), members=fastq._bgzf_blocks(bytes(bgzf)))


def test_gunzip_file_routes_to_the_device(tmp_path, monkeypatch):
    path = tmp_path / "x.fq.gz"
    path.write_bytes(gzip.compress(text(), 6))
    calls = []
    real = _lib.gpu_inflate
    monkeypatch.setattr(_lib, "gpu_inflate", lambda *a, **k: calls.append(1) or real(*a, **k))
    assert bytes(fastq.gunzip_file(str(path))) == text()
    assert calls


def test_decombine_same_from_text_gzip_and_bgzf(tmp_path):
    from decombinator_b200 import decombine, io
    t1, t2 = _pairs(30000, seed=77)
    rows, counts, n12 = {}, {}, {}
    for kind in ("text", "gzip", "bgzf"):
        d = tmp_path / kind
        d.mkdir()
        for name, t in (("S_1.fq", t1), ("S_2.fq", t2)):
            if kind == "text":
                (d / name).write_bytes(t)
            else:
                (d / (name + ".gz")).write_bytes(gzip.compress(t, 6) if kind == "gzip" else _bgzf(t))
        infile = str(d / ("S_1.fq" + ("" if kind == "text" else ".gz")))
        ia = io.create_args_dict(infile=infile, chain="b", bc_read="R2", suppresssummary=True, dontcheck=True, dontcount=True, outpath=str(d) + "/",
                                 dontgzip=True)
        decombine.counts = collections.Counter()
        rows[kind] = [list(r) for r in decombine.decombinator(dict(ia))]
        counts[kind] = {k: v for k, v in decombine.counts.items() if not k.endswith("_time")}
        subprocess.run([sys.executable, "-m", "decombinator_b200", "decombine", "-in", infile, "-br", "R2", "-c", "b", "-dz", "-s", "-dk", "-dc",
                        "-op", str(d) + "/"], check=True, cwd=ROOT, capture_output=True)
        n12[kind] = (d / "dcr_S_1_beta.n12").read_bytes()
    assert len(rows["text"]) > 1000
    assert rows["gzip"] == rows["text"] and rows["bgzf"] == rows["text"]
    assert counts["gzip"] == counts["text"] and counts["bgzf"] == counts["text"]
    assert n12["gzip"] == n12["text"] and n12["bgzf"] == n12["text"]
