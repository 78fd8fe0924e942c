#!/usr/bin/env python
"""Inflate rate of gzip FASTQ on the GPU (dcb_inflate_*) and on the host (the paths fastq.gunzip_file takes without a
device), on the same files, alternated, outputs compared byte for byte (GPU box only).

    python tools/bench_inflate.py [--reads 10000000] [--reps 2] [--chunks 65536,262144,1048576]

R1 of the configs[1] recipe (the synthetic reads of tools/e2e_fastq.py: 250 nt, quality strings as a sequencer writes
them) is compressed twice: one gzip stream at level 6, and BGZF (64 KB members, level 6).  Each line is GB/s of output
(inflated text) over wall time, the device's including the copy of the file to the GPU and of the text back.  The first
device line of each file is a warm-up (CUDA context, module load).  The card's name and power limit are read in the
same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time
import zlib
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402


def fastq_text(n):
    from decombinator_b200 import _lib, tags
    info = tags.load("human", "extended", "b")
    syn = _lib.Synth([(info.v_regions, info.j_regions)], 20260002, 250, 62, 0.0, 0.0, 0.0)
    r1, _ = syn.reads(0, n, want_r2=False)
    a = r1.reshape(n, 250)
    rng = np.random.default_rng(7)
    q = rng.choice(np.frombuffer(b"FFFFFFF:,#", np.uint8), size=(n, 250), p=[0.12] * 7 + [0.08, 0.06, 0.02])
    step = 200_000
    parts = []
    for lo in range(0, n, step):
        hi = min(n, lo + step)
        parts.append(b"".join(b"@SYN:%d 1:N:0\n%s\n+\n%s\n" % (i, a[i].tobytes(), q[i].tobytes()) for i in range(lo, hi)))
    return b"".join(parts)


def bgzf(data, block=65280, threads=32):
    import struct

    def one(lo):
        chunk = data[lo:lo + block]
        c = zlib.compressobj(6, zlib.DEFLATED, -15)
        body = c.compress(chunk) + c.flush()
        bsize = 12 + 6 + len(body) + 8
        return (b"\x1f\x8b\x08\x04\0\0\0\0\0\xff" + struct.pack("<H", 6) + b"BC" + struct.pack("<HH", 2, bsize - 1) + body +
                struct.pack("<II", zlib.crc32(chunk), len(chunk)))
    with ThreadPoolExecutor(threads) as ex:
        parts = list(ex.map(one, range(0, len(data), block)))
    return b"".join(parts) + b"\x1f\x8b\x08\x04\0\0\0\0\0\xff\x06\0BC\x02\0\x1b\0\x03\0\0\0\0\0\0\0\0\0"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=10_000_000)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--chunks", default="65536,262144,1048576", help="nominal chunk sizes of the single-stream device runs")
    args = ap.parse_args()
    from decombinator_b200 import _lib, fastq
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    t0 = time.perf_counter()
    text = fastq_text(args.reads)
    t_gen = time.perf_counter() - t0
    t0 = time.perf_counter()
    with ThreadPoolExecutor(2) as ex:
        fut_b = ex.submit(bgzf, text)
        c = zlib.compressobj(6, zlib.DEFLATED, 31)
        single = c.compress(text) + c.flush()
        blocked = fut_b.result()
    t_comp = time.perf_counter() - t0
    tmp = "/tmp/bench_inflate"
    os.makedirs(tmp, exist_ok=True)
    files = {"gzip6": os.path.join(tmp, "R1.fq.gz"), "bgzf": os.path.join(tmp, "R1.bgzf.fq.gz")}
    with open(files["gzip6"], "wb") as fh:
        fh.write(single)
    with open(files["bgzf"], "wb") as fh:
        fh.write(blocked)
    del single, blocked
    print(json.dumps({"gpu": gpu, "reads": args.reads, "text_bytes": len(text), "generate_s": round(t_gen, 1), "compress_s": round(t_comp, 1),
                      "gzip6_bytes": os.path.getsize(files["gzip6"]), "bgzf_bytes": os.path.getsize(files["bgzf"])}), flush=True)
    real_device = fastq._device_gunzip
    chunks = [int(x) for x in args.chunks.split(",")]

    def device(path, chunk):
        t = time.perf_counter()
        with open(path, "rb") as fh:
            raw = fh.read()
        blocks = fastq._bgzf_blocks(raw)
        out = _lib.gpu_inflate(raw, members=blocks, chunk_bytes=chunk)
        return out, time.perf_counter() - t

    def host(path):
        fastq._device_gunzip = lambda raw, blocks: None
        try:
            t = time.perf_counter()
            out = fastq.gunzip_file(path)
            return out, time.perf_counter() - t
        finally:
            fastq._device_gunzip = real_device

    for name, path in files.items():
        device(path, chunks[0])                                    # warm-up
        modes = ["host"] + (["device_chunk_%d" % c for c in chunks] if name == "gzip6" else ["device"])
        for rep in range(args.reps):
            for mode in modes:
                if mode == "host":
                    out, dt = host(path)
                else:
                    out, dt = device(path, int(mode.rsplit("_", 1)[1]) if "chunk" in mode else 0)
                with memoryview(out) as mv:
                    same = len(mv) == len(text) and mv == text
                print(json.dumps({"file": name, "mode": mode, "rep": rep, "seconds": round(dt, 3), "out_GB_per_s": round(len(text) / dt / 1e9, 3),
                                  "same_bytes": bool(same)}), flush=True)
                del out


if __name__ == "__main__":
    main()
