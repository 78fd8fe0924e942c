#!/usr/bin/env python
"""e2e of dcb_decombine_ascii (ASCII reads in page-locked host memory -> records in host memory) with the chunks shared
from both ends at several chunk sizes, against the device packing every chunk.
usage (GPU box): python tools/e2e_share.py [reads]"""
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

from decombinator_b200 import _lib, tags  # noqa: E402

n = int(sys.argv[1]) if len(sys.argv) > 1 else 10_000_000
L = 250
info = tags.load("human", "extended", "b")
vt, jt = info.tables()
syn = _lib.Synth([(info.v_regions, info.j_regions)], 20260002, L, 0, 0.0, 0.0, 0.0)
r1, _ = syn.reads(0, n)
text = _lib.PinnedBytes(r1)
ctx = _lib.Context(vt, jt, device=0)
want = None
for name, env in (("two-ended, 128 K", {"DCB_CHUNK_READS": "131072"}), ("two-ended, 256 K", {"DCB_CHUNK_READS": "262144"}),
                  ("two-ended, 512 K", {"DCB_CHUNK_READS": "524288"}), ("two-ended, 1 M", {"DCB_CHUNK_READS": "1048576"}),
                  ("device only", {"DCB_HOST_SHARE": "0"})):
    for k in ("DCB_CHUNK_READS", "DCB_HOST_SHARE"):
        os.environ.pop(k, None)
    os.environ.update(env)
    for _ in range(3):
        res, cnt = ctx.decombine_ascii(text.a, None, None, True, uniform_len=L, pinned=True)
    if want is None:
        want = (res.copy(), cnt.copy())
    t0 = time.perf_counter()
    steps = 10
    for _ in range(steps):
        res, cnt = ctx.decombine_ascii(text.a, None, None, True, uniform_len=L, pinned=True)
    dt = (time.perf_counter() - t0) / steps
    assert np.array_equal(res, want[0]) and np.array_equal(cnt, want[1])
    host, dev = ctx.last_pack_shares()
    print(json.dumps({"scheme": name, "reads_per_s": n / dt, "ms": dt * 1e3, "host_chunks": host, "device_chunks": dev}), flush=True)
