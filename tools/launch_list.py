#!/usr/bin/env python
"""Launch list of resident steps on bench.py's headline batch (configs[1]), from torch.profiler's CUDA activity trace
(GPU box): every kernel and memset of a few steps, with its start relative to the first, its duration and the gap from
the end of the activity before it (negative: the two overlapped).  Timing is on, as in bench.py's timed loop.

    python tools/launch_list.py [--reads 10000000] [--steps 8] --out launches.csv

Run it once per DCB_PDL setting; the CSV's setting column says which."""
import argparse
import csv
import json
import os
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=10_000_000)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile
    from decombinator_b200 import _lib, tags
    info = tags.load("human", "extended", "b")
    n, L = args.reads, 250
    syn = _lib.Synth([(info.v_regions, info.j_regions)], 20260002, L, 0, 0.0, 0.0, 0.0)
    r1, _ = syn.reads(0, n, n_threads=os.cpu_count() or 8)
    packed = _lib.pack_arrays(r1, np.arange(n, dtype=np.uint64) * L, np.full(n, L, dtype=np.uint32), revcomp=True,
                              n_threads=os.cpu_count() or 8)
    vt, jt = info.tables()
    ctx = _lib.Context(vt, jt, device=0)
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)
    ctx.upload(packed)
    with torch.cuda.stream(stream):
        for _ in range(200):
            ctx.run_resident()
        torch.cuda.synchronize()
        ctx.timing_enable(True)
        ctx.timing_reset()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(args.steps):
                ctx.run_resident()
            torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        trace = json.load(open(path))
    acts = sorted((e for e in trace["traceEvents"] if e.get("ph") == "X" and e.get("cat") in ("kernel", "gpu_memset")),
                  key=lambda e: e["ts"])
    setting = os.environ.get("DCB_PDL", "1")
    t0, prev_end = acts[0]["ts"], None
    with open(args.out, "w", newline="") as fh:
        w = csv.writer(fh)
        w.writerow(["setting", "activity", "start_us", "dur_us", "gap_from_previous_end_us"])
        for e in acts:
            name = e["name"].split("(")[0].split("<")[0].replace("void ", "")
            w.writerow([setting, name, "%.3f" % (e["ts"] - t0), "%.3f" % e["dur"],
                        "" if prev_end is None else "%.3f" % (e["ts"] - prev_end)])
            prev_end = e["ts"] + e["dur"] if prev_end is None else max(prev_end, e["ts"] + e["dur"])
    exact = [e for e in acts if "exact" in e["name"]]
    period = (exact[-1]["ts"] - exact[0]["ts"]) / max(1, len(exact) - 1)
    print(json.dumps({"setting": setting, "activities": len(acts), "step_period_us": period,
                      "exact_kernel_us": float(np.mean([e["dur"] for e in exact])),
                      "by_name_us": {k: float(np.mean([e["dur"] for e in acts if k in e["name"]]))
                                     for k in ("exact", "halftag", "general", "emset", "Memset")
                                     if any(k in e["name"] for e in acts)}}))
    ctx.close(); packed.free()


if __name__ == "__main__":
    main()
