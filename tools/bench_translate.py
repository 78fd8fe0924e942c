#!/usr/bin/env python
"""The translate stage on the device against the host path, on the same seeded rows (GPU box only).

    python tools/bench_translate.py [--rows 1000000 5000000] [--chains b a] [--out profiles/r03_bench_translate.json]

Rows are synthetic unique DCRs (tests/test_gpu_translate.synthetic_rows: random V / J of the chain, deletions 0..15,
inserts of 0..30 bases with rare N) for human beta and human alpha (extended tags).  Per chain and size:
  kernel_ms      dcb_translate's two kernels and the scan between them (CUDA events);
  text_s         what the command line does with -dz: translate_tsv + write_out_translated of the text;
  frame_s        cdr3translator(), i.e. the text turned into the DataFrame the Python interface returns;
  host_s         the host path (get_cdr3 loop, DataFrame, to_csv) on the same rows, in the same process;
  same_text      the device's .tsv bytes equal the host path's.
The golden 37-row .freq goes through the translate command both ways too, so that the cost of CUDA start-up and table
set-up on a tiny input shows.  Each measured call is preceded by one untimed call of the same shape."""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=60).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in out.split(",")]
        return name, power
    except Exception as e:      # noqa: BLE001
        return "unknown (%s)" % e, "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, nargs="+", default=[1_000_000, 5_000_000])
    ap.add_argument("--chains", nargs="+", default=["b", "a"], choices=["b", "a"])
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from decombinator_b200 import io, translate
    from test_gpu_translate import synthetic_rows

    tmp = tempfile.mkdtemp(prefix="bench_translate_")
    quiet = open(os.devnull, "w")

    def args_for(chain, infile, command, **kw):
        d = io.create_args_dict(infile=infile, chain=chain, bc_read="R2", dontgzip=True, outpath=tmp + os.sep, command=command,
                                suppresssummary=True)
        d.update(kw)
        return d

    def timed(fn):
        stdout = sys.stdout
        sys.stdout = quiet
        try:
            t0 = time.perf_counter()
            out = fn()
            return out, time.perf_counter() - t0
        finally:
            sys.stdout = stdout

    def host(fn):
        saved = translate._dist
        translate._dist = False
        try:
            return fn()
        finally:
            translate._dist = saved

    name, power = gpu_info()
    result = {"gpu": name, "power_limit": power, "runs": []}

    # the golden .freq: start-up on a tiny input
    for chain, cname in (("b", "beta"), ("a", "alpha")):
        src = os.path.join(ROOT, "tests", "golden", "dcr_TINY_1_%s.freq" % cname)
        freq = os.path.join(tmp, os.path.basename(src))
        shutil.copy(src, freq)
        args = args_for(chain, freq, "translate")
        first = translate._dist is None
        _, t_first = timed(lambda: io.write_out_translated(translate.translate_tsv(dict(args)), dict(args)))
        _, t_text = timed(lambda: io.write_out_translated(translate.translate_tsv(dict(args)), dict(args)))
        _, t_host = timed(lambda: host(lambda: io.write_out_translated(translate.translate_tsv(dict(args)), dict(args))))
        result["runs"].append({"chain": cname, "rows": 37, "input": "golden .freq, translate command, -dz",
                               "text_first_call_s": round(t_first, 4), "first_call_creates_context": first,
                               "text_s": round(t_text, 4), "host_s": round(t_host, 4)})
        print(json.dumps(result["runs"][-1]), flush=True)

    for chain, cname in (("b", "beta"), ("a", "alpha")):
        if chain not in a.chains:
            continue
        translate.import_gene_information({"species": "human", "tags": "extended", "chain": chain, "tagfastadir": None})
        g = translate._genes
        for n in a.rows:
            rows = synthetic_rows(g, n, 20261020 + n)
            args = args_for(chain, "bench.freq", None)
            out_tsv = os.path.join(tmp, "dcr_bench_%s.tsv" % cname)     # write_out_translated: prefix + file id + chain
            timed(lambda: translate.translate_tsv(dict(args), rows[:1000]))          # warm-up of the same path
            tsv, t_text = timed(lambda: io.write_out_translated(translate.translate_tsv(dict(args), rows), dict(args)))
            kernel_ms = translate._dist.last_ms()
            dev_bytes = open(out_tsv, "rb").read()
            _, t_frame = timed(lambda: translate.cdr3translator(dict(args), rows))
            _, t_host = timed(lambda: host(lambda: io.write_out_translated(translate.cdr3translator(dict(args), rows), dict(args))))
            same = open(out_tsv, "rb").read() == dev_bytes
            line = {"chain": cname, "rows": n, "tsv_bytes": len(dev_bytes), "kernel_ms": round(kernel_ms, 2),
                    "text_s": round(t_text, 2), "frame_s": round(t_frame, 2), "host_s": round(t_host, 2),
                    "text_rows_per_s": round(n / t_text), "host_rows_per_s": round(n / t_host),
                    "speedup_text_vs_host": round(t_host / t_text, 1), "same_text": bool(same)}
            result["runs"].append(line)
            print(json.dumps(line), flush=True)
            del rows, dev_bytes
    shutil.rmtree(tmp, ignore_errors=True)
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(result, fh, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
