#!/usr/bin/env python
"""User-facing path from FASTQ text: `decombinator(inputargs)` on a synthetic paired FASTQ (GPU box only).

    python tools/e2e_fastq.py [--reads 2000000] [--python-fastq]
    python tools/e2e_fastq.py --pipeline [--oligo I8_single|NEBIO|TAKARA] [--cli]
    python tools/e2e_fastq.py --pipeline --fuzzy-ab [--oligo ...] [--sub2 0.01]

Writes R1/R2 files of the configs[1] recipe under /tmp, runs the drop-in stage function (decombine.py:881 of the
reference) and prints where the wall time goes: ingest (FASTQ text -> record index), pack, device, row assembly.  With --pipeline --oligo, read 2 is re-laid out for that ligation-oligo design
(tests/oligo_layouts.py) and `pipeline` runs twice: as shipped, and with the barcodes of that design located on the
host (the device path restricted to M13 and I8 in this process, as before the device took the other designs).  With
--pipeline --cli, `pipeline` runs as the command line runs it (the .n12, .freq and .tsv written with -dz, the translate
stage handing its text to the writer), twice with the translate stage on the device and twice on the host, alternated.
With --pipeline --fuzzy-ab, read 2 gets --sub2 substitutions and 0.1 % indels per base of its barcode region, and
`pipeline` runs twice with DCB_BC_FUZZY=0 (the fuzzy spacer searches on the host) and twice as shipped, alternated.
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=2_000_000)
    ap.add_argument("--python-fastq", action="store_true", help="use the general (Python) parser instead of the native index")
    ap.add_argument("--gz", choices=["gzip", "bgzf"], default=None, help="compress the two files first: one gzip stream each, or BGZF blocks")
    ap.add_argument("--host-inflate", action="store_true", help="with --gz: inflate on the host as without a GPU (the path before dcb_inflate)")
    ap.add_argument("--rows-as-text", action="store_true", help="what the `decombine` command does: rows handed over as .n12 text")
    ap.add_argument("--profile", action="store_true", help="cProfile of the timed decombinator() call")
    ap.add_argument("--pipeline", action="store_true", help="decombine + collapse (pipeline.run) on reads with repeated UMIs")
    ap.add_argument("--oligo", default="M13", choices=["M13", "I8", "I8_single", "NEBIO", "TAKARA"],
                    help="with --pipeline: read 2 laid out for this ligation-oligo design")
    ap.add_argument("--cli", action="store_true", help="with --pipeline: the command line's path, translate on the device and on the host")
    ap.add_argument("--fuzzy-ab", action="store_true", help="with --pipeline: DCB_BC_FUZZY=0 against the default, alternated")
    ap.add_argument("--sub2", type=float, default=0.0, help="substitution rate of read 2")
    args = ap.parse_args()
    from decombinator_b200 import _lib, decombine, fastq, io, tags
    if args.host_inflate:
        fastq._device_gunzip = lambda raw, blocks: None
    info = tags.load("human", "extended", "b")
    L, n = 250, args.reads
    syn = _lib.Synth([(info.v_regions, info.j_regions)], 20260002, L, 42 + 20, 0.0, 0.0, 0.0,
                     umi_pool=(max(1000, n // 20) if args.pipeline else 0), sub_rate2=args.sub2)
    r1, r2 = syn.reads(0, n, want_r2=True)
    if args.oligo != "M13":
        import oligo_layouts
        r2 = oligo_layouts.relayout_array(r2.reshape(n, 62), args.oligo).reshape(-1)
    if args.fuzzy_ab:
        sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
        from bench_collapse import _indels
        r2 = _indels(np.ascontiguousarray(r2.reshape(n, 62)), np.random.default_rng(20261022), 0.001).reshape(-1)
    os.makedirs("/tmp/e2e", exist_ok=True)
    p1, p2 = "/tmp/e2e/syn_1.fq", "/tmp/e2e/syn_2.fq"
    t0 = time.perf_counter()
    for path, arr, ln in ((p1, r1, L), (p2, r2, 62)):
        a = arr.reshape(n, ln)
        with open(path, "wb") as fh:
            step = 200_000
            for lo in range(0, n, step):
                hi = min(n, lo + step)
                rows = [b"@SYN:%d 1:N:0\n%s\n+\n%s\n" % (i, a[i - lo + lo].tobytes(), b"I" * ln) for i in range(lo, hi)]
                fh.write(b"".join(rows))
    t_write = time.perf_counter() - t0
    if args.gz:
        import subprocess
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        for q in (p1, p2):
            if args.gz == "gzip":
                subprocess.run(["gzip", "-kf", q], check=True)
            else:
                from test_fastq_native import _bgzf
                with open(q, "rb") as fh, open(q + ".gz", "wb") as out:
                    out.write(_bgzf(fh.read()))
        p1, p2 = p1 + ".gz", p2 + ".gz"
    ia = io.create_args_dict(infile=p1, chain="b", bc_read="R2", suppresssummary=True, dontcheck=True, dontcount=True,
                             outpath="/tmp/e2e/")
    ia["python_fastq"] = args.python_fastq
    ia["rows_as_text"] = args.rows_as_text
    if args.pipeline:
        from decombinator_b200 import pipeline
        ia.update(dontsave=True, oligo=args.oligo, command="pipeline")
        t0 = time.perf_counter()
        rows = decombine.decombinator(dict(ia))
        t_dec = time.perf_counter() - t0
        if args.fuzzy_ab:
            from decombinator_b200 import collapse
            times, outs = {"0": [], "1": []}, {}
            for rep in range(2):
                for mode in ("0", "1"):
                    os.environ["DCB_BC_FUZZY"] = mode
                    t0 = time.perf_counter()
                    out = pipeline.run(dict(ia))
                    times[mode].append(round(time.perf_counter() - t0, 2))
                    outs[mode] = (out, {k: v for k, v in collapse.counts.items() if isinstance(v, int) and not k.startswith("time_")})
            same = outs["0"][0].equals(outs["1"][0]) and outs["0"][1] == outs["1"][1]
            print(json.dumps({"reads": n, "oligo": args.oligo, "sub2": args.sub2, "indels_per_base": 0.001,
                              "pipeline_s_DCB_BC_FUZZY_0": times["0"], "pipeline_s_default": times["1"],
                              "regexmatch": outs["1"][1].get("getbarcode_pass_regexmatch", 0), "same_output": bool(same)}))
            return
        if args.cli:
            import hashlib
            from decombinator_b200 import translate
            ia.update(dontsave=False, dontgzip=True)
            os.makedirs(ia["outpath"], exist_ok=True)
            tsv = ia["outpath"] + "dcr_" + os.path.basename(p1).split(".")[0] + "_beta.tsv"
            times, digests, device_ctx = {"device": [], "host": []}, {}, None
            for rep in range(2):
                for mode in ("device", "host"):
                    translate._dist = device_ctx if mode == "device" else False
                    t0 = time.perf_counter()
                    pipeline._run(dict(ia), frame=False)
                    times[mode].append(round(time.perf_counter() - t0, 2))
                    if mode == "device":
                        device_ctx = translate._dist
                    digests[mode] = hashlib.sha256(open(tsv, "rb").read()).hexdigest()
            print(json.dumps({"reads": n, "oligo": args.oligo, "cli_pipeline_s_translate_device": times["device"],
                              "cli_pipeline_s_translate_host": times["host"], "same_tsv": digests["device"] == digests["host"]}))
            return
        if args.profile:
            import cProfile, pstats
            pr = cProfile.Profile()
            pr.enable()
        t0 = time.perf_counter()
        out = pipeline.run(dict(ia))
        t_pipe = time.perf_counter() - t0
        if args.profile:
            pr.disable()
            pstats.Stats(pr).sort_stats("cumulative").print_stats(28)
        line = {"reads": n, "oligo": args.oligo, "decombinator_s": round(t_dec, 2), "pipeline_s": round(t_pipe, 2), "rows": len(rows),
                "translated": len(out), "pipeline_reads_per_s": round(n / t_pipe)}
        if args.oligo.lower() not in ("m13", "i8"):
            from decombinator_b200 import collapse
            device_counts = dict(collapse.counts)
            _lib.OLIGOS_ON_DEVICE = {"m13": 0, "i8": 1}          # this process only: the barcodes of args.oligo on the host
            t0 = time.perf_counter()
            host = pipeline.run(dict(ia))
            t_host = time.perf_counter() - t0
            same = host.equals(out) and all(collapse.counts[k] == v for k, v in device_counts.items() if isinstance(v, int) and not k.startswith("time_"))
            line.update(host_barcodes_pipeline_s=round(t_host, 2), host_barcodes_pipeline_reads_per_s=round(n / t_host), same_output=bool(same))
        print(json.dumps(line))
        return
    # warm-up: tables, context, CUDA
    small = dict(ia)
    decombine.import_tcr_info(small)
    t0 = time.perf_counter()
    opener = fastq.opener_check(ia)
    batch = fastq.load_pairs(ia, opener)
    t_ingest = time.perf_counter() - t0
    decombine.decombinator(dict(ia))          # first run: CUDA context, tables, page-locked buffers
    os.environ["DCB_TIMING"] = "1"
    if args.profile:
        import cProfile, pstats
        pr = cProfile.Profile()
        pr.enable()
    t0 = time.perf_counter()
    rows = decombine.decombinator(ia)
    t_total = time.perf_counter() - t0
    if args.profile:
        pr.disable()
        pstats.Stats(pr).sort_stats("cumulative").print_stats(22)
    print(json.dumps({"reads": n, "gz": args.gz, "host_inflate": bool(args.host_inflate), "parser": "python" if args.python_fastq else "native", "rows_as_text": bool(args.rows_as_text), "fastq_write_s": round(t_write, 2),
                      "ingest_only_s": round(t_ingest, 3), "decombinator_s": round(t_total, 2), "rows": len(rows),
                      "reads_per_s": round(n / t_total), "ingest_reads_per_s": round(n / t_ingest)}))


if __name__ == "__main__":
    main()
