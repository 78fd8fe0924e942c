#!/usr/bin/env python
"""Throughput of the collapse primitives (SURVEY 8(d)): pair verifications/s of dcb_umi_pairs and verdicts/s of
dcb_lev_leq on synthetic inputs shaped like configs[3] (12-nt UMIs, <= 130-nt inter-tag sequences), and rows/s of
dcb_barcodes for each ligation-oligo design on 42-nt barcode regions (the generator's read 2 with 0.5 % substitutions,
re-laid out per design by tests/oligo_layouts.py).

    python tools/bench_collapse.py [--umis 200000] [--pairs 2000000] [--barcode-rows 10000000]     (GPU box)
    python tools/bench_collapse.py --fuzzy-rows 1000000                                           (GPU box)

Prints one JSON line; device times come from the library's own CUDA events (dcb_dist_last_ms).  --fuzzy-rows measures
only the fuzzy spacer searches of dcb_barcodes_fuzzy (bench_fuzzy)."""
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
    ap.add_argument("--umis", type=int, default=200_000)
    ap.add_argument("--pairs", type=int, default=2_000_000)
    ap.add_argument("--big", type=int, default=2_000_000, help="UMIs of the configs[3]-scale pair search (0 = skip)")
    ap.add_argument("--barcode-rows", type=int, default=10_000_000, help="barcode regions per design for dcb_barcodes (0 = skip)")
    ap.add_argument("--fuzzy-rows", type=int, default=0, help="only bench_fuzzy, over this many barcode regions per design and rate")
    args = ap.parse_args()
    if args.fuzzy_rows:
        print(json.dumps(bench_fuzzy(args.fuzzy_rows)))
        return
    from decombinator_b200 import _lib
    rng = np.random.default_rng(20260004)
    U = args.umis
    # distinct random 12-nt UMIs + 5 % one-edit neighbours of earlier ones (so pairs exist), as 3-bit codes
    base = rng.integers(0, 4, size=(U, 12), dtype=np.uint64)
    nb = rng.random(U) < 0.05
    src = rng.integers(0, np.maximum(np.arange(U), 1))
    base[nb] = base[src[nb]]
    pos = rng.integers(0, 12, size=U)
    base[nb, pos[nb]] = (base[nb, pos[nb]] + 1 + rng.integers(0, 3, size=int(nb.sum()), dtype=np.uint64)) % 4
    codes = (np.uint64(12) << np.uint64(58)) | (base << (np.uint64(3) * np.arange(12, dtype=np.uint64))).sum(axis=1, dtype=np.uint64)
    codes = np.unique(codes)
    U = len(codes)
    d = _lib.Dist(0)
    d.umi_pairs(codes[:1000], 2)
    d.umi_pairs(codes[:8192], 2)            # both forms of the search loaded before anything is timed
    t0 = time.perf_counter()
    row, col = d.umi_pairs(codes, 2)
    wall_pairs = time.perf_counter() - t0
    ms_pairs = d.last_ms()
    method = d.last_method()
    checks = U * (U - 1) / 2
    # the same list through the all-pairs sweep (what round 1 shipped), for the comparison
    os.environ["DCB_UMI_SYMDEL_MIN"] = "1000000000"
    row_ap, col_ap = d.umi_pairs(codes, 2)
    ms_ap = d.last_ms()
    del os.environ["DCB_UMI_SYMDEL_MIN"]
    assert np.array_equal(row, row_ap) and np.array_equal(col, col_ap)
    # BASELINE configs[3] scale: 2 M distinct random 12-nt UMIs
    big = None
    if args.big:
        vals = np.unique(rng.integers(0, 4 ** 12, size=int(args.big * 1.1), dtype=np.uint64))[:args.big]
        rng.shuffle(vals)
        cb = np.full(len(vals), 12 << 58, dtype=np.uint64)
        for k in range(12):
            cb |= ((vals >> np.uint64(2 * k)) & np.uint64(3)) << np.uint64(3 * k)
        t0 = time.perf_counter()
        rb, _ = d.umi_pairs(cb, 2)
        big = {"unique_umis": int(len(cb)), "pairs_found": int(len(rb)), "device_ms": d.last_ms(), "method": d.last_method(),
               "wall_s_incl_copy_of_pairs_to_host": time.perf_counter() - t0,
               "all_pairs_checks_avoided": len(cb) * (len(cb) - 1) / 2}
    # bounded Levenshtein verdicts on inter-tag sequences: random 60..130-nt strings, half of the pairs near-identical
    n_seq = 200_000
    lens = rng.integers(60, 131, size=n_seq).astype(np.uint32)
    off = np.zeros(n_seq, dtype=np.uint64)
    off[1:] = np.cumsum(lens[:-1], dtype=np.uint64)
    sym = rng.integers(0, 4, size=int(lens.sum()), dtype=np.uint8)
    a = rng.integers(0, n_seq, size=args.pairs).astype(np.uint32)
    b = rng.integers(0, n_seq, size=args.pairs).astype(np.uint32)
    b[::2] = a[::2]                                  # identical pairs (distance 0) for the accepting half
    d.lev_leq(sym, off, lens, a[:1000], b[:1000], 0.1)
    t0 = time.perf_counter()
    verdict = d.lev_leq(sym, off, lens, a, b, 0.1)
    wall_lev = time.perf_counter() - t0
    ms_lev = d.last_ms()
    barcodes = bench_barcodes(d, args.barcode_rows) if args.barcode_rows else None
    print(json.dumps({
        "umi_pairs": {"unique_umis": U, "pairs_found": int(len(row)), "method": method, "device_ms": ms_pairs, "wall_s": wall_pairs,
                      "all_pairs_sweep": {"pair_checks": checks, "device_ms": ms_ap, "checks_per_s": checks / (ms_ap / 1e3)},
                      "algorithmic_bytes": 8 * U + 8 * int(len(row)), "hbm_GBps": (8 * U + 8 * len(row)) / (ms_pairs / 1e3) / 1e9},
        "umi_pairs_2M": big,
        "lev_leq": {"pairs": int(args.pairs), "accepted": int(verdict.sum()), "device_ms": ms_lev,
                    "verdicts_per_s": args.pairs / (ms_lev / 1e3), "wall_s": wall_lev},
        "barcodes": barcodes}))


def bench_barcodes(d, n):
    """dcb_barcodes over n 42-nt barcode regions per design, quality all 'I', -N off, the default quality filter."""
    import oligo_layouts
    from decombinator_b200 import _lib, tags
    info = tags.load("human", "extended", "b")
    syn = _lib.Synth([(info.v_regions, info.j_regions)], 20260004, 250, 62, 0.0, 0.0, 0.0, umi_pool=max(1000, n // 50),
                     sub_rate2=0.005)
    step = 1_000_000
    r2 = np.concatenate([syn.reads(lo, min(step, n - lo), want_r2=True)[1].reshape(-1, 62) for lo in range(0, n, step)])
    bo = np.arange(n, dtype=np.uint64) * np.uint64(62)
    bl = np.full(n, 42, dtype=np.uint32)
    qbuf, qo = np.full(64, ord("I"), dtype=np.uint8), np.zeros(n, dtype=np.uint64)
    out = {"rows": n, "region": "42 nt of a 62-nt read 2, 0.5 % substitutions"}
    for oligo in ("M13", "I8", "I8_single", "NEBIO", "TAKARA"):
        text = np.ascontiguousarray(r2 if oligo == "M13" else oligo_layouts.relayout_array(r2, oligo)).reshape(-1)
        code = _lib.OLIGOS_ON_DEVICE[oligo.lower()]
        d.barcodes_arrays(text, bo[:1000], bl[:1000], qbuf, qo[:1000], bl[:1000], code, False, 20, 1, 30)
        st, _, _ = d.barcodes_arrays(text, bo, bl, qbuf, qo, bl, code, False, 20, 1, 30)
        ms = d.last_ms()
        out[oligo] = {"device_ms": ms, "rows_per_s": n / (ms / 1e3), "decided_on_device": float((st != _lib.BC_HOST).mean()),
                      "passed": float((st == _lib.BC_OK).mean())}
    return out


def _indels(a, rng, rate, span=42):
    """Each of the first `span` bases of every row of a (uint8, rows x width) deleted (a random base appended) or followed by
    an inserted base (the last base dropped) with probability `rate`."""
    k = rng.binomial(span, rate, size=len(a))
    for i in np.nonzero(k)[0].tolist():
        row = a[i].tolist()
        for _ in range(int(k[i])):
            p = int(rng.integers(span))
            if rng.random() < 0.5:
                row = row[:p] + row[p + 1:] + [int(rng.choice(list(b"ACGT")))]
            else:
                row = row[:p] + [int(rng.choice(list(b"ACGT")))] + row[p:-1]
        a[i] = row
    return a


def bench_fuzzy(n):
    """Per design and read-2 substitution rate (0.5, 1 and 2 %, plus 0.1 % indels per base of the 42-nt region): the rows
    dcb_barcodes hands back (exact spacer searches only) and dcb_barcodes_fuzzy hands back, the kernel time of each (CUDA
    events, best of three, the quality text one cached row), and the wall time of collapse._filter_rows over the same
    regions as the columns of an .n12 file (the `collapse` command's path) with DCB_BC_FUZZY=0 and with the default,
    alternated, with the kept rows and counters compared."""
    import tempfile
    import oligo_layouts
    from decombinator_b200 import _lib, collapse, tags
    info = tags.load("human", "extended", "b")
    rng = np.random.default_rng(20261022)
    d = _lib.Dist(0)
    bo = np.arange(n, dtype=np.uint64) * np.uint64(62)
    bl = np.full(n, 42, dtype=np.uint32)
    qbuf, qo = np.full(64, ord("I"), dtype=np.uint8), np.zeros(n, dtype=np.uint64)
    out = {"rows": n, "region": "42 nt of a 62-nt read 2, substitutions at the rate given + 0.1 % indels per base", "runs": []}
    seqs = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=(n, 30))]
    head = np.frombuffer(b"".join(b"12, 3, 1, 2, ACGT, SYN:%07d, " % i for i in range(n)), dtype=np.uint8).reshape(n, -1)
    comma = np.frombuffer(b", ", dtype=np.uint8)
    tmp = tempfile.mkdtemp()
    for rate in (0.005, 0.01, 0.02):
        syn = _lib.Synth([(info.v_regions, info.j_regions)], 20260004, 250, 62, 0.0, 0.0, 0.0, umi_pool=max(1000, n // 50),
                         sub_rate2=rate)
        r2 = syn.reads(0, n, want_r2=True)[1].reshape(n, 62)
        for oligo in ("M13", "I8", "I8_single", "NEBIO", "TAKARA"):
            reg = np.ascontiguousarray(r2 if oligo == "M13" else oligo_layouts.relayout_array(r2, oligo))
            reg = _indels(reg, rng, 0.001)
            text = reg.reshape(-1)
            code = _lib.OLIGOS_ON_DEVICE[oligo.lower()]
            d.barcodes_arrays(text, bo[:1000], bl[:1000], qbuf, qo[:1000], bl[:1000], code, False, 20, 1, 30)
            d.barcodes_arrays(text, bo[:1000], bl[:1000], qbuf, qo[:1000], bl[:1000], code, False, 20, 1, 30, True)
            ms_off, ms_on = [], []
            for _ in range(3):
                st_off = d.barcodes_arrays(text, bo, bl, qbuf, qo, bl, code, False, 20, 1, 30)[0]
                ms_off.append(d.last_ms())
                st_on, _, _, match = d.barcodes_arrays(text, bo, bl, qbuf, qo, bl, code, False, 20, 1, 30, True)
                ms_on.append(d.last_ms())
            # the same regions as an .n12 file: what collapse reads, timed through _filter_rows
            q = np.full((n, 30), ord("I"), dtype=np.uint8)
            rows = np.concatenate([head, seqs, np.tile(comma, (n, 1)), q, np.tile(comma, (n, 1)), reg[:, :42], np.tile(comma, (n, 1)),
                                   np.full((n, 42), ord("I"), dtype=np.uint8), np.full((n, 1), ord("\n"), dtype=np.uint8)], axis=1)
            path = os.path.join(tmp, "rows.n12")
            rows.tofile(path)
            n12 = collapse.N12Columns.from_file(path, open)
            args = {"oligo": oligo, "sampling_analysis": False, "allowNs": False, "lenthreshold": 130}
            wall = {"0": [], "1": []}
            result = {}
            for _ in range(2):
                for mode in ("0", "1"):
                    os.environ["DCB_BC_FUZZY"] = mode
                    collapse.counts = collapse.coll.Counter()
                    t0 = time.perf_counter()
                    kept, dcrs, _ = collapse._filter_rows(n12, args, [20, 1, 30], True, False)
                    wall[mode].append(round(time.perf_counter() - t0, 3))
                    result[mode] = (kept, dcrs, {k: v for k, v in collapse.counts.items() if isinstance(v, int)})
            del os.environ["DCB_BC_FUZZY"]
            placed = (st_on == _lib.BC_OK) | (st_on == _lib.BC_FAIL_QUALITY)
            out["runs"].append({
                "oligo": oligo, "sub_rate2": rate, "handed_back_exact_only": float((st_off == _lib.BC_HOST).mean()),
                "handed_back_fuzzy": float((st_on == _lib.BC_HOST).mean()), "placed_by_fuzzy_text": float((placed & (match != 0)).mean()),
                "kernel_ms_exact_only": min(ms_off), "kernel_ms_fuzzy": min(ms_on),
                "filter_rows_s_DCB_BC_FUZZY_0": wall["0"], "filter_rows_s_default": wall["1"],
                "filter_rows_same_output": result["0"] == result["1"]})
            print(json.dumps(out["runs"][-1]), file=sys.stderr, flush=True)
    return out


if __name__ == "__main__":
    main()
