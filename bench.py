#!/usr/bin/env python
"""Benchmark of the decombine hot path on B200 (driver contract: one JSON line on stdout from rank 0).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--reads R] [--impl reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): synthetic 10 M x 250-nt reads, human beta, extended tag set,
-br R2 -bl 42 -ol M13.  One "step" = one pass of the decombine kernels over the whole batch of packed
reads.  Weak scaling: every GPU gets its own 10 M-read shard of the same deterministic stream
(contiguous index ranges, no data-path collective: reads are independent).

  value     whole-job reads/s with the packed batch resident in HBM (K steps, CUDA events, max over ranks)
  e2e       the same through the C-ABI call dcb_decombine_ascii: ASCII reads in pinned HOST memory in (what the
            reference arm consumes), packed on the device, result records in host memory out, copies inside the
            timed region; e2e_packed: dcb_decombine_batch on reads already 2-bit packed on the host
  roofline  exact-tag kernel: algorithmic bytes (ceil(L/4)+16 per read) / its mean device time, against the
            measured HBM copy bandwidth in MEASURED_PEAKS.json
  cpu_baseline  the oracle's C port of the reference's dcr() on this box's host cores (a reported baseline)

`--impl reference` times only that CPU port (the reference itself is pure Python + absent wheels and cannot be
installed offline; its algorithm is what oracle/dcr_oracle.c restates and pins against reference fixtures).
"""
import argparse
import atexit
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

# stdout carries ONE JSON line: keep a private handle on it and point file descriptor 1 at stderr, so that whatever a
# library prints there (NCCL's version banner at NCCL_DEBUG=VERSION/WARN/INFO, for one) cannot end up beside the line
_JSON_OUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)

METRIC = "decombined_reads_per_sec"
UNIT = "reads/s"
READ_LEN = 250
SEED = 20260002
WORKLOAD = "synthetic 250-nt reads, human beta, extended tag set, -br R2 -bl 42 -ol M13 (BASELINE configs[1])"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--reads", type=int, default=10_000_000, help="reads per GPU")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-sample", type=int, default=0, help="reads in the cpu_baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--sub-rate", type=float, default=0.0, help="per-base substitution rate of the synthetic reads (default: the headline workload, 0)")
    ap.add_argument("--n-rate", type=float, default=0.0, help="per-base N rate")
    ap.add_argument("--no-workloads", action="store_true", help="skip the extra workload blocks (configs[2])")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write rank 0's results of the last resident step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the results of the CUDA path; --impl reference has none")
    return args


DUMP_READS = 1 << 20     # 10 record fields as float32 + the index as float64: 48 MiB of the 64 MB a dump may take


def dump_outputs(dirname, res, cnt):
    """What a caller of the resident path receives (the counters and every field of the result records), as .npy files
    that two builds can be compared by: the records of a fixed, seeded sample of DUMP_READS reads (all reads when there
    are no more), their read indices in read_index.npy."""
    os.makedirs(dirname, exist_ok=True)
    n = len(res)
    if n > DUMP_READS:
        idx = np.sort(np.random.default_rng(SEED).choice(n, DUMP_READS, replace=False))
    else:
        idx = np.arange(n)
    np.save(os.path.join(dirname, "read_index.npy"), idx.astype(np.float64))
    for f in res.dtype.names:
        np.save(os.path.join(dirname, f + ".npy"), res[f][idx].astype(np.float32))
    np.save(os.path.join(dirname, "counters.npy"), cnt.astype(np.float64))


def make_reads(info, first, n, threads, sub_rate=0.0, n_rate=0.0):
    from decombinator_b200 import _lib
    syn = _lib.Synth([(info.v_regions, info.j_regions)], SEED, READ_LEN, 0, sub_rate, n_rate, 0.0)
    r1, _ = syn.reads(first, n, n_threads=threads)
    off = np.arange(n, dtype=np.uint64) * READ_LEN
    ln = np.full(n, READ_LEN, dtype=np.uint32)
    return r1, off, ln


def cpu_reference_run(r1, off, ln, threads, steps=1, warmup=0):
    """The oracle's C port of dcr() (incl. the reverse complement) over ASCII reads in host memory."""
    import decombine_oracle as O
    orc = O.Oracle(O.TagSet("human", "extended", "b"))
    for _ in range(warmup):
        orc.decombine_arrays(r1, off, ln, "reverse", nthreads=threads)
    t0 = time.perf_counter()
    for _ in range(steps):
        res = orc.decombine_arrays(r1, off, ln, "reverse", nthreads=threads)
    dt = time.perf_counter() - t0
    return len(off) * steps / dt, dt / steps, int(res["ok"].sum())


def reference_timing():
    """The unmodified reference (pure Python + stand-ins for its absent wheels, compiled Aho-Corasick behind `acora`) on one
    core: measured by oracle/time_reference.py in the build container -- /root/reference does not exist on the GPU box --
    and committed under profiles/."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "r02_reference_cpu_timing.json")))
        return {"value": t["value"], "unit": UNIT, "cores": 1, "kind": "reference", "cpu": t["cpu"], "where": t["where"],
                "sample": t["workload"], "source": "profiles/r02_reference_cpu_timing.json (oracle/time_reference.py)"}
    except Exception:
        return None


def run_mixed(args, rank, world, local_rank, host_threads, stream, barrier, species, tagset, chains, seed, sub, nrate, label):
    """One mixed file (read i is a molecule of chain i % len(chains)) analysed once per chain, as the reference's example
    runs `-c a` and `-c b` on the same FASTQ.  Batch resident in HBM, K passes of all kernels per chain, CUDA events on
    the launching stream, max over ranks."""
    import torch
    import torch.distributed as dist
    from decombinator_b200 import _lib, tags
    infos = [tags.load(species, tagset, c) for c in chains]
    n = args.reads
    syn = _lib.Synth([(i.v_regions, i.j_regions) for i in infos], seed, READ_LEN, 0, sub, nrate, 0.0)
    r1, _ = syn.reads(rank * n, n, n_threads=host_threads)
    off = np.arange(n, dtype=np.uint64) * READ_LEN
    ln = np.full(n, READ_LEN, dtype=np.uint32)
    packed = _lib.pack_arrays(r1, off, ln, revcomp=True, n_threads=host_threads)
    del r1
    steps = args.steps
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    out = {"workload": label % n, "seed": seed, "steps": steps, "chains": {}}
    total_ms = 0.0
    for chain, info in zip(chains, infos):
        vt, jt = info.tables()
        ctx = _lib.Context(vt, jt, device=local_rank)
        ctx.set_stream(stream.cuda_stream)
        ctx.upload(packed)
        with torch.cuda.stream(stream):
            for _ in range(5):
                ctx.run_resident()
            torch.cuda.synchronize()
            res, cnt = ctx.download()
            ctx.timing_enable(True); ctx.timing_reset()
            barrier()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record(stream)
            for _ in range(steps):
                ctx.run_resident()
            ev1.record(stream)
            barrier()
            ms = ev0.elapsed_time(ev1)
        if world > 1:
            t = torch.tensor([ms], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t[0])
        kms, kl = ctx.timing_get()
        per = [kms[i] / max(1, kl[i]) for i in range(3)]
        bpr = (READ_LEN + 3) // 4 + 16
        out["chains"][chain] = {
            "value": world * n * steps / (ms / 1e3), "unit": UNIT, "ms_per_step": ms / steps,
            "decombined_fraction": float(res["status"].mean()),
            "queued_by_exact_kernel": ctx.last_deferred() / n, "deferred_to_general_kernel": ctx.last_general() / n,
            "kernels_ms": {ctx.exact_kernel_name(): per[0], "dcb_halftag_kernel": per[2], "dcb_general_kernel": per[1]},
            "roofline_frac_all_kernels": bpr * n / (ms / steps / 1e3) / 1e9 / peak,
            "gpu_launches": int(kl.sum()),
        }
        total_ms += ms / steps
        ctx.close()
    packed.free()
    out["value"] = world * n / (total_ms / 1e3)
    out["unit"] = "reads of the file/s, all chains analysed"
    out["ms_per_file_pass"] = total_ms
    return out


def run_cfg2(args, rank, world, local_rank, host_threads, stream, barrier):
    """BASELINE configs[2]: human alpha / beta, extended tag sets, 1 % substitutions + 0.1 % N per base."""
    return run_mixed(args, rank, world, local_rank, host_threads, stream, barrier, "human", "extended", ("a", "b"), 20260003, 0.01, 0.001,
                     "synthetic 250-nt reads, one mixed file (even reads human alpha, odd reads human beta), extended tag sets, "
                     "1 %% substitutions + 0.1 %% N per base, analysed once per chain (BASELINE configs[2] shape, %d reads per GPU)")


def run_cfg4(args, rank, world, local_rank, host_threads, stream, barrier):
    """BASELINE configs[4]: mouse gamma / delta, original tag sets (12-nt J tags: the bit-filter exact kernel), 0.5 % substitutions."""
    return run_mixed(args, rank, world, local_rank, host_threads, stream, barrier, "mouse", "original", ("g", "d"), 20260005, 0.005, 0.0,
                     "synthetic 250-nt reads, one mixed file (even reads mouse gamma, odd reads mouse delta), original tag sets, "
                     "0.5 %% substitutions per base, analysed once per chain (BASELINE configs[4] shape, %d reads per GPU; the named "
                     "500 M reads on 8 GPUs are 6.25 such shards per GPU)")


def run_cfg3(args, rank, world, local_rank, host_threads, stream, barrier):
    """BASELINE configs[3] in the same run: decombine + the device steps of collapse on reads with UMI barcodes (human beta,
    0.5 % substitutions in R1 and in the 42-nt barcode region, every molecule ~50 copies): the decombine kernels, the
    barcode-extraction kernel, the barcode-hash all-to-all of 64-byte records between the GPUs (NCCL, device tensors;
    N > 1 only) and the UMI neighbour search over the gathered unique barcodes.  The order-dependent grouping that follows
    is host code (collapse.py) and is not part of this block."""
    import torch
    import torch.distributed as dist
    from decombinator_b200 import _lib, parallel, tags
    info = tags.load("human", "extended", "b")
    n, seed = args.reads, 20260004
    pool = max(1000, n * world // 50)
    syn = _lib.Synth([(info.v_regions, info.j_regions)], seed, READ_LEN, 62, 0.005, 0.0, 0.0, umi_pool=pool, sub_rate2=0.005)
    r1, r2 = syn.reads(rank * n, n, want_r2=True, n_threads=host_threads)
    off = np.arange(n, dtype=np.uint64) * READ_LEN
    ln = np.full(n, READ_LEN, dtype=np.uint32)
    packed = _lib.pack_arrays(r1, off, ln, revcomp=True, n_threads=host_threads)
    del r1
    steps = args.steps
    vt, jt = info.tables()
    ctx = _lib.Context(vt, jt, device=local_rank)
    ctx.set_stream(stream.cuda_stream)
    ctx.upload(packed)
    with torch.cuda.stream(stream):
        for _ in range(5):
            ctx.run_resident()
        torch.cuda.synchronize()
        res, _ = ctx.download()
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        for _ in range(steps):
            ctx.run_resident()
        ev1.record(stream)
        barrier()
        ms = ev0.elapsed_time(ev1)
    if world > 1:
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t[0])
    queued, general = ctx.last_deferred() / n, ctx.last_general() / n
    ctx.close(); packed.free()
    out = {"workload": "synthetic 250-nt reads with UMI barcodes (M13 oligo, 42-nt barcode region in R2), human beta, 0.5 %% substitutions in R1 "
                       "and in the barcode region, %d molecules x ~50 copies (BASELINE configs[3] shape, %d reads per GPU)" % (pool, n),
           "seed": seed,
           "decombine": {"value": world * n * steps / (ms / 1e3), "unit": UNIT, "ms_per_step": ms / steps,
                         "decombined_fraction": float(res["status"].mean()), "queued_by_exact_kernel": queued,
                         "deferred_to_general_kernel": general}}
    # barcode extraction of the decombined rows (exact-spacer fast path + quality filter on the device)
    hits = np.nonzero(res["status"])[0]
    d = _lib.Dist(local_rank)
    qbuf = np.full(62, ord("I"), dtype=np.uint8)
    bo = hits.astype(np.uint64) * np.uint64(62)
    bl = np.full(len(hits), 42, dtype=np.uint32)
    qo = np.zeros(len(hits), dtype=np.uint64)
    st, n1, code = d.barcodes_arrays(r2, bo, bl, qbuf, qo, bl, 0, False, 20, 1, 30)
    bc_ms = d.last_ms()
    ok = st == _lib.BC_OK
    out["barcodes"] = {"rows": int(len(hits)), "device_ms": bc_ms, "rows_per_s": len(hits) / (bc_ms / 1e3),
                       "decided_on_device": float((st != _lib.BC_HOST).mean()), "passed": float(ok.mean()),
                       "algorithmic_GBps": len(hits) * (84 + 10) / (bc_ms / 1e3) / 1e9}
    # the 64-byte records of the surviving rows, exchanged by barcode hash
    rec = np.zeros(int(ok.sum()), dtype=parallel.RECORD)
    rec["idx"] = (rank * n + hits[ok]).astype(np.uint64)
    rec["code"] = code[ok]
    for f in ("v", "j", "vdel", "jdel"):
        rec[f] = res[f][hits[ok]]
    ex = {"records_per_gpu": int(len(rec)), "bytes_per_record": 64}
    if world > 1:
        mine = parallel.exchange_records(rec)                      # warm-up of the same call (NCCL channels)
        reps, tot = 5, 0.0
        for _ in range(reps):
            mine = parallel.exchange_records(rec)
            tot += parallel._last_exchange["ms"]
        t = torch.tensor([tot / reps, float(parallel._last_exchange["sent_bytes"])], device="cuda", dtype=torch.float64)
        tmax = t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone(); dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        a2a_ms, total_bytes = float(tmax[0]), float(tsum[1])
        off_rank = total_bytes * (world - 1) / world
        ex.update({"all_to_all_ms": a2a_ms, "bytes_sent_all_gpus": total_bytes,
                   "GBps_per_gpu_off_rank": off_rank / world / (a2a_ms / 1e3) / 1e9, "bound_GBps_per_gpu": 770.0,
                   "frac_of_bound": off_rank / world / (a2a_ms / 1e3) / 1e9 / 770.0,
                   "how": "torch.distributed.all_to_all_single on device tensors (NCCL), CUDA events, max over ranks"})
    else:
        mine = rec
        ex["note"] = "one GPU: no exchange"
    out["exchange"] = ex
    # UMI neighbour search over the unique barcodes of the whole job (all-gather of the codes, search on every rank's GPU;
    # rank 0's time is reported)
    uniq = np.unique(mine["code"])
    codes, sizes = parallel.all_gather_codes(uniq)
    d.umi_pairs(codes[:1000], 2)
    row, _ = d.umi_pairs(codes, 2)
    out["umi_pairs"] = {"unique_umis": int(len(codes)), "pairs": int(len(row)), "device_ms": d.last_ms(), "method": d.last_method(),
                        "max_edits": 2}
    d.close()
    return out


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            atexit.register(self.proc.kill)   # the sampler loops until killed: never outlive a run that fails before stop()
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for t, line in self.rows:
            if t < t0 - 0.05 or t > t1 + 0.05:
                continue
            parts = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(parts[0])); mx = float(parts[1])
            except Exception:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:  # region shorter than the sampling period: use the nearest samples
            for t, line in self.rows[-3:]:
                try:
                    parts = [x.strip() for x in line.split(",")]
                    sm.append(float(parts[0])); mx = float(parts[1])
                except Exception:
                    pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    host_threads = max(1, (os.cpu_count() or 1) // max(1, world if args.impl == "b200" else 1))

    from decombinator_b200 import tags
    info = tags.load("human", "extended", "b")
    config = {"workload": WORKLOAD, "reads_per_gpu": args.reads, "read_len": READ_LEN, "seed": SEED,
              "l2": "packed batch (64 B/read) is larger than the 126 MB L2; no flush needed",
              "spin_up": "0.5 s of untimed passes before the W warm-up steps (clock ramp); clocks are sampled from the spin-up to the end of the timed region (the same kernels back to back)",
              "sharding": "contiguous read-index shards, one per GPU, no collective"}

    if args.sub_rate or args.n_rate:
        config["workload"] += " + %.3g substitutions, %.3g N per base (NOT the headline workload)" % (args.sub_rate, args.n_rate)
    # ---------------------------------------------------------------------------------------------
    if args.impl == "reference":
        if rank != 0:
            return
        # Nothing of the product is on this path: reads come from libdcbsynth.so (the generator alone), the timed call is the
        # oracle's C port (oracle/liboracle.so) on all host threads.  The reference itself is pure Python with native deps that
        # cannot be installed offline; its own speed (with stand-ins) is quoted from profiles/r02_reference_cpu_timing.json.
        threads = os.cpu_count() or 1
        n = args.reads
        r1, off, ln = make_reads(info, 0, n, threads, args.sub_rate, args.n_rate)
        rps, sec, _ = cpu_reference_run(r1, off, ln, threads, steps=1, warmup=1)        # warm pass, then the size of a step
        steps = max(1, args.steps)
        # a step is a bounded sample of the workload: the whole run (K steps + W warm-ups) stays under about two minutes
        sample = int(min(n, max(100_000, rps * 100.0 / (steps + max(1, args.warmup)))))
        rps, sec, _ = cpu_reference_run(r1[:sample * READ_LEN], off[:sample], ln[:sample], threads, steps=steps, warmup=max(1, args.warmup))
        line = {"impl": "reference", "metric": METRIC, "value": rps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": rps, "unit": UNIT, "cores": threads, "kind": "port",
                                 "sample": "first %d reads of the workload per step (of %d), ASCII in host memory, C port of the "
                                           "reference's dcr() incl. revcomp, pthreads, after %d warm-up passes" % (sample, n, max(1, args.warmup))},
                "cpu_baseline_reference": reference_timing(),
                "e2e": {"value": rps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "note": "the reference is pure Python with un-installable native deps (acora, Levenshtein, biopython); "
                        "this arm times the oracle's C restatement of the same algorithm, which is pinned against "
                        "fixtures recorded from the unmodified reference; cpu_baseline_reference is the unmodified reference "
                        "itself, timed in the build container"}
        print(json.dumps(line), file=_JSON_OUT, flush=True)
        return

    # ---------------------------------------------------------------------------------------------
    import torch
    import torch.distributed as dist
    from decombinator_b200 import _lib

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the decombine path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    n = args.reads
    r1, off, ln = make_reads(info, rank * n, n, host_threads, args.sub_rate, args.n_rate)
    packed = _lib.pack_arrays(r1, off, ln, revcomp=True, n_threads=host_threads)
    vt, jt = info.tables()
    ctx = _lib.Context(vt, jt, device=local_rank)
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)
    ctx.upload(packed)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- resident: K steps of the kernels over the batch in HBM --------------------------------------
    with torch.cuda.stream(stream):
        # spin-up: a step is ~0.4 ms, so W steps alone end before the SM clocks have ramped from idle (measured: the
        # same binary at 19.7 or 25.1 G reads/s depending on it); run untimed passes for ~0.5 s first
        sampler = ClockSampler(local_rank) if rank == 0 else None   # from here on: the spin-up runs the timed region's load
        t_spin = time.perf_counter()
        while time.perf_counter() - t_spin < 0.5:
            for _ in range(50):
                ctx.run_resident()
            torch.cuda.synchronize()
        for _ in range(max(3, args.warmup)):
            ctx.run_resident()
        torch.cuda.synchronize()
        res0, cnt0 = ctx.download()
        n_deferred = ctx.last_deferred()
        ctx.timing_enable(True)
        ctx.timing_reset()
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        ev0.record(stream)
        for _ in range(args.steps):
            ctx.run_resident()
        ev1.record(stream)
        barrier()
        t1 = time.perf_counter()
        ms_total = ev0.elapsed_time(ev1)
        kms, klaunch = ctx.timing_get()
        ctx.timing_enable(False)
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, *ctx.download())
        clocks = sampler.stop(t_spin + 0.1, t1) if sampler else None   # samples under load: spin-up (same kernels) + timed region

        # ---- e2e_packed: host packed buffers -> results in host memory through dcb_decombine_batch ----
        for _ in range(3):
            ctx.decombine(packed, pinned=True)
        barrier()
        e0 = time.perf_counter()
        e2e_steps = args.steps
        for _ in range(e2e_steps):
            res_e, cnt_e = ctx.decombine(packed, pinned=True)   # synchronous: results are in host memory on return
        ep_ms = (time.perf_counter() - e0) * 1e3
        assert np.array_equal(res_e, res0) and np.array_equal(cnt_e, cnt0)
        # ---- e2e: ASCII reads in page-locked host memory -> results in host memory through dcb_decombine_ascii: what
        #      the reference arm starts from (text in memory; reverse complement, packing, matching inside the timed region)
        text = _lib.PinnedBytes(r1)
        for _ in range(3):
            ctx.decombine_ascii(text.a, None, None, True, uniform_len=READ_LEN, pinned=True)
        barrier()
        e0 = time.perf_counter()
        for _ in range(e2e_steps):
            res_a, cnt_a = ctx.decombine_ascii(text.a, None, None, True, uniform_len=READ_LEN, pinned=True)
        e_ms = (time.perf_counter() - e0) * 1e3
        assert np.array_equal(res_a, res0) and np.array_equal(cnt_a, cnt0)
        host_chunks, device_chunks = ctx.last_pack_shares()
        # the same with every chunk packed by the device (the whole text crosses the link): what the ceiling below bounds
        os.environ["DCB_HOST_SHARE"] = "0"
        ctx.decombine_ascii(text.a, None, None, True, uniform_len=READ_LEN, pinned=True)
        barrier()
        e0 = time.perf_counter()
        for _ in range(e2e_steps):
            res_d, cnt_d = ctx.decombine_ascii(text.a, None, None, True, uniform_len=READ_LEN, pinned=True)
        ed_ms = (time.perf_counter() - e0) * 1e3
        del os.environ["DCB_HOST_SHARE"]
        assert np.array_equal(res_d, res0) and np.array_equal(cnt_d, cnt0)
        # ---- the ceiling e2e runs against: page-locked host -> device copies of the same text, all ranks at once --------
        dev_buf = torch.empty(len(text.a), dtype=torch.uint8, device="cuda")
        host_t = torch.from_numpy(text.a)          # a view of the page-locked buffer
        for _ in range(2):
            dev_buf.copy_(host_t, non_blocking=True)
        barrier()
        c0 = time.perf_counter()
        for _ in range(5):
            dev_buf.copy_(host_t, non_blocking=True)
        torch.cuda.synchronize()
        h2d_gbps = 5 * len(text.a) / (time.perf_counter() - c0) / 1e9
        del dev_buf, host_t
        text.free()
    exact_name, h2d_bytes, slot_bytes = ctx.exact_kernel_name(), packed.h2d_bytes(), packed.slot_words * 4

    n_general = ctx.last_general()
    cfg2 = cfg3 = cfg4 = None
    if not args.no_workloads:
        ctx.close(); ctx = None
        packed.free()
        cfg2 = run_cfg2(args, rank, world, local_rank, host_threads, stream, barrier)
        cfg4 = run_cfg4(args, rank, world, local_rank, host_threads, stream, barrier)
        cfg3 = run_cfg3(args, rank, world, local_rank, host_threads, stream, barrier)
        packed = None

    if world > 1:
        t = torch.tensor([ms_total, e_ms, ep_ms, ed_ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total, e_ms, ep_ms, ed_ms = float(t[0]), float(t[1]), float(t[2]), float(t[3])
        t = torch.tensor([h2d_gbps], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        h2d_gbps = float(t[0])
        ok = torch.tensor([int(res0["status"].sum())], device="cuda", dtype=torch.int64)
        dist.all_reduce(ok)
        decombined = int(ok[0])
    else:
        decombined = int(res0["status"].sum())

    if rank == 0:
        value = world * n * args.steps / (ms_total / 1e3)
        e2e = world * n * e2e_steps / (e_ms / 1e3)
        e2e_dev = world * n * e2e_steps / (ed_ms / 1e3)
        bytes_per_read = (READ_LEN + 3) // 4 + 16
        exact_ms = kms[0] / max(1, klaunch[0])
        general_ms = kms[1] / max(1, klaunch[1])
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        achieved = bytes_per_read * n / (exact_ms / 1e3) / 1e9
        traffic = None   # dram__bytes_read.sum + dram__bytes_write.sum of one exact-kernel launch (ncu --set full), per read
        try:
            t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            traffic = float(t["dram_bytes_per_read"]) * n
        except Exception:
            pass
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32", "data": "synthetic", "config": config,
            "decombined_fraction": decombined / (world * n), "queued_by_exact_kernel": n_deferred / n,
            "deferred_to_general_kernel": n_general / n,
            "kernels_ms": {"dcb_exact_kernel": exact_ms, "dcb_halftag_kernel": kms[2] / max(1, klaunch[2]),
                           "dcb_general_kernel": general_ms},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": "profiles/traffic.json (one ncu --set full capture of this kernel, per read) x reads",
                         "kernel": exact_name, "bytes_per_read": bytes_per_read,
                         "peak_source": "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback 6650"},
            "e2e": {"value": e2e, "unit": UNIT,
                    "h2d_bytes_per_step": int(n * (READ_LEN * device_chunks + slot_bytes * host_chunks) / max(1, host_chunks + device_chunks)),
                    "d2h_bytes_per_step": int(n * 16 + 8 * _lib.NCOUNTERS), "steps": e2e_steps,
                    "call": "dcb_decombine_ascii: ASCII reads in page-locked host memory in (the reference arm's input), result records in "
                            "host memory out; the chunks are shared from both ends -- the device packs chunks from the front (their text crosses "
                            "the link), a worker with the host threads packs chunks of clean reads from the back (AVX-512, a quarter of the "
                            "bytes crosses) until the two meet",
                    "chunks_packed_by": {"host_threads": host_chunks, "device": device_chunks, "rank": 0},
                    "device_packed_only": {"value": e2e_dev, "unit": UNIT, "h2d_bytes_per_step": int(n * READ_LEN),
                                           "how": "DCB_HOST_SHARE=0: the whole text crosses the link",
                                           "frac_of_h2d_ceiling": e2e_dev / (h2d_gbps * 1e9 / READ_LEN * world)},
                    "h2d_ceiling": {"GBps_per_gpu": h2d_gbps, "GBps_all_gpus": h2d_gbps * world,
                                    "how": "torch copy_ of the same page-locked text to the device, all ranks at once, slowest rank",
                                    "reads_per_s_at_ceiling": h2d_gbps * 1e9 / READ_LEN * world,
                                    "e2e_frac_of_ceiling": e2e / (h2d_gbps * 1e9 / READ_LEN * world)}},
            "e2e_packed": {"value": world * n * e2e_steps / (ep_ms / 1e3), "unit": UNIT, "h2d_bytes_per_step": int(h2d_bytes),
                           "d2h_bytes_per_step": int(n * 16 + 8 * _lib.NCOUNTERS), "steps": e2e_steps,
                           "call": "dcb_decombine_batch: reads 2-bit packed on the host beforehand (outside the timed region)"},
            "gpu_launches": int(klaunch.sum()),
            "clocks": clocks,
        }
        if cfg2:
            line["workloads"] = {"cfg2": cfg2, "cfg3": cfg3, "cfg4": cfg4}
        if not args.no_cpu_baseline and world == 1:      # the CPU baseline is reported at N = 1 only
            threads = os.cpu_count() or 1
            sample = args.cpu_sample or min(n, 2_000_000 if threads < 16 else 10_000_000)
            rps, sec, _ = cpu_reference_run(r1[:sample * READ_LEN], off[:sample], ln[:sample], threads, steps=2, warmup=1)
            line["cpu_baseline"] = {"value": rps, "unit": UNIT, "cores": threads, "kind": "port",
                                    "sample": "first %d reads of rank 0's shard, mean of two passes after a warm-up pass, %.1f s each" % (sample, sec)}
            line["cpu_baseline_reference"] = reference_timing()
        print(json.dumps(line), file=_JSON_OUT, flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
