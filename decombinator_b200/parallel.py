"""Multi-GPU runs: one process per GPU (``torchrun``), ``torch.distributed`` for the plumbing.

* **decombine** shards trivially -- reads are independent (``dcr`` touches only the read and read-only tables,
  reference decombine.py:534-585; counters are sums): rank r analyses the contiguous index range
  ``shard_bounds(n, r, world)`` on its own GPU and stream, with NO data-path collective; rows are concatenated in
  rank order, which reproduces the reference's input-order ``.n12``.
* **collapse** has one real exchange step: the order-dependent grouping of collapse.py:595-682 only ever relates rows
  with the SAME barcode, so the surviving rows are repartitioned with ONE all-to-all keyed by ``hash(barcode) % world``
  (NCCL over NVLink on GPUs; gloo in the CPU tests).  Every rank then groups its own barcodes on its own GPU (the
  Levenshtein verdict batches), and the finished groups -- small: one per UMI -- are gathered on rank 0, put back in the
  reference's dict order by their insertion tick, and clustered there.

Nothing here has a CPU compute path: the kernels are reached through decombine.py / collapse.py as in a 1-GPU run.
"""
import collections as coll
import os
import pickle
import time
import zlib

import numpy as np
import torch
import torch.distributed as dist

from . import _lib
from . import collapse as C
from . import decombine as D


def init_from_env(backend=None):
    """Join the torchrun rendezvous (RANK / WORLD_SIZE / MASTER_*); NCCL when a GPU is visible, else gloo."""
    if dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world == 1:
        return 0, 1
    backend = backend or ("nccl" if torch.cuda.is_available() else "gloo")
    if backend == "nccl":
        local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:
        dist.init_process_group(backend)
    return dist.get_rank(), dist.get_world_size()


def _rank_world():
    return (dist.get_rank(), dist.get_world_size()) if dist.is_initialized() else (0, 1)


def _comm_device():
    return torch.device("cuda", torch.cuda.current_device()) if dist.is_initialized() and dist.get_backend() == "nccl" else torch.device("cpu")


def shard_bounds(n, rank, world):
    """Contiguous shard [lo, hi) of n items for `rank`: sizes differ by at most one, concatenation restores order."""
    base, extra = divmod(n, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def barcode_owner(barcode, world):
    """The rank that groups this barcode: a hash every process computes alike (not Python's salted hash())."""
    return zlib.crc32(barcode.encode("latin-1")) % world


def all_to_all_bytes(chunks):
    """chunks[r] = bytes for rank r  ->  list of the bytes every rank sent to this one.  Two collectives: the sizes
    (all_to_all_single of int64) and the payload (all_to_all_single with split sizes), on the GPU under NCCL."""
    rank, world = _rank_world()
    if world == 1:
        return [chunks[0]]
    dev = _comm_device()
    send_sizes = torch.tensor([len(c) for c in chunks], dtype=torch.int64, device=dev)
    recv_sizes = torch.empty(world, dtype=torch.int64, device=dev)
    dist.all_to_all_single(recv_sizes, send_sizes)
    rs = recv_sizes.tolist()
    payload = np.frombuffer(b"".join(chunks), dtype=np.uint8)
    send = torch.from_numpy(payload.copy() if len(payload) else np.zeros(0, dtype=np.uint8)).to(dev)
    recv = torch.empty(int(sum(rs)), dtype=torch.uint8, device=dev)
    dist.all_to_all_single(recv, send, output_split_sizes=rs, input_split_sizes=[len(c) for c in chunks])
    flat = recv.cpu().numpy().tobytes()
    out, pos = [], 0
    for n in rs:
        out.append(flat[pos:pos + n])
        pos += n
    return out


# ---------------------------------------------------------------------------------------------------------
# The collapse exchange: 64-byte records (SURVEY.md 8(d)), one NCCL all-to-all straight from device buffers.
#   u64 global row index | u64 barcode (up to 19 symbols x 3 bits over ACGTNSL, length in the top bits: what dcb_umi_pairs takes)
#   u8 v, u8 j, u16 vdel, u16 jdel | u8 inter-tag length, u8 insert offset in it, u8 insert length, u8 flags
#   33 B inter-tag sequence, 2 bits per base (<= 132 nt; -ln defaults to 130) | 5 B padding
# The barcode was located and quality-filtered on the source rank, so the 42-nt barcode region, the quality strings and
# the read id do not travel (they are only needed again for -wc / sampling analysis, which use the pickled rows below).
# ---------------------------------------------------------------------------------------------------------
RECORD = np.dtype([("idx", "<u8"), ("code", "<u8"), ("v", "u1"), ("j", "u1"), ("vdel", "<u2"), ("jdel", "<u2"), ("seq_len", "u1"),
                   ("ins_off", "u1"), ("ins_len", "u1"), ("flags", "u1"), ("seq", "u1", (33,)), ("pad", "u1", (5,))])
assert RECORD.itemsize == 64
_SYM = {c: i for i, c in enumerate("ACGTNSL")}
_B2 = {"A": 0, "C": 1, "G": 2, "T": 3}
_PACK4 = {a + b + c + d: _B2[a] | (_B2[b] << 2) | (_B2[c] << 4) | (_B2[d] << 6) for a in "ACGT" for b in "ACGT" for c in "ACGT" for d in "ACGT"}
_UNPACK4 = ["".join("ACGT"[(v >> (2 * k)) & 3] for k in range(4)) for v in range(256)]


def encode_records(kept):
    """[(global row index, barcode, inter-tag seq, dcretc), ...] -> RECORD array, or None when a row does not fit the record
    (a symbol outside ACGT in the inter-tag sequence, more than 132 nt, a field out of range): the caller then falls back
    to pickled rows."""
    import ast
    out = np.zeros(len(kept), dtype=RECORD)
    try:
        for t, (idx, barcode, seq, dcretc) in enumerate(kept):
            v, j, vdel, jdel, ins = ast.literal_eval(dcretc.split("|", 1)[0])
            off = seq.find(ins)
            n = len(seq)
            if n > 132 or off < 0 or len(barcode) > 19:
                return None
            code = len(barcode) << 58
            for k, ch in enumerate(barcode):
                code |= _SYM[ch] << (3 * k)
            r = out[t]
            r["idx"], r["code"], r["v"], r["j"], r["vdel"], r["jdel"] = idx, code, int(v), int(j), int(vdel), int(jdel)
            r["seq_len"], r["ins_off"], r["ins_len"] = n, off, len(ins)
            padded = seq + "A" * (-n % 4)
            r["seq"][:len(padded) // 4] = [_PACK4[padded[k:k + 4]] for k in range(0, len(padded), 4)]
    except (KeyError, ValueError, OverflowError, SyntaxError):
        return None
    return out


def decode_records(rec):
    """RECORD array -> the (global row index, barcode, inter-tag seq, dcretc) tuples the grouping takes; the dcretc of a
    decoded row is ``str(dcr)|seq||`` (quality string and read id did not travel)."""
    rows = []
    for r in rec:
        code, n = int(r["code"]), int(r["seq_len"])
        barcode = "".join("ACGTNSL"[(code >> (3 * k)) & 7] for k in range(code >> 58))
        seq = "".join(_UNPACK4[b] for b in r["seq"][:(n + 3) // 4].tolist())[:n]
        ins = seq[int(r["ins_off"]):int(r["ins_off"]) + int(r["ins_len"])]
        dcr = [str(int(r["v"])), str(int(r["j"])), str(int(r["vdel"])), str(int(r["jdel"])), ins]
        rows.append((int(r["idx"]), barcode, seq, "|".join([str(dcr), seq, "", ""])))
    return rows


def record_owner(codes, world):
    """Destination rank of every record: a multiplicative hash of the barcode code (the same on every rank)."""
    h = (np.asarray(codes, dtype=np.uint64) * np.uint64(0x9E3779B97F4A7C15)) >> np.uint64(40)
    return (h % np.uint64(world)).astype(np.int64)


_last_exchange = {}


def exchange_records(rec):
    """All-to-all of RECORD rows keyed by the barcode hash: every rank gets the records whose barcode it owns.  The send
    buffer (records ordered by destination) and the receive buffer are DEVICE tensors under NCCL -- the collective moves
    them GPU to GPU over NVLink --, CPU tensors under gloo.  Two collectives: the counts, then the payload."""
    rank, world = _rank_world()
    if world == 1:
        return rec
    dev = _comm_device()
    owner = record_owner(rec["code"], world)
    order = np.argsort(owner, kind="stable")
    send_counts = np.bincount(owner, minlength=world).astype(np.int64)
    send = torch.from_numpy(np.ascontiguousarray(rec[order]).view(np.uint8).reshape(-1, 64).copy()).to(dev)
    sc = torch.from_numpy(send_counts).to(dev)
    rc = torch.empty(world, dtype=torch.int64, device=dev)
    dist.all_to_all_single(rc, sc)
    recv_counts = rc.tolist()
    recv = torch.empty((int(sum(recv_counts)), 64), dtype=torch.uint8, device=dev)
    timed = dev.type == "cuda"
    if timed:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    dist.all_to_all_single(recv, send, output_split_sizes=recv_counts, input_split_sizes=send_counts.tolist())
    if timed:
        e1.record()
        torch.cuda.synchronize()
        _last_exchange.update(ms=e0.elapsed_time(e1), sent_bytes=int(send.numel()), received_bytes=int(recv.numel()))
    return np.ascontiguousarray(recv.cpu().numpy()).view(RECORD).reshape(-1)


def all_gather_codes(codes):
    """Every rank's UMI codes (uint64) concatenated in rank order, on every rank: one all_gather of the counts and one of
    the padded payload (device tensors under NCCL)."""
    rank, world = _rank_world()
    codes = np.ascontiguousarray(codes, dtype=np.uint64)
    if world == 1:
        return codes, [len(codes)]
    dev = _comm_device()
    n = torch.tensor([len(codes)], dtype=torch.int64, device=dev)
    sizes = [torch.empty(1, dtype=torch.int64, device=dev) for _ in range(world)]
    dist.all_gather(sizes, n)
    sizes = [int(x.item()) for x in sizes]
    width = max(max(sizes), 1)
    mine = torch.zeros(width, dtype=torch.int64, device=dev)
    mine[:len(codes)] = torch.from_numpy(codes.view(np.int64)).to(dev)
    parts = [torch.empty(width, dtype=torch.int64, device=dev) for _ in range(world)]
    dist.all_gather(parts, mine)
    flat = np.concatenate([p[:k].cpu().numpy() for p, k in zip(parts, sizes)]).view(np.uint64)
    return flat, sizes


def _sum_counters(local):
    """Counter summed over ranks (every rank gets the total)."""
    rank, world = _rank_world()
    if world == 1:
        return coll.Counter(local)
    parts = [None] * world
    dist.all_gather_object(parts, dict(local))
    total = coll.Counter()
    for p in parts:
        total.update(p)
    return total


def decombinator_shard(inputargs):
    """This rank's part of ``decombinator(inputargs)``: -> (rows of its shard, global row index of the first one).
    ``decombine.counts`` ends up holding the whole-job totals on every rank."""
    rank, world = _rank_world()
    if world == 1:
        return D.decombinator(dict(inputargs)), 0
    args = dict(inputargs)
    args["shard"] = (rank, world)
    # No rank writes the summary from inside decombinator(): its counters cover one shard.  Rank 0 writes it below from
    # the summed counters.  The FASTQ check runs on rank 0 and its verdict is broadcast, so that a bad input makes EVERY
    # rank raise instead of leaving the others waiting in the next collective.
    args["suppresssummary"] = True
    args["dontcheck"] = True
    want_summary = inputargs["suppresssummary"] == False  # noqa: E712
    t0 = time.time()
    verdict = [None]
    if rank == 0 and inputargs["dontcheck"] == False:  # noqa: E712
        try:
            from time import strftime
            D.import_tcr_info(dict(inputargs))                      # sets the chain the stub summary is named after
            samplenam, date = D.sample_name(inputargs), strftime("%Y_%m_%d")
            logpath = summaryname = None
            if want_summary:
                logpath, summaryname = D.summary_location(inputargs, samplenam, date)
            D.check_fastq(inputargs, D.opener_check(inputargs), summaryname, logpath, date, samplenam)
        except BaseException as exc:  # noqa: BLE001 -- re-raised on every rank
            verdict[0] = exc
    dist.broadcast_object_list(verdict, src=0)
    if verdict[0] is not None:
        raise verdict[0]
    rows = D.decombinator(args)
    sizes = [None] * world
    dist.all_gather_object(sizes, len(rows))
    skip = ("start_time", "end_time", "pc_decombined", "chain_detected")
    total = _sum_counters({k: v for k, v in D.counts.items() if k not in skip})
    for k, v in total.items():
        D.counts[k] = v
    if rank == 0 and want_summary:
        from time import strftime
        samplenam, date = D.sample_name(inputargs), strftime("%Y_%m_%d")
        logpath, summaryname = D.summary_location(inputargs, samplenam, date)
        D.write_summary(inputargs, summaryname, logpath, date, samplenam, time.time() - t0)
    return rows, sum(sizes[:rank])


def gather_rows(rows):
    """Rank 0 gets the rows of all ranks concatenated in rank order (= input order); the others get []."""
    rank, world = _rank_world()
    if world == 1:
        return rows
    parts = [None] * world if rank == 0 else None
    dist.gather_object(rows, parts, dst=0)
    return [r for p in parts for r in p] if rank == 0 else []


def decombinator_sharded(inputargs):
    """``decombinator(inputargs)`` over all ranks: rank 0 returns every row in input order (and ``counts`` holds the
    whole-job totals), the other ranks return [].  Each rank packs and analyses only its own shard of the reads."""
    rows, _ = decombinator_shard(inputargs)
    return gather_rows(rows)


def collapsinator_sharded(inputargs, data=None, first_index=0, n_total=None):
    """``collapsinator`` over all ranks.  `data`: THIS rank's shard of the decombined rows (global index of its first
    row = first_index) -- or, for the ``collapse`` sub-command, nothing: every rank then reads its own slice of the file.
    Rank 0 returns the ``.freq`` rows; the others return []."""
    rank, world = _rank_world()
    if world == 1:
        return C.collapsinator(inputargs, data=data)
    inputargs = dict(inputargs)
    if inputargs["extension"] == "n12":
        inputargs["extension"] = "freq"
    C.counts = coll.Counter()
    C.counts["start_time"] = time.time()
    qp = [inputargs["minbcQ"], inputargs["bcQbelowmin"], inputargs["avgQthreshold"]]
    frac = inputargs["percentlevdist"] / 100
    from_file = inputargs["command"] == "collapse"
    if from_file:
        import gzip
        opener = gzip.open if inputargs["infile"].endswith(".gz") else open
        verdict = [True]
        if rank == 0 and not inputargs["dontcheckinput"]:
            verdict[0] = bool(C.check_dcr_file(inputargs["infile"], opener))
        dist.broadcast_object_list(verdict, src=0)           # every rank stops on a bad file, none is left in a collective
        if not verdict[0]:
            raise SystemExit("Please check that file contains suitable Decombinator output for collapsing.")
        with opener(inputargs["infile"], "rt") as fh:
            lines = fh.readlines()
        lo, hi = shard_bounds(len(lines), rank, world)
        data, first_index = lines[lo:hi], lo
    # 1. per-row filters on the source rank
    kept, dcr_counts, _ = C._filter_rows(data, inputargs, qp, True, from_file, first_index=first_index)
    # 2. ONE all-to-all keyed by hash(exact barcode): 64-byte records from device buffers.  Rows that do not fit a record
    #    (and runs that need the quality strings / read ids again: -wc, sampling analysis) travel as pickled rows instead;
    #    the ranks agree on the form first.
    rec = None if (inputargs["writeclusters"] or inputargs["sampling_analysis"]) else encode_records(kept)
    flag = torch.tensor([0 if rec is None else 1], dtype=torch.int64, device=_comm_device())
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    _last_exchange.clear()
    _last_exchange["form"] = "records" if int(flag.item()) else "pickled rows"
    if int(flag.item()):
        mine = decode_records(exchange_records(rec))
    else:
        outbox = [[] for _ in range(world)]
        for item in kept:
            outbox[barcode_owner(item[1], world)].append(item)
        inbox = all_to_all_bytes([pickle.dumps(x, protocol=4) for x in outbox])
        mine = [item for blob in inbox for item in pickle.loads(blob)]
    mine.sort(key=lambda item: item[0])                      # global input order within every barcode
    # 3. group this rank's barcodes (Levenshtein verdicts on this rank's GPU)
    groups, dropped, dead = C._group_rows(mine, frac)
    local = {"groups": groups, "dropped": dropped, "dead": dead, "dcr_counts": dict(dcr_counts)}
    parts = [None] * world if rank == 0 else None
    dist.gather_object(local, parts, dst=0)
    totals = _sum_counters({k: v for k, v in C.counts.items() if k != "start_time"})
    # 3b. the UMI neighbour search over ALL groups, split over the GPUs: an all-gather of the barcode codes (rank order), every
    #     rank verifies its share of the deletion-variant runs on its own GPU, the shares are gathered on rank 0
    #     (barcodes with symbols outside ACGTNSL -- IUPAC codes from the host's fuzzy path -- have no rank-independent code:
    #     rank 0 then searches alone, as a 1-GPU run does)
    try:
        local_codes, codable = _lib.encode_umis_fixed([g[1] for g in groups]), 1
    except _lib.DcbError:
        local_codes, codable = np.zeros(0, dtype=np.uint64), 0
    flag = torch.tensor([codable], dtype=torch.int64, device=_comm_device())
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    split_search = bool(int(flag.item()))
    shares = None
    if split_search:
        all_codes, sizes = all_gather_codes(local_codes)
        if len(all_codes) > 1:
            row, col = C._gpu().umi_pairs(all_codes, inputargs["bcthreshold"], part=rank, n_parts=world)
        else:
            row = col = np.zeros(0, dtype=np.int64)
        shares = [None] * world if rank == 0 else None
        dist.gather_object((row, col), shares, dst=0)
    if rank != 0:
        return []
    # 4. rank 0: the reference's dict order back from the ticks, then clustering and counting as in a 1-GPU run
    for k, v in totals.items():
        C.counts[k] = v
    all_dcr = coll.Counter()
    for p in parts:
        all_dcr.update(p["dcr_counts"])
    gathered = [g for p in parts for g in p["groups"]]            # rank order = the order of the gathered codes
    barcode_dcretc = C._groups_to_dict(gathered, all_dcr, sum(p["dropped"] for p in parts), sum(p["dead"] for p in parts))

    def find_pairs(umi_protoseq_tuple, barcode_threshold, dont_count):
        """The pairs of the split search, renumbered from the gathered (rank) order to the dict's order and sorted row-major."""
        n_groups = len(gathered)
        if n_groups == 0:
            raise ValueError("No UMIs to cluster, check .n12 file for errors")
        order = sorted(range(n_groups), key=lambda g: gathered[g][0])           # dict order = ascending tick (stable)
        pos = np.empty(n_groups, dtype=np.int64)
        pos[np.asarray(order, dtype=np.int64)] = np.arange(n_groups, dtype=np.int64)
        r = np.concatenate([np.asarray(x[0], dtype=np.int64) for x in shares])
        c = np.concatenate([np.asarray(x[1], dtype=np.int64) for x in shares])
        a, b = pos[r], pos[c]
        key = np.unique(np.minimum(a, b) * np.int64(n_groups) + np.maximum(a, b))
        print("Clustering UMIs...")
        print("  ", n_groups, "unique UMIs")
        print("  ", len(key), "UMIs within edit distance of", barcode_threshold)
        return C._PairList(key // n_groups, key % n_groups)

    file_id = inputargs["infile"].split("/")[-1].split(".")[0]
    out_data, _, sizes = C._count_clusters(barcode_dcretc, inputargs, inputargs["bcthreshold"], frac, True, "", file_id,
                                           find_pairs if split_search else None)
    C.counts["end_time"] = time.time()
    C.counts["time_taken_total_s"] = C.counts["end_time"] - C.counts["start_time"]
    if inputargs["suppresssummary"] == False:  # noqa: E712
        C._write_summary(inputargs, file_id, sizes)
    return out_data
