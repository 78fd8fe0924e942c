"""Two ranks, two GPUs, NCCL: the collapse exchange (64-byte records through all_to_all_single on device tensors), the
UMI-code all-gather and the sharded decombine -> collapse pipeline must reproduce the single-process results recorded from
the reference.  Needs two devices: skipped on a machine with one GPU."""
import gzip
import json
import os
import shutil
import socket
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _n_gpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


def _worker(rank, world, port, tmp, out_path):
    for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
        if p not in sys.path:
            sys.path.insert(0, p)
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import numpy as np
    import torch
    import torch.distributed as dist
    from decombinator_b200 import collapse, decombine as D, io, parallel
    parallel.init_from_env("nccl")
    assert dist.get_backend() == "nccl" and torch.cuda.current_device() == rank
    # 1. recorded collapse runs, rows sharded over the two ranks
    with gzip.open(os.path.join(ROOT, "tests", "golden", "collapse_cases.json.gz"), "rt") as fh:
        cases = json.load(fh)["cases"]
    results = []
    for case in cases:
        rows = [list(r) for r in case["rows"]]
        lo, hi = parallel.shard_bounds(len(rows), rank, world)
        out = parallel.collapsinator_sharded(dict(case["args"]), data=rows[lo:hi], first_index=lo)
        assert parallel._last_exchange["form"] == "records"
        assert parallel._last_exchange.get("sent_bytes", 0) % 64 == 0 and "ms" in parallel._last_exchange   # device tensors, timed by CUDA events
        results.append(out)
    codes, sizes = parallel.all_gather_codes(np.arange(5 + rank, dtype=np.uint64) + np.uint64(1000 * rank))
    assert sizes == [5, 6] and codes.tolist() == list(range(5)) + [1000 + k for k in range(6)]
    # 2. the TINY pipeline: decombine sharded (no collective), collapse with the exchange, translate on rank 0
    args = io.create_args_dict(infile=os.path.join(tmp, "TINY_1.fq"), chain="b", bc_read="R2", dontgzip=True, dontcount=True,
                               outpath=os.path.join(tmp, "out") + os.sep, tagfastadir="Decombinator-Tags-FASTAs", command="pipeline",
                               oligo="M13")
    from decombinator_b200 import pipeline
    pipeline.run(args)
    if rank == 0:
        json.dump({"freq": results, "vj": int(D.counts["vj_count"])}, open(out_path, "w"))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(_n_gpus() < 2, reason="needs two GPUs")
def test_two_gpus_nccl_exchange_and_pipeline(golden_dir, tmp_path):
    import torch.multiprocessing as mp
    for f in ("TINY_1.fq", "TINY_2.fq"):
        shutil.copy(os.path.join(golden_dir, f), tmp_path / f)
    (tmp_path / "out").mkdir()
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    out_path = str(tmp_path / "out.json")
    mp.spawn(_worker, args=(2, port, str(tmp_path), out_path), nprocs=2, join=True)
    got = json.load(open(out_path))
    with gzip.open(os.path.join(golden_dir, "collapse_cases.json.gz"), "rt") as fh:
        cases = json.load(fh)["cases"]
    assert got["freq"] == [c["freq"] for c in cases]
    assert got["vj"] == 48
    for ext in ("n12", "freq", "tsv"):
        assert (tmp_path / "out" / ("dcr_TINY_1_beta." + ext)).read_bytes() == open(os.path.join(golden_dir, "dcr_TINY_1_beta." + ext), "rb").read()
