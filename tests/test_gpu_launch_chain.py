"""The resident step as one chain of launches (dcb_run_resident, csrc/decombine.cu).

By default the kernels of a resident step are launched with programmatic dependent launch: each one is scheduled while
its predecessor finishes, and the next step's exact kernel while this step's general kernel finishes.  Nothing else may
change: no memset sits between the steps, so the steps alternate between two counter sets, each step's general kernel
clearing the set of the step after it.  DCB_PDL=0 launches the same kernels plainly behind a memset of the counters.

Here, on reads whose queues are not empty (1 % substitutions + 0.1 % N, the configs[2] shape, so that the half-tag and
general kernels do real work behind the chain), the two settings must give the same records, counters and exact-kernel
queue counts after every step, however many steps run back to back; the resident steps must stay right when the chunked
path (dcb_decombine_ascii, which counts in the first set) or an empty batch comes in between on the same context; and the
device-side timing must count one launch of each kernel per step."""
import functools

import numpy as np
import pytest

from decombinator_b200 import _lib, tags
from helpers import synth_batch

pytestmark = pytest.mark.gpu

N, L = 1 << 20, 250
# chain analysed, the chains of the mixed file
SHAPES = {
    "cfg2": (("human", "extended", "a"), (("human", "extended", "a"), ("human", "extended", "b")), 0.01, 0.001),
    "cfg4": (("mouse", "original", "g"), (("mouse", "original", "g"), ("mouse", "original", "d")), 0.005, 0.0),
}


@functools.lru_cache(maxsize=None)
def _batch(shape):
    chain, mix, sub, nrate = SHAPES[shape]
    infos = [tags.load(*c) for c in mix]
    r1, off, ln = synth_batch(infos[0], N, L, sub, nrate, 0.0, seed=20260003,
                              sets=[(i.v_regions, i.j_regions) for i in infos])
    return tags.load(*chain), r1, off, ln


def _step(ctx, monkeypatch, pdl, steps=1):
    monkeypatch.setenv("DCB_PDL", pdl)
    for _ in range(steps):
        ctx.run_resident()
    res, cnt = ctx.download()
    return res, cnt, ctx.last_deferred(), ctx.last_general()


def _same(a, b, what):
    assert np.array_equal(a[0], b[0]), what + ": records differ"
    assert np.array_equal(a[1], b[1]), what + ": counters differ"
    assert a[2] == b[2], what + ": reads queued by the exact kernel differ (%d vs %d)" % (a[2], b[2])
    # What the half-tag kernel passes on is not a property of the reads alone: a read goes on when its warp's work lists
    # are full, and which reads share a warp follows the order of the exact kernel's atomic appends, which differs from
    # run to run in either setting (the records do not).  Without the half-tag kernel the two counts are one.
    if b[3] == b[2]:
        assert a[3] == b[3], what + ": reads that reached the general kernel differ (%d vs %d)" % (a[3], b[3])
    else:
        assert 0 < a[3] < a[2], what + ": reads that reached the general kernel: %d of %d queued" % (a[3], a[2])


@pytest.mark.parametrize("shape,force_general", [("cfg2", 0), ("cfg2", 1), ("cfg2", 2), ("cfg2", 3), ("cfg4", 0)])
def test_chained_steps_match_plain_launches(monkeypatch, shape, force_general):
    info, r1, off, ln = _batch(shape)
    packed = _lib.pack_arrays(r1, off, ln, revcomp=True)
    vt, jt = info.tables()
    ctx = _lib.Context(vt, jt, device=0, force_general=force_general)
    ctx.upload(packed)
    plain = _step(ctx, monkeypatch, "0")
    if force_general != 1:
        assert plain[2] > 0, "nothing queued: the follow-up kernels would not run behind the chain"
    for i, steps in enumerate((1, 1, 2, 3, 8, 17)):          # odd and even runs: both counter sets, either parity
        _same(_step(ctx, monkeypatch, "1", steps), plain, "%d chained steps (run %d)" % (steps, i))
    _same(_step(ctx, monkeypatch, "0"), plain, "plain step after chained ones")
    _same(_step(ctx, monkeypatch, "1", 5), plain, "chained steps after a plain one")
    # the chunked path reports the same, and the resident steps after it too (the chunked path counts in the first set)
    res_b, cnt_b = ctx.decombine(packed)
    assert np.array_equal(res_b, plain[0]) and np.array_equal(cnt_b, plain[1])
    _same(_step(ctx, monkeypatch, "1", 3), plain, "chained steps after decombine_batch")
    ctx.close(); packed.free()


def test_chained_steps_alternate_with_decombine_ascii(monkeypatch):
    info, r1, off, ln = _batch("cfg2")
    packed = _lib.pack_arrays(r1, off, ln, revcomp=True)
    vt, jt = info.tables()
    ctx = _lib.Context(vt, jt, device=0)
    ctx.upload(packed)
    plain = _step(ctx, monkeypatch, "0")
    for rnd in range(4):
        monkeypatch.setenv("DCB_PDL", "1")
        res_a, cnt_a = ctx.decombine_ascii(r1, None, None, True, uniform_len=L)
        assert np.array_equal(res_a, plain[0]) and np.array_equal(cnt_a, plain[1]), "decombine_ascii, round %d" % rnd
        assert ctx.last_deferred() == plain[2], "decombine_ascii queue count, round %d" % rnd
        # the resident steps now run on the batch decombine_ascii packed on the device: the same reads
        _same(_step(ctx, monkeypatch, "1", 1 + rnd), plain, "chained steps after decombine_ascii, round %d" % rnd)
        if rnd == 2:
            ctx.upload(packed)
            _same(_step(ctx, monkeypatch, "1", 2), plain, "chained steps after a new upload")
    ctx.close(); packed.free()


def test_chained_steps_around_an_empty_batch(monkeypatch):
    """An empty batch launches no kernel, so no general kernel clears the next step's counter set: the steps before and
    after it must still count from zero (and the exact kernel append to an empty queue)."""
    info, r1, off, ln = _batch("cfg2")
    packed = _lib.pack_arrays(r1, off, ln, revcomp=True)
    empty = _lib.pack_strings([], revcomp=True)
    vt, jt = info.tables()
    ctx = _lib.Context(vt, jt, device=0)
    ctx.upload(packed)
    plain = _step(ctx, monkeypatch, "0")
    for pdl in ("1", "0", "1"):
        for steps in (1, 2):
            ctx.upload(packed)
            _same(_step(ctx, monkeypatch, pdl, steps), plain, "DCB_PDL=%s, %d steps before an empty batch" % (pdl, steps))
            ctx.upload(empty)
            res, cnt, deferred, general = _step(ctx, monkeypatch, pdl, steps)
            assert len(res) == 0 and not cnt.any() and deferred == 0 and general == 0, "DCB_PDL=%s: empty batch" % pdl
            ctx.upload(packed)
            _same(_step(ctx, monkeypatch, pdl, steps), plain, "DCB_PDL=%s, %d steps after an empty batch" % (pdl, steps))
    ctx.close(); packed.free(); empty.free()


def test_pdl_setting_is_checked(monkeypatch):
    info, r1, off, ln = _batch("cfg2")
    n = 4096
    packed = _lib.pack_arrays(r1[:n * L], off[:n], ln[:n], revcomp=True)
    vt, jt = info.tables()
    ctx = _lib.Context(vt, jt, device=0)
    ctx.upload(packed)
    monkeypatch.setenv("DCB_PDL", "2")
    with pytest.raises(_lib.DcbError, match="DCB_PDL"):
        ctx.run_resident()
    monkeypatch.setenv("DCB_PDL", "1")
    ctx.run_resident()
    ctx.download()
    ctx.close(); packed.free()


@pytest.mark.parametrize("pdl", ["0", "1"])
def test_timing_counts_one_launch_per_kernel_per_step(monkeypatch, pdl):
    info, r1, off, ln = _batch("cfg2")
    packed = _lib.pack_arrays(r1, off, ln, revcomp=True)
    vt, jt = info.tables()
    ctx = _lib.Context(vt, jt, device=0)
    ctx.upload(packed)
    monkeypatch.setenv("DCB_PDL", pdl)
    ctx.run_resident()
    ctx.timing_enable(True)
    ctx.timing_reset()
    steps = 25
    for _ in range(steps):
        ctx.run_resident()
    ms, launches = ctx.timing_get()
    assert list(launches) == [steps, steps, steps, 0], launches     # exact, general, half-tag; slot 3 unused
    assert all(ms[i] > 0 for i in range(3)), ms
    assert ms[0] / steps < 50.0, ms                                 # per launch: a 1 M-read batch, not seconds
    ctx.timing_reset()
    ms, launches = ctx.timing_get()
    assert not launches.any() and not ms.any()
    # timing off: nothing is counted
    ctx.timing_enable(False)
    ctx.run_resident()
    ms, launches = ctx.timing_get()
    assert not launches.any()
    ctx.close(); packed.free()
