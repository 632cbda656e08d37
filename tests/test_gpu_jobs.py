"""Jobs on the device (fadegpu_submit_pairs / fadegpu_submit_regions / fadegpu_job_wait): with 1 to 6 jobs in flight,
every job's records and ops are byte-equal to the synchronous call on the same input (a sample also against the
scalar oracle); mixed queues waited out of order, many launches, the caller's arrays overwritten after submit,
resubmitted jobs, errors found on the device, every FADEGPU_E_STATE case, FADEGPU_F_SYNC_SUBMIT, lifetimes and stats.
Run with `pytest -m gpu` on a B200."""
import ctypes as C
import os
import random

import numpy as np
import pytest

from fade_b200 import Context, Job, _lib, api, default_params, sim
from fade_b200._lib import FadeGpuError
from oracle import oracle as orc
from test_gpu_pairs import _census, _check, _oracle
from test_gpu_regions import _regions, _wild_contigs

pytestmark = pytest.mark.gpu

E_ARG, E_STATE = -1, -4
SAME_STATS = ("n_reads", "n_aligned", "n_generic", "cells", "h2d_bytes", "d2h_bytes", "kernel_launches", "n_oversize",
              "scratch_bytes", "host_threads")
MODES = [("pairs", False), ("pairs", True), ("regions", False), ("regions", True)]


def _sync(ctx, kind, score_only, x):
    if kind == "pairs":
        q, qo, t, to = x
        f = ctx.score_pairs if score_only else ctx.align_pairs
        return f(q, t, query_offsets=qo, target_offsets=to)
    qs, tids, starts, ends, strands = x
    f = ctx.score_regions if score_only else ctx.align_regions
    return f(qs, tids, starts, ends, strands)


def _submit(job, kind, score_only, x):
    if kind == "pairs":
        q, qo, t, to = x
        return job.submit_pairs(q, t, score_only=score_only, query_offsets=qo, target_offsets=to)
    qs, tids, starts, ends, strands = x
    return job.submit_regions(qs, tids, starts, ends, strands, score_only=score_only)


def _equal(got, want, stats=True):
    assert type(got) is type(want) and got.records.tobytes() == want.records.tobytes()
    if isinstance(want, api.PairResults):
        assert got.ops.shape == want.ops.shape and got.ops.tobytes() == want.ops.tobytes()
    if stats:
        for f in SAME_STATS:
            assert getattr(got.stats, f) == getattr(want.stats, f), f
        if want.stats.n_reads:
            assert got.stats.host_submit_ms > 0 and got.stats.total_ms > 0 and got.stats.kernel_ms >= 0


def _pair_chunks(packed, sizes):
    q, qo, t, to = packed
    out, k = [], 0
    for n in sizes:
        out.append((q, qo[k:k + n + 1].copy(), t, to[k:k + n + 1].copy()))
        k += n
    return out


def _region_chunks(regs, sizes):
    out, k = [], 0
    for n in sizes:
        out.append(tuple(list(a[k:k + n]) for a in regs))
        k += n
    return out


@pytest.fixture(scope="module")
def c1():
    """a ctx with C1's reference, C1's census pairs and C1's aligned reads as regions on both strands"""
    names, contigs, cfg, n = sim.config_c1()
    rd = sim.make_reads(cfg, 0, n, contigs)
    W = 300
    with Context(0) as ctx:
        ctx.load_reference(names, [c.tobytes() for c in contigs])
        b = ctx.alloc_batch(rd.n, int(rd.seq_off[rd.n]))
        b.fill(rd.seq4, rd.seq_off, rd.l_qseq, rd.tid, rd.pos, rd.aligned_len, rd.clip_left, rd.clip_right).run()
        al = np.nonzero(b.flags[:rd.n] & api.R_ALIGNED)[0]
        starts = b.win_start[al].astype(np.int64).tolist()
        b.close()
        qs, strands = [], []
        for r in al:
            so, lq = int(rd.seq_off[r]), int(rd.l_qseq[r])
            fwd = orc.decode_nt16(rd.seq4[so:so + (lq + 1) // 2], lq)
            qs.append(fwd if r % 2 else orc.revcomp_nt16(rd.seq4[so:so + (lq + 1) // 2], lq))
            strands.append(1 if r % 2 else 0)
        ends = np.minimum(rd.pos[al] + rd.aligned_len[al] + W, len(contigs[0])).tolist()
        regions = (qs, rd.tid[al].tolist(), starts, ends, strands)
        packed, pqs, pts = _census(11, 60_000, 72, 160)
        yield ctx, {"pairs": (packed, pqs, pts), "regions": regions}


SIZES = {"pairs": [4000, 17000, 1, 9000, 23000, 6000]}


@pytest.mark.parametrize("kind,score_only", MODES)
@pytest.mark.parametrize("depth", [1, 2, 3, 6])
def test_jobs_equal_the_synchronous_call(c1, kind, score_only, depth):
    ctx, data = c1
    if kind == "pairs":
        chunks = _pair_chunks(data["pairs"][0], SIZES["pairs"])
    else:
        n = len(data["regions"][0])
        assert n > 1000
        cut = sorted({0, n} | {n * f // 100 for f in (7, 30, 31, 55, 80)})
        chunks = _region_chunks(data["regions"], [b - a for a, b in zip(cut, cut[1:])])
    want = [_sync(ctx, kind, score_only, x) for x in chunks]
    jobs = [Job(ctx) for _ in range(depth)]
    got, flight = [None] * len(chunks), []
    for k, x in enumerate(chunks):
        if len(flight) == depth:
            i = flight.pop(0)
            got[i] = jobs[i % depth].wait()
        _submit(jobs[k % depth], kind, score_only, x)
        flight.append(k)
    for i in flight:
        got[i] = jobs[i % depth].wait()
    for g, w in zip(got, want):
        _equal(g, w)
    if kind == "pairs" and not score_only and depth == 3:     # a sample of the first chunk against fo_sw_trace
        _, pqs, pts = data["pairs"]
        idx = list(range(0, SIZES["pairs"][0], 7))
        _check(got[0], _oracle([pqs[k] for k in idx], [pts[k] for k in idx]), idx)
    for j in jobs:
        j.close()


@pytest.fixture(scope="module")
def wild():
    contigs = _wild_contigs(7, [300_000, 2_600_000, 90_000])
    with Context(0) as ctx:
        ctx.load_reference(["c0", "c1", "c2"], contigs)
        yield ctx, contigs


def _mixed(contigs):
    """(kind, score_only, inputs) of very different sizes: an empty job, oversize items, generic-kernel items
    (wildcards, queries over 304) and windows past 4,000 columns, planted and random"""
    rng = random.Random(23)
    big = [contigs[1]]
    small = _regions(rng, contigs, [rng.randrange(1, 300) for _ in range(2000)], lambda ql: rng.randrange(ql, 1500))
    wide = _regions(rng, big, [rng.choice((60, 150, 300)) for _ in range(8)], lambda ql: rng.randrange(4_001, 9_000))
    wide = ([q for q in wide[0]], [1] * 8, wide[2], wide[3], wide[4])
    gen = _regions(rng, big, list(range(305, 700, 25)), lambda ql: rng.randrange(300, 1500))
    gen = (gen[0] + ["ACGT" * 250, "", "ACGT"], [1] * len(gen[0]) + [1, 0, 0], gen[2] + [100, 5, 7],
           gen[3] + [2_200_100, 50, 7], gen[4] + [0, 1, 1])                   # + oversize, empty query, empty interval
    many = _regions(rng, contigs, [rng.randrange(20, 260) for _ in range(30_000)], lambda ql: rng.randrange(ql, 900))
    pq = ["".join(rng.choice("ACGT") for _ in range(rng.randrange(1, 300))) for _ in range(3000)]
    pq = [q[:-1] + "R" if k % 50 == 0 else q for k, q in enumerate(pq)]                  # wildcards: generic kernel
    pt = ["".join(rng.choice("ACGTNRYK") for _ in range(rng.randrange(1, 6000 if k % 60 == 0 else 700)))
          for k in range(3000)]
    pq += ["ACGT" * 300, "", "A"]
    pt += ["C" * 2_000_000, "ACGT", ""]                                       # oversize, empty query, empty target
    pairs = api.pack_pairs(pq, pt)
    empty = api.pack_pairs([], [])
    return [("regions", False, many), ("pairs", True, empty), ("regions", False, wide), ("pairs", False, pairs),
            ("regions", True, gen), ("regions", True, small), ("pairs", True, pairs), ("regions", False, gen),
            ("regions", True, wide), ("pairs", False, empty)]


@pytest.mark.parametrize("order", ["reverse", "shuffled", "submit"])
def test_mixed_queue_waited_in_any_order(wild, order):
    ctx, contigs = wild
    work = _mixed(contigs)
    want = [_sync(ctx, k, s, x) for k, s, x in work]
    assert want[3].stats.n_oversize == 1 and want[4].stats.n_oversize == 1 and want[7].stats.n_generic >= 10
    assert not want[3].ops[-3:].any() and not want[7].ops[-3:].any()   # oversize and empty items: zero ops
    jobs = [_submit(Job(ctx), k, s, x) for k, s, x in work]
    idx = list(range(len(jobs)))
    if order == "reverse":
        idx.reverse()
    elif order == "shuffled":
        random.Random(5).shuffle(idx)
    got = {i: jobs[i].wait() for i in idx}
    for i in range(len(jobs)):
        _equal(got[i], want[i])
        jobs[i].close()


def test_many_launches_give_the_synchronous_records():
    rng = random.Random(17)
    contigs = [sim.make_contig(1002, 0, 4_000_000, 0, 0, 0.0)]
    regs = _regions(rng, contigs, [rng.randrange(30, 300) for _ in range(24_000)], lambda ql: rng.randrange(ql, 900))
    chunks = _region_chunks(regs, [8_000, 10_000, 6_000])
    with Context(0) as ctx:
        ctx.load_reference(["chrS"], contigs)
        want = [_sync(ctx, "regions", s, x) for x in chunks for s in (False, True)]
    with Context(0, default_params(scratch_bytes=4 << 20)) as ctx:
        ctx.load_reference(["chrS"], contigs)
        jobs = [_submit(Job(ctx), "regions", s, x) for x in chunks for s in (False, True)]
        got = [j.wait() for j in jobs]
    for g, w in zip(got, want):
        assert g.stats.kernel_launches > 2 * w.stats.kernel_launches
        _equal(g, w, stats=False)


def test_inputs_may_be_overwritten_after_submit_and_jobs_resubmitted(c1):
    ctx, data = c1
    packed = data["pairs"][0]
    q, qo, t, to = (np.array(a, copy=True) for a in packed)
    n = 20_000
    qo, to = qo[:n + 1].copy(), to[:n + 1].copy()
    want = ctx.align_pairs(q, t, query_offsets=qo, target_offsets=to)
    job = Job(ctx).submit_pairs(q, t, query_offsets=qo, target_offsets=to)
    q[:] = ord("T")
    t[:] = ord("A")
    qo[1:] = qo[0]
    _equal(job.wait(), want)
    # the same job again, on other inputs: its new results, then the regions of C1
    q2, qo2, t2, to2 = packed
    want2 = ctx.score_pairs(q2, t2, query_offsets=qo2[n:2 * n + 1], target_offsets=to2[n:2 * n + 1])
    job.submit_pairs(q2, t2, score_only=True, query_offsets=qo2[n:2 * n + 1], target_offsets=to2[n:2 * n + 1])
    _equal(job.wait(), want2)
    regs = data["regions"]
    _equal(_submit(job, "regions", False, regs).wait(), _sync(ctx, "regions", False, regs))
    job.close()


def _nonempty(qo, k):
    """the first pair at or after k with a non-empty query"""
    return next(i for i in range(k, len(qo) - 1) if qo[i + 1] > qo[i])


def _raises(code, fn, *a, **kw):
    with pytest.raises(FadeGpuError) as e:
        fn(*a, **kw)
    assert e.value.code == code, str(e.value)
    return str(e.value)


def test_device_found_errors_fail_only_their_job(c1):
    ctx, data = c1
    chunks = _pair_chunks(data["pairs"][0], [3000, 3000, 3000])
    q, qo, t, to = chunks[1]
    bad = np.array(q, copy=True)
    k = _nonempty(qo, 5)
    bad[qo[k]] = ord("-")
    msg = _raises(E_ARG, ctx.align_pairs, bad, t, query_offsets=qo, target_offsets=to)
    assert f"fadegpu_align_pairs: the query of pair {k} holds" in msg
    jobs = [Job(ctx) for _ in range(3)]
    _submit(jobs[0], "pairs", False, chunks[0])
    jobs[1].submit_pairs(bad, t, query_offsets=qo, target_offsets=to)
    _submit(jobs[2], "pairs", True, chunks[2])
    _equal(jobs[2].wait(), _sync(ctx, "pairs", True, chunks[2]))
    assert _raises(E_ARG, jobs[1].wait) == msg.replace("fadegpu_align_pairs", "fadegpu_submit_pairs")
    _equal(jobs[0].wait(), _sync(ctx, "pairs", False, chunks[0]))
    _raises(E_STATE, jobs[1].wait)                                  # the failed job is idle again
    regs = data["regions"]
    qs = list(regs[0][:50])
    qs[7] = qs[7][:3] + "X" + qs[7][4:]
    sub = [list(a[:50]) for a in regs[1:]]
    rmsg = _raises(E_ARG, ctx.score_regions, qs, *sub)
    assert "fadegpu_score_regions: the query of region 7 holds" in rmsg
    jobs[1].submit_regions(qs, *sub, score_only=True)
    assert _raises(E_ARG, jobs[1].wait) == rmsg.replace("fadegpu_score_regions", "fadegpu_submit_regions")
    _equal(_submit(jobs[1], "pairs", False, chunks[1]).wait(), _sync(ctx, "pairs", False, chunks[1]))
    for j in jobs:
        j.close()


def test_state_and_argument_errors(c1, wild):
    ctx, data = c1
    L = _lib.lib()
    x = _pair_chunks(data["pairs"][0], [2000])[0]
    job = Job(ctx)
    # host-side E_ARG at submit, under the submit's name, leaves the job idle and usable
    for kw in (dict(query_offsets=[0, 4, 2]), ):
        msg = _raises(E_ARG, job.submit_pairs, b"ACGTACGT", b"ACGTACGT", target_offsets=[0, 4, 8], **kw)
        assert msg.endswith("fadegpu_submit_pairs: offsets decrease at pair 1")
    msg = _raises(E_ARG, job.submit_regions, ["ACGT"], [9], [0], [4])
    assert "fadegpu_submit_regions: region 0: tid 9 is not a contig of the reference" in msg
    _raises(E_STATE, job.wait)                                      # never submitted
    res = _submit(job, "pairs", False, x)
    _raises(E_STATE, _submit, job, "pairs", False, x)               # in flight
    v = _lib.JobResults()
    assert L.fadegpu_job_results_view(job._h, C.byref(v)) == E_STATE
    # a job with another ctx, and jobs / batches excluding each other
    other, _ = wild
    pin = _lib.PairsIn()
    assert L.fadegpu_submit_pairs(other._h, job._h, 0, C.byref(pin), 0, 0) == E_STATE
    assert L.fadegpu_job_wait(other._h, job._h, None) == E_STATE
    assert b"another ctx" in L.fadegpu_last_error(other._h)
    names, c1c, cfg, n = sim.config_c1()
    rd = sim.make_reads(cfg, 0, 2000, c1c)
    b = ctx.alloc_batch(rd.n, int(rd.seq_off[rd.n]))
    b.fill(rd.seq4, rd.seq_off, rd.l_qseq, rd.tid, rd.pos, rd.aligned_len, rd.clip_left, rd.clip_right)
    assert "a job of this ctx is in flight" in _raises(E_STATE, b.submit)
    _raises(E_STATE, b.submit_arrays, rd.n, rd.seq4, rd.seq_off, rd.l_qseq, rd.tid, rd.pos, rd.aligned_len,
            rd.clip_left, rd.clip_right)
    b.fill_compact(rd.seq4, rd.seq_off, rd.l_qseq, rd.tid, rd.pos, rd.aligned_len, rd.clip_left, rd.clip_right)
    _raises(E_STATE, b.submit_compact)
    want = _sync(ctx, "pairs", False, x)                            # a synchronous call runs after the job
    _equal(res.wait(), want)
    _raises(E_STATE, job.wait)                                      # waited already
    b.fill(rd.seq4, rd.seq_off, rd.l_qseq, rd.tid, rd.pos, rd.aligned_len, rd.clip_left, rd.clip_right)
    b.submit()
    assert "a batch of this ctx is in flight" in _raises(E_STATE, _submit, job, "pairs", False, x)
    _raises(E_STATE, job.submit_regions, ["ACGT"], [0], [0], [4])
    b.wait()
    rec0 = b.results()[0].copy()
    _equal(_submit(job, "pairs", False, x).wait(), want)
    assert np.array_equal(b.results()[0], rec0) and b.replay_kernels(1) > 0
    b.close()
    # max_ops with FADEGPU_JOB_SCORE_ONLY, unknown flags, no reference for regions
    assert L.fadegpu_submit_pairs(ctx._h, job._h, 0, C.byref(pin), 3, api.JOB_SCORE_ONLY) == E_ARG
    assert L.fadegpu_submit_pairs(ctx._h, job._h, 0, C.byref(pin), 0, 2) == E_ARG
    with Context(0) as bare:
        j2 = Job(bare)
        assert "no reference is loaded" in _raises(E_STATE, j2.submit_regions, ["ACGT"], [0], [0], [4])
        _raises(E_STATE, j2.wait)
        _equal(_submit(j2, "pairs", True, x).wait(), _sync(ctx, "pairs", True, x))
    job.close()


def test_sync_submit_returns_device_errors_from_submit(c1):
    ctx, data = c1
    x = _pair_chunks(data["pairs"][0], [5000])[0]
    q, qo, t, to = x
    bad = np.array(q, copy=True)
    k = _nonempty(qo, 17)
    bad[qo[k]] = ord("*")
    with Context(0, default_params(flags=api.F_SYNC_SUBMIT)) as sctx:
        j = Job(sctx)
        msg = _raises(E_ARG, j.submit_pairs, bad, t, query_offsets=qo, target_offsets=to)
        assert f"fadegpu_submit_pairs: the query of pair {k} holds" in msg
        _raises(E_STATE, j.wait)
        _equal(_submit(j, "pairs", False, x).wait(), _sync(ctx, "pairs", False, x))


def _threads():
    return len(os.listdir("/proc/self/task"))


def _raw_pair_job(L, ctx, x):
    """a job the Python layer does not track, submitted through the C ABI"""
    q, qo, t, to = x
    h = C.c_void_p()
    assert L.fadegpu_job_create(ctx._h, C.byref(h)) == 0
    pin = _lib.PairsIn(q.ctypes.data, qo.ctypes.data, t.ctypes.data, to.ctypes.data)
    assert L.fadegpu_submit_pairs(ctx._h, h, len(qo) - 1, C.byref(pin), 0, api.JOB_SCORE_ONLY) == 0
    return h


def test_lifetimes(c1):
    ctx, data = c1
    L = _lib.lib()
    chunks = _pair_chunks(data["pairs"][0], [8000, 8000, 8000])
    regs = data["regions"]
    want = [_sync(ctx, "pairs", s, x) for x in chunks for s in (False, True)]
    with Context(0) as c2:                                          # warm-up: what a ctx and a job start once
        _submit(Job(c2), "pairs", False, chunks[0]).wait()
    n0 = _threads()
    with Context(0) as c2:
        c2.share_reference_from(ctx)
        # a job destroyed in flight; synchronous calls while jobs are in flight give their usual records
        j = _submit(Job(c2), "pairs", False, chunks[0])
        j.close()
        jobs = [_submit(Job(c2), "pairs", s, x) for x in chunks for s in (False, True)]
        _equal(_sync(c2, "regions", False, regs), _sync(ctx, "regions", False, regs))
        _equal(_sync(c2, "pairs", True, chunks[1]), want[3])
        for g, w in zip([jb.wait() for jb in jobs], want):
            _equal(g, w)
        assert _threads() == n0 + 1                                 # the ctx's helper thread
        # the ctx destroyed with jobs in flight: tracked ones (closed first) and ones only the ctx knows
        keep = [_submit(Job(c2), "regions", True, regs) for _ in range(2)]
        raw = [_raw_pair_job(L, c2, x) for x in chunks]
        assert keep and raw
    assert _threads() == n0
