"""fadegpu_score_pairs / fadegpu_score_regions on the device.  Every check compares score, end_query, end_ref and flags
with the traced call (align_pairs / align_regions) on the same inputs and with the scalar oracle (fo_sw_trace), and
checks that beg_query, beg_ref and n_ops are 0: the census pairs, other scorings, the generic kernel, the diagonal
shortcut switched off, the annotate path's own alignments as regions, a multi-contig wildcard reference, sizes across
every kernel, global offsets past 2^31, the calls' contract and many launches.  Run with `pytest -m gpu` on a B200."""
import os
import random
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from fade_b200 import Context, api, default_params, sim
from fade_b200._lib import FadeGpuError
from oracle import oracle as orc
from test_gpu_pairs import CHEAP_GAPS, _census, _planted
from test_gpu_regions import _as_pairs, _rc, _regions, _wild_contigs

pytestmark = pytest.mark.gpu

E_ARG, E_STATE = -1, -4
KEPT = ("score", "end_query", "end_ref", "flags")


def _score_pairs(ctx, packed):
    q, qo, t, to = packed
    return ctx.score_pairs(q, t, query_offsets=qo, target_offsets=to)


def _align_pairs(ctx, packed):
    q, qo, t, to = packed
    return ctx.align_pairs(q, t, query_offsets=qo, target_offsets=to)


def _same_as_traced(s, traced):
    """the score-only records against the traced call's (default max_ops: nothing truncated) on the same inputs"""
    assert len(s) == len(traced)
    for f in KEPT:
        assert np.array_equal(s.records[f], traced.records[f]), (f, np.nonzero(s.records[f] != traced.records[f])[0][:10])
    for f in ("beg_query", "beg_ref", "n_ops", "reserved"):
        assert not s.records[f].any(), f
    assert not (s.records["flags"] & (api.R_OPS_TRUNC | api.R_SCORE_ONLY)).any()
    for f in ("n_reads", "n_aligned", "n_generic", "cells", "n_oversize"):
        assert getattr(s.stats, f) == getattr(traced.stats, f), f
    # no ops come home: the traced call's D2H less its max_ops words per item
    assert traced.stats.d2h_bytes - s.stats.d2h_bytes == 4 * traced.ops.size
    assert s.stats.h2d_bytes == traced.stats.h2d_bytes
    assert 0 < s.stats.kernel_launches <= traced.stats.kernel_launches or len(s) == 0


def _check_oracle(s, qs, ts, idx=None, params=None):
    """score and end cell of s at idx against fo_sw_trace of the upper-cased (qs[k], ts[k])"""
    idx = list(range(len(qs))) if idx is None else list(idx)

    def one(k):
        return orc.sw_trace(qs[k].upper(), ts[k].upper(), params=params)
    with ThreadPoolExecutor(os.cpu_count() or 4) as ex:
        ref = list(ex.map(one, idx, chunksize=256))
    rec = s.records
    bad = [k for k, r in zip(idx, ref)
           if (int(rec["score"][k]), int(rec["end_query"][k]), int(rec["end_ref"][k])) !=
           ((r.score, r.end_query, r.end_ref) if r.score > 0 else (0, 0, 0)) or not rec["flags"][k] & api.R_ALIGNED]
    assert not bad, f"{len(bad)} items differ from the oracle, first {bad[0]}: {rec[bad[0]]}"


@pytest.fixture(scope="module")
def census_short():
    return _census(11, 200_000, 72, 160)


def test_census_pairs(census_short):
    packed, qs, ts = census_short
    with Context(0) as ctx:
        s, traced = _score_pairs(ctx, packed), _align_pairs(ctx, packed)
    assert s.stats.n_aligned == 200_000 and (s.records["flags"] & api.R_GENERIC != 0).sum() > 1000
    _same_as_traced(s, traced)
    _check_oracle(s, qs, ts)
    assert not hasattr(s, "cigar") and not hasattr(s, "ops")


def test_read_sized_census_pairs():
    packed, qs, ts = _census(41, 20_000, 260, 1000)
    with Context(0) as ctx:
        s, traced = _score_pairs(ctx, packed), _align_pairs(ctx, packed)
    _same_as_traced(s, traced)
    _check_oracle(s, qs, ts)


@pytest.mark.parametrize("scoring", CHEAP_GAPS + [(10, 2, 9, -3), (10, 2, 2, -9)])
def test_other_scorings(scoring):
    """the six extra scorings of the pair tests: every score-only step (score_step_for) runs in the scan rounds"""
    o, e, m, x = scoring
    packed, qs, ts = _census(21, 20_000, 72, 160)
    with Context(0, default_params(gap_open=o, gap_extend=e, match=m, mismatch=x)) as ctx:
        s, traced = _score_pairs(ctx, packed), _align_pairs(ctx, packed)
    _same_as_traced(s, traced)
    _check_oracle(s, qs, ts, params=orc.default_params(gap_open=o, gap_extend=e, match=m, mismatch=x))


@pytest.mark.parametrize("flags", [api.F_FORCE_GENERIC, api.F_NO_SHORTCUT, api.F_TAGS_ONLY])
def test_ctx_flags(census_short, flags):
    """F_FORCE_GENERIC serves every pair from the generic kernel with the same score and end cell; F_NO_SHORTCUT and
    F_TAGS_ONLY change no record"""
    packed, qs, ts = census_short
    with Context(0) as ctx:
        base = _score_pairs(ctx, packed)
    with Context(0, default_params(flags=flags)) as ctx:
        s, traced = _score_pairs(ctx, packed), _align_pairs(ctx, packed)
    _same_as_traced(s, traced)
    a, b = base.records.copy(), s.records.copy()
    if flags == api.F_FORCE_GENERIC:
        assert s.stats.n_generic == 200_000 and (s.records["flags"] & api.R_GENERIC).all()
        a["flags"] &= ~np.uint32(api.R_GENERIC)
        b["flags"] &= ~np.uint32(api.R_GENERIC)
    assert np.array_equal(a, b)
    _check_oracle(s, qs, ts, range(0, 200_000, 20))


def test_annotate_alignments_as_regions():
    """C1's aligned reads as regions on both strands: the annotate path's score and end cell; the waited batch keeps its
    results and its kernel replay afterwards"""
    names, contigs, cfg, n = sim.config_c1()
    rd = sim.make_reads(cfg, 0, n, contigs)
    clen = len(contigs[0])
    with Context(0) as ctx:
        ctx.load_reference(names, [c.tobytes() for c in contigs])
        b = ctx.alloc_batch(rd.n, int(rd.seq_off[rd.n]))
        b.fill(rd.seq4, rd.seq_off, rd.l_qseq, rd.tid, rd.pos, rd.aligned_len, rd.clip_left, rd.clip_right).run()
        rec0, ws0, ri0 = (x.copy() for x in b.results())
        al = np.nonzero(b.flags[:rd.n] & api.R_ALIGNED)[0]
        assert len(al) > 1000
        W = ctx.params.window_size
        fwd, rcs = [], []
        for r in al:
            so, lq = int(rd.seq_off[r]), int(rd.l_qseq[r])
            fwd.append(orc.decode_nt16(rd.seq4[so:so + (lq + 1) // 2], lq))
            rcs.append(orc.revcomp_nt16(rd.seq4[so:so + (lq + 1) // 2], lq))
        starts = b.win_start[al].astype(np.int64)
        ends = np.minimum(rd.pos[al] + rd.aligned_len[al] + W, clen)
        for qs, strand in ((fwd, 1), (rcs, 0)):
            args = (qs, rd.tid[al], starts, ends, np.full(len(al), strand))
            s, traced = ctx.score_regions(*args), ctx.align_regions(*args)
            _same_as_traced(s, traced)
            for f in ("score", "end_query", "end_ref"):
                assert np.array_equal(s.records[f], getattr(b, f)[al]), (strand, f)
        rec1, ws1, ri1 = b.results()
        assert np.array_equal(rec0, rec1) and np.array_equal(ws0, ws1) and np.array_equal(ri0, ri1)
        assert b.replay_kernels(2) > 0
        rec2, _, _ = b.results()
        assert np.array_equal(rec0, rec2)
        b.close()


@pytest.fixture(scope="module")
def wild():
    contigs = _wild_contigs(7, [300_000, 2_600_000, 90_000])
    with Context(0) as ctx:
        ctx.load_reference(["c0", "c1", "c2"], contigs)
        yield ctx, contigs


def test_regions_on_a_wildcard_reference(wild):
    ctx, contigs = wild
    rng = random.Random(3)
    qlens = [rng.choice((rng.randrange(1, 105), rng.randrange(105, 153), rng.randrange(153, 201),
                         rng.randrange(201, 257), rng.randrange(257, 305), rng.randrange(305, 420)))
             for _ in range(6000)]
    args = _regions(rng, contigs, qlens, lambda ql: rng.randrange(max(1, ql // 2), 3000))
    s, traced = ctx.score_regions(*args), ctx.align_regions(*args)
    _same_as_traced(s, traced)
    assert s.stats.n_generic > 500 and (s.records["score"] > 100).sum() > 1500
    sp, qq, ts = _as_pairs(ctx, *(args[:1] + (contigs,) + args[1:]))
    assert np.array_equal(ctx.score_pairs(qq, ts).records, s.records)     # the same records through the pair call
    _check_oracle(s, qq, ts)


def test_sizes_across_every_kernel(wild):
    """R = 13 / 19 / 25 / 32 / 38, windows past 1024 and 4000 columns (restaged chunks, shared sort keys), and the generic
    kernel for queries over 304, windows over 10^6 columns and wildcards -- as pairs and as regions"""
    ctx, contigs = wild
    rng = random.Random(5)
    qs, ts = [], []
    for ql in list(range(1, 305, 3)) + [104, 105, 152, 153, 200, 201, 256, 257, 304]:
        q, t = _planted(rng, ql, rng.randrange(max(8, ql // 2), 4000)); qs.append(q); ts.append(t)
    for ql in range(305, 601, 15):
        q, t = _planted(rng, ql, rng.randrange(300, 2000)); qs.append(q); ts.append(t)
    for tl in (1_500, 5_000, 9_999, 33_000, 70_000):
        q, t = _planted(rng, rng.choice((100, 250, 300)), tl); qs.append(q); ts.append(t)
    q, t = _planted(rng, 60, 1_200_000); qs.append(q); ts.append(t)
    s, traced = ctx.score_pairs(qs, ts), ctx.align_pairs(qs, ts)
    _same_as_traced(s, traced)
    _check_oracle(s, qs, ts)
    assert s.stats.n_generic >= 21 and s.records["flags"][-1] & api.R_GENERIC
    big = [contigs[1]]
    qlens = list(range(1, 305, 3)) + [104, 105, 152, 153, 200, 201, 256, 257, 304] + list(range(305, 601, 15))
    qr, tids, starts, ends, strands = _regions(rng, big, qlens, lambda ql: rng.randrange(max(8, ql // 2), 6000))
    args = (qr, [1] * len(qr), starts, ends, strands)
    s, traced = ctx.score_regions(*args), ctx.align_regions(*args)
    _same_as_traced(s, traced)
    _, qq, tt = _as_pairs(ctx, qr, contigs, *args[1:])
    _check_oracle(s, qq, tt)


def test_global_offsets_past_2_31():
    import psutil
    from test_gpu_fullconfigs import c3_contigs
    if psutil.virtual_memory().available < 14 * (1 << 30):
        pytest.skip("needs 14 GB of free host RAM for the 3.1 Gbp synthetic reference")
    names, contigs = c3_contigs()
    assert sum(len(c) for c in contigs[:20]) > 2 ** 31
    rng = random.Random(9)
    late = contigs[20:]
    qs, tids, starts, ends, strands = _regions(rng, late, [rng.randrange(20, 400) for _ in range(2000)],
                                               lambda ql: rng.randrange(max(1, ql // 2), 2000))
    args = (qs, [t + 20 for t in tids], starts, ends, strands)
    with Context(0) as ctx:
        ctx.load_reference(names, contigs)
        s, traced = ctx.score_regions(*args), ctx.align_regions(*args)
    _same_as_traced(s, traced)
    assert (s.records["score"] > 100).sum() > 500
    qq = [_rc(q) if st else q for q, st in zip(qs, strands)]
    ts = [late[t][a:b].tobytes().decode() for t, a, b in zip(tids, starts, ends)]
    _check_oracle(s, qq, ts, range(0, 2000, 4))


def test_contract(wild):
    ctx, contigs = wild
    L0 = len(contigs[0])
    # empty items, an oversize item, and no items at all
    qs = ["ACGTACGTAA", "", "ACGT", "", "ACGT" * 250]
    ts = ["TTACGTACGTAATT", "ACGT", "", "", "A" * 2_200_000]
    for s, traced in ((ctx.score_pairs(qs, ts), ctx.align_pairs(qs, ts)),
                      (ctx.score_regions(qs, [0, 0, 1, 2, 1], [5, 9, 0, 7, 100], [45, 13, 0, 7, 2_200_100]),
                       ctx.align_regions(qs, [0, 0, 1, 2, 1], [5, 9, 0, 7, 100], [45, 13, 0, 7, 2_200_100]))):
        _same_as_traced(s, traced)
        for k in (1, 2, 3):
            assert s.records[k].tolist() == (0,) * 8
        assert s.records[4].tolist() == (0,) * 6 + (api.R_OVERSIZE, 0) and s.stats.n_oversize == 1
        assert s.stats.n_aligned == 1
    assert tuple(ctx.score_pairs(["ACGTACGTAA"], ["TTACGTACGTAATT"]).records[0].tolist()) == (20, 9, 11, 0, 0, 0, 1, 0)
    for e in (ctx.score_pairs([], []), ctx.score_regions([], [], [], [])):
        assert len(e) == 0 and e.stats.n_reads == 0
    # argument errors: the traced calls' cases and messages, with the score call's name
    for call, name in ((ctx.score_pairs, "fadegpu_score_pairs"), (ctx.align_pairs, "fadegpu_align_pairs")):
        for bad, k in ((["ACGT", "ACGT", "ACGT", "AC-T"], 3), (["ACGT", "ACXT", "ACGT", "AC-T"], 1)):
            with pytest.raises(FadeGpuError) as e:
                call(bad, ["ACGT"] * 4)
            assert e.value.code == E_ARG and f"{name}: the query of pair {k} holds" in str(e.value)
    ok = dict(qs=["ACGT"] * 4, tids=[0, 1, 2, 0], starts=[0, 10, 20, 30], ends=[40, 50, 60, 70], strands=[0, 1, 0, 1])
    for k, kw in [(2, dict(tids=[0, 1, 3, 0])), (3, dict(starts=[0, 10, 20, -1])), (0, dict(starts=[41, 10, 20, 30])),
                  (1, dict(tids=[0, 0, 2, 0], ends=[40, L0 + 1, 60, 70])), (2, dict(strands=[0, 1, 2, 1])),
                  (3, dict(qs=["ACGT", "ACGT", "ACGT", "AC-T"]))]:
        a = dict(ok, **kw)
        msgs = []
        for call in (ctx.score_regions, ctx.align_regions):
            with pytest.raises(FadeGpuError) as e:
                call(a["qs"], a["tids"], a["starts"], a["ends"], a["strands"])
            assert e.value.code == E_ARG and f"region {k}" in str(e.value), (k, kw, str(e.value))
            msgs.append(str(e.value))
        assert msgs[0].replace("fadegpu_score_regions", "fadegpu_align_regions") == msgs[1]
    with pytest.raises(FadeGpuError) as e:
        ctx.score_regions(b"ACGTACGTAC", [0] * 3, [0] * 3, [40] * 3, query_offsets=[0, 4, 2, 6])
    assert e.value.code == E_ARG and "fadegpu_score_regions: offsets decrease at region 1" in str(e.value)
    with pytest.raises(FadeGpuError) as e:
        ctx.score_pairs(b"ACGTACGTAC", b"ACGT", query_offsets=[0, 4, 2], target_offsets=[0, 2, 4])
    assert e.value.code == E_ARG and "fadegpu_score_pairs: offsets decrease at pair 1" in str(e.value)
    # no reference (regions only), a batch in flight, and the batch's results and replay untouched afterwards
    with Context(0) as bare:
        with pytest.raises(FadeGpuError) as e:
            bare.score_regions(["ACGT"], [0], [0], [4])
        assert e.value.code == E_STATE and "fadegpu_score_regions: no reference is loaded" in str(e.value)
        assert bare.score_pairs(["ACGT"], ["ACGT"]).records["score"][0] == 8   # a ctx used only for pairs
        names, c1, cfg, n = sim.config_c1()
        bare.load_reference(names, [c.tobytes() for c in c1])
        rd = sim.make_reads(cfg, 0, 2000, c1)
        b = bare.alloc_batch(rd.n, int(rd.seq_off[rd.n]))
        b.fill(rd.seq4, rd.seq_off, rd.l_qseq, rd.tid, rd.pos, rd.aligned_len, rd.clip_left, rd.clip_right)
        b.submit()
        for call in (lambda: bare.score_regions(["ACGT"], [0], [0], [4]), lambda: bare.score_pairs(["ACGT"], ["ACGT"])):
            with pytest.raises(FadeGpuError) as e:
                call()
            assert e.value.code == E_STATE
        b.wait()
        rec0 = b.results()[0].copy()
        ms0 = b.replay_kernels(1)
        assert bare.score_regions(["ACGTACGTAA"], [0], [1000], [1040]).stats.n_aligned == 1
        assert bare.score_pairs(["ACGT"], ["ACGT"]).stats.n_aligned == 1
        assert np.array_equal(b.results()[0], rec0)
        assert b.replay_kernels(2) > 0 and ms0 > 0
        assert np.array_equal(b.results()[0], rec0)
        b.close()


def test_many_launches_give_the_same_records():
    """a 4 MB checkpoint scratch splits the call into many launches, each with its own scan rounds"""
    packed, qs, ts = _census(51, 200_000, 160, 700)
    with Context(0) as ctx:
        a = _score_pairs(ctx, packed)
    with Context(0, default_params(scratch_bytes=4 << 20)) as ctx:
        b, traced = _score_pairs(ctx, packed), _align_pairs(ctx, packed)
    assert b.stats.kernel_launches > 2 * a.stats.kernel_launches
    assert np.array_equal(a.records, b.records)
    _same_as_traced(b, traced)
    _check_oracle(b, qs, ts, range(0, 200_000, 50))
