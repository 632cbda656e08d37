"""fadegpu_align_regions on the device: the annotate path's own alignments given as regions, equality with
fadegpu_align_pairs on the sliced targets (and with the scalar oracle) over a multi-contig reference with N runs and
wildcard letters, sizes across every kernel, global offsets past 2^31, the call's contract and many launches.
Run with `pytest -m gpu` on a B200."""
import ctypes as C
import os
import random
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from fade_b200 import Context, _lib, api, default_params, sim
from fade_b200._lib import FadeGpuError
from oracle import oracle as orc

pytestmark = pytest.mark.gpu

FIELDS = ("score", "end_query", "end_ref", "beg_query", "beg_ref", "n_ops")
NT16 = "=ACMGRSVTWYHKDBN"
COMP16 = [0, 8, 4, 12, 2, 10, 6, 14, 1, 9, 5, 13, 3, 11, 7, 15]
E_ARG, E_STATE = -1, -4


def _rc(s: str) -> str:
    """nt16 reverse complement of ASCII letters (source/util.d:18-34)"""
    return "".join(NT16[COMP16[NT16.index(c)]] for c in reversed(s.upper()))


def _as_pairs(ctx, qs, contigs, tids, starts, ends, strands, max_ops=None):
    """the same alignments through fadegpu_align_pairs: the sliced targets, strand-1 queries reverse-complemented"""
    ts = [contigs[t][s:e].tobytes() for t, s, e in zip(tids, starts, ends)]
    qq = [_rc(q) if st else q for q, st in zip(qs, strands)]
    return ctx.align_pairs(qq, ts, max_ops), qq, ts


def _same(a, b):
    assert np.array_equal(a.records, b.records), np.nonzero(a.records != b.records)[0][:10]
    assert np.array_equal(a.ops, b.ops)


def _check_oracle(res, qs, ts, idx):
    """records and full CIGARs of res at idx against fo_sw_trace of (qs[k], ts[k]), upper-cased"""
    def one(k):
        return orc.sw_trace(qs[k].upper(), ts[k].upper(), ops_cap=4096)
    with ThreadPoolExecutor(os.cpu_count() or 4) as ex:
        ref = list(ex.map(one, idx, chunksize=64))
    rec = res.records
    bad = []
    for k, r in zip(idx, ref):
        if r.score <= 0:
            ok = rec["score"][k] == 0 and rec["n_ops"][k] == 0 and rec["flags"][k] & 1
        else:
            ok = all(int(rec[f][k]) == getattr(r, f) for f in FIELDS) and rec["flags"][k] & 1 and \
                res.ops[k, :r.n_ops].tolist() == r.ops and not res.ops[k, r.n_ops:].any()
        if not ok:
            bad.append(k)
    assert not bad, f"{len(bad)} regions differ from the oracle, first {bad[0]}: {rec[bad[0]]} {res.cigar(bad[0])}"


def _wild_contigs(seed, lens):
    """contigs with N runs, 1 % lower-case tiles and scattered IUPAC wildcard letters (upper and lower case)"""
    rng = np.random.default_rng(seed)
    out = []
    for i, n in enumerate(lens):
        c = sim.make_contig(seed, i, n, 20_000, 300, 0.01)
        at = rng.choice(n, n // 2000, replace=False)
        c[at] = rng.choice(np.frombuffer(b"RYKMSWBDHVrykn", np.uint8), len(at))
        out.append(c)
    return out


def _mutate(rng, s, gapped):
    s = [c if rng.random() > 0.04 else rng.choice("ACGT") for c in s]
    if gapped and len(s) > 40:
        cut = rng.randrange(10, len(s) - 10)
        s = s[:cut] + list("TGA") + s[cut:] if rng.random() < 0.5 else s[:cut] + s[cut + 4:]
    return "".join(s)


def _regions(rng, contigs, qlens, tlen_of, planted=0.7):
    """one region per query length: a random interval of length tlen_of(qlen), a random strand, and a query planted
    from the interval (mutated, sometimes gapped, with IUPAC letters now and then) or random"""
    qs, tids, starts, ends, strands = [], [], [], [], []
    for ql in qlens:
        t = rng.randrange(len(contigs))
        tl = min(tlen_of(ql), len(contigs[t]))
        s = rng.randrange(0, len(contigs[t]) - tl + 1)
        st = rng.randrange(2)
        if ql and rng.random() < planted and tl:
            a = rng.randrange(s, s + tl)
            piece = contigs[t][a:a + ql].tobytes().decode().upper()
            piece = "".join(c if c in "ACGTN" else "N" for c in piece)
            piece += "".join(rng.choice("ACGT") for _ in range(ql - len(piece)))
            q = _mutate(rng, list(piece), rng.random() < 0.4)[:ql]
            q = _rc(q) if st else q
        else:
            q = "".join(rng.choice("ACGT") for _ in range(ql))
        if q and rng.random() < 0.1:
            i = rng.randrange(len(q))
            q = q[:i] + rng.choice("RYKMSWBDHVNacgtn") + q[i + 1:]
        qs.append(q); tids.append(t); starts.append(s); ends.append(s + tl); strands.append(st)
    return qs, tids, starts, ends, strands


@pytest.fixture(scope="module")
def wild():
    contigs = _wild_contigs(7, [300_000, 2_600_000, 90_000])
    with Context(0) as ctx:
        ctx.load_reference(["c0", "c1", "c2"], contigs)
        yield ctx, contigs


def test_annotate_alignments_as_regions():
    """C1's aligned reads as (forward letters, strand 1, their window) and as (reverse complement, strand 0) give what
    the annotate path gave them, and the batch's results and a replay of its kernels are unaffected"""
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
            res = ctx.align_regions(qs, rd.tid[al], starts, ends, np.full(len(al), strand))
            for f in FIELDS:
                assert np.array_equal(res.records[f], getattr(b, f)[al]), (strand, f)
            k = np.minimum(res.records["n_ops"], api.MAX_OPS)
            m = np.arange(api.MAX_OPS)[None, :] < k[:, None]
            assert np.array_equal(np.where(m, res.ops[:, :api.MAX_OPS], 0), np.where(m, b.ops[al], 0))
            assert res.stats.n_aligned == len(al)
        rec1, ws1, ri1 = b.results()
        assert np.array_equal(rec0, rec1) and np.array_equal(ws0, ws1) and np.array_equal(ri0, ri1)
        assert b.replay_kernels(2) > 0
        rec2, _, _ = b.results()
        assert np.array_equal(rec0, rec2)
        b.close()


def test_regions_equal_pairs_and_the_oracle(wild):
    ctx, contigs = wild
    rng = random.Random(3)
    qlens = [rng.choice((rng.randrange(1, 105), rng.randrange(105, 153), rng.randrange(153, 201),
                         rng.randrange(201, 257), rng.randrange(257, 305), rng.randrange(305, 420)))
             for _ in range(6000)]
    qs, tids, starts, ends, strands = _regions(rng, contigs, qlens, lambda ql: rng.randrange(max(1, ql // 2), 3000))
    res = ctx.align_regions(qs, tids, starts, ends, strands)
    pr, qq, ts = _as_pairs(ctx, qs, contigs, tids, starts, ends, strands)
    _same(res, pr)
    assert res.stats.n_aligned == 6000 and res.stats.n_generic > 500
    assert (res.records["score"] > 100).sum() > 1500          # the planted queries are found
    assert sum(strands) > 2500 and 0 < sum(1 for q in qs if set(q) - set("ACGT")) < 2000
    _check_oracle(res, qq, ts, list(range(0, 6000, 12)))


def test_sizes_across_every_kernel(wild):
    ctx, contigs = wild
    rng = random.Random(5)
    big = [contigs[1]]                                                                     # 2.6 Mbp
    qlens = list(range(1, 305, 3)) + [104, 105, 152, 153, 200, 201, 256, 257, 304]         # the five row classes
    qs, tids, starts, ends, strands = _regions(rng, big, qlens, lambda ql: rng.randrange(max(8, ql // 2), 4000))
    more = [_regions(rng, big, range(305, 601, 15), lambda ql: rng.randrange(300, 2000)),   # generic kernel
            _regions(rng, big, [rng.choice((100, 250, 300)) for _ in range(4)],             # restaged target chunks
                     lambda ql, it=iter((5_000, 9_999, 33_000, 70_000)): next(it)),
            _regions(rng, big, [60], lambda ql: 1_200_000)]                                # beyond the packed kernels
    for m in more:
        for acc, x in zip((qs, tids, starts, ends, strands), m):
            acc += x
    tids = [1] * len(qs)                                                                   # big[0] is contig 1
    n_checked = len(qs)
    # oversize, empty query, empty interval, both empty
    qs += ["ACGT" * 250, "", "ACGT", ""]
    tids += [1, 0, 0, 0]
    starts += [100, 5, 7, 9]
    ends += [2_200_100, 50, 7, 9]
    strands += [0, 1, 1, 0]
    res = ctx.align_regions(qs, tids, starts, ends, strands)
    pr, qq, ts = _as_pairs(ctx, qs, contigs, tids, starts, ends, strands)
    _same(res, pr)
    _check_oracle(res, qq, ts, list(range(n_checked)))
    assert res.stats.n_generic >= 21 and res.records["flags"][n_checked - 1] & api.R_GENERIC
    assert res.records[n_checked].tolist() == (0,) * 6 + (api.R_OVERSIZE, 0) and res.stats.n_oversize == 1
    for k in range(n_checked + 1, n_checked + 4):
        assert res.records[k].tolist() == (0,) * 8
    assert res.stats.n_aligned == n_checked


def test_global_offsets_past_2_31():
    """regions on the last contigs of the C3 reference (3.1 Gbp, 24 contigs), whose global offsets exceed 2^31"""
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
    with Context(0) as ctx:
        ctx.load_reference(names, contigs)
        res = ctx.align_regions(qs, [t + 20 for t in tids], starts, ends, strands)
        pr, _, _ = _as_pairs(ctx, qs, late, tids, starts, ends, strands)
    _same(res, pr)
    assert (res.records["score"] > 100).sum() > 500


def _staged_regions(qs):
    a16 = lambda x: (x + 15) & ~15                                                        # noqa: E731
    n, qb = len(qs), sum(len(q) for q in qs)
    return a16((n + 1) * 8) + a16(n * 4) + 2 * a16(n * 8) + a16(n) + a16(qb)


def _staged_pairs(qs, ts):
    a16 = lambda x: (x + 15) & ~15                                                        # noqa: E731
    n = len(qs)
    return 2 * a16((n + 1) * 8) + a16(sum(len(q) for q in qs)) + a16(sum(len(t) for t in ts))


def test_contract(wild):
    ctx, contigs = wild
    L0, L1 = len(contigs[0]), len(contigs[1])
    ok = dict(qs=["ACGT"] * 4, tids=[0, 1, 2, 0], starts=[0, 10, 20, 30], ends=[40, 50, 60, 70], strands=[0, 1, 0, 1])

    def call(**kw):
        a = dict(ok, **kw)
        return ctx.align_regions(a["qs"], a["tids"], a["starts"], a["ends"], a["strands"])

    # host-side argument errors name the region; an interval may end at the contig's end but not beyond
    for k, kw in [(2, dict(tids=[0, 1, 3, 0])), (1, dict(tids=[0, -1, 2, 0])), (3, dict(starts=[0, 10, 20, -1])),
                  (0, dict(starts=[41, 10, 20, 30])), (1, dict(tids=[0, 0, 2, 0], ends=[40, L0 + 1, 60, 70])),
                  (2, dict(strands=[0, 1, 2, 1]))]:
        with pytest.raises(FadeGpuError) as e:
            call(**kw)
        assert e.value.code == E_ARG and f"region {k}" in str(e.value), (k, kw, str(e.value))
    assert call(tids=[0, 1, 2, 1], starts=[L0 - 40, 10, 20, L1 - 4], ends=[L0, 50, 60, L1]).stats.n_aligned == 4
    with pytest.raises(FadeGpuError) as e:
        ctx.align_regions(b"ACGTACGTAC", [0] * 3, [0] * 3, [40] * 3, query_offsets=[0, 4, 2, 6])
    assert e.value.code == E_ARG and "region 1" in str(e.value)
    with pytest.raises(FadeGpuError) as e:                          # a letter outside nt16 (found on the device)
        call(qs=["ACGT", "ACGT", "ACGT", "AC-T"])
    assert e.value.code == E_ARG and "region 3" in str(e.value)
    with pytest.raises(FadeGpuError) as e:
        call(qs=["ACGT", "ACXT", "ACGT", "AC-T"])
    assert "region 1" in str(e.value)
    rin = _lib.RegionsIn()                                          # null arrays
    out = (_lib.PairResult * 1)()
    assert _lib.lib().fadegpu_align_regions(ctx._h, 1, C.byref(rin), 0, out, None, None) == E_ARG
    # no reference, and a batch in flight
    with Context(0) as bare:
        with pytest.raises(FadeGpuError) as e:
            bare.align_regions(["ACGT"], [0], [0], [4])
        assert e.value.code == E_STATE
        names, c1, cfg, n = sim.config_c1()
        bare.load_reference(names, [c.tobytes() for c in c1])
        rd = sim.make_reads(cfg, 0, 2000, c1)
        b = bare.alloc_batch(rd.n, int(rd.seq_off[rd.n]))
        b.fill(rd.seq4, rd.seq_off, rd.l_qseq, rd.tid, rd.pos, rd.aligned_len, rd.clip_left, rd.clip_right)
        b.submit()
        with pytest.raises(FadeGpuError) as e:
            bare.align_regions(["ACGT"], [0], [0], [4])
        assert e.value.code == E_STATE
        b.wait()
        r = bare.align_regions(["ACGTACGTAA"], [0], [1000], [1040])
        assert r.stats.n_aligned == 1
        b.close()
    # tags-only does not apply, the forced generic kernel gives the same records, max_ops truncates as pairs do
    rng = random.Random(13)
    qs, tids, starts, ends, strands = _regions(rng, contigs, [rng.randrange(30, 300) for _ in range(3000)],
                                               lambda ql: rng.randrange(ql, 1500))
    full = ctx.align_regions(qs, tids, starts, ends, strands)
    cut = ctx.align_regions(qs, tids, starts, ends, strands, max_ops=3)
    pcut, qq, ts = _as_pairs(ctx, qs, contigs, tids, starts, ends, strands, max_ops=3)
    _same(cut, pcut)
    long = full.records["n_ops"] > 3
    assert long.sum() > 100 and np.array_equal((cut.records["flags"] & api.R_OPS_TRUNC) != 0, long)
    assert np.array_equal(cut.ops, full.ops[:, :3]) and not (full.records["flags"] & api.R_OPS_TRUNC).any()
    for flags in (api.F_TAGS_ONLY, api.F_FORCE_GENERIC):
        with Context(0, default_params(flags=flags)) as other:
            other.share_reference_from(ctx)
            r = other.align_regions(qs, tids, starts, ends, strands)
        a, b2 = full.records.copy(), r.records.copy()
        if flags == api.F_FORCE_GENERIC:
            assert (r.records["flags"] & api.R_GENERIC).all() and r.stats.n_generic == 3000
            a["flags"] &= ~np.uint32(api.R_GENERIC)
            b2["flags"] &= ~np.uint32(api.R_GENERIC)
        assert np.array_equal(a, b2) and np.array_equal(full.ops, r.ops), flags
        assert not (r.records["flags"] & api.R_SCORE_ONLY).any()
    # H2D: the staged inputs (no reference letters) plus the same launch plan as the pair call
    pfull, _, _ = _as_pairs(ctx, qs, contigs, tids, starts, ends, strands)
    plan = pfull.stats.h2d_bytes - _staged_pairs(qq, ts)
    assert plan > 0 and full.stats.h2d_bytes == _staged_regions(qs) + plan
    assert full.stats.h2d_bytes < pfull.stats.h2d_bytes


def test_many_launches_give_the_same_results():
    rng = random.Random(17)
    contigs = [sim.make_contig(1002, 0, 4_000_000, 0, 0, 0.0)]
    qs, tids, starts, ends, strands = _regions(rng, contigs, [rng.randrange(30, 300) for _ in range(100_000)],
                                               lambda ql: rng.randrange(ql, 900))
    with Context(0) as ctx:
        ctx.load_reference(["chrS"], contigs)
        a = ctx.align_regions(qs, tids, starts, ends, strands)
    with Context(0, default_params(scratch_bytes=4 << 20)) as ctx:
        ctx.load_reference(["chrS"], contigs)
        b = ctx.align_regions(qs, tids, starts, ends, strands)
    assert b.stats.kernel_launches > 3 * a.stats.kernel_launches
    _same(a, b)
