"""fadegpu_align_pairs on the device: the striped-parity census pairs, other scorings, both kernel families, the annotate
path's own alignments, sizes across every kernel, the call's contract and many launches -- every record field and the
full CIGAR against the scalar oracle (and the striped restatement of parasail).  Run with `pytest -m gpu` on a B200."""
import os
import random
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import pair_census
import readsets
from fade_b200 import Context, api, default_params, sim
from fade_b200._lib import FadeGpuError
from oracle import oracle as orc

pytestmark = pytest.mark.gpu

FIELDS = ("score", "end_query", "end_ref", "beg_query", "beg_ref", "n_ops")
CHEAP_GAPS = [(3, 1, 2, -3), (4, 2, 2, -3), (2, 2, 1, -1), (6, 1, 5, -4)]


def _oracle(qs, ts, params=None, lanes=0):
    """fo_sw_trace (lanes 0) or ps_sw_trace of every pair, upper-cased as the device sees them; ctypes drops the GIL"""
    def one(k):
        q, t = qs[k].upper(), ts[k].upper()
        if lanes:
            return orc.sw_trace_striped(q, t, lanes, params=params, ops_cap=4096)
        return orc.sw_trace(q, t, params=params, ops_cap=4096)
    with ThreadPoolExecutor(os.cpu_count() or 4) as ex:
        return list(ex.map(one, range(len(qs)), chunksize=256))


def _check(res, ref, idx=None, generic=None):
    """records and full CIGARs of res (pair order) against oracle results ref (for the pairs idx)"""
    idx = range(len(ref)) if idx is None else idx
    rec = res.records
    bad = []
    for k, r in zip(idx, ref):
        if r.score <= 0:
            ok = rec["score"][k] == 0 and rec["n_ops"][k] == 0 and rec["flags"][k] & 1
        else:
            ok = all(int(rec[f][k]) == getattr(r, f) for f in FIELDS) and rec["flags"][k] & 1 and \
                res.ops[k, :r.n_ops].tolist() == r.ops and not res.ops[k, r.n_ops:].any()
        if generic is not None:
            ok = ok and bool(rec["flags"][k] & api.R_GENERIC) == generic
        if not ok:
            bad.append(k)
    assert not bad, (f"{len(bad)} pairs differ, first {bad[0]}: "
                     f"gpu {rec[bad[0]]} {res.cigar(bad[0])} / oracle {ref[list(idx).index(bad[0])]}")


def _census(seed, n, qmax, tmax):
    q, qo, t, to = pair_census.gen_pairs(seed, 0, n, qmax, tmax)
    return (q, qo, t, to), [s.decode() for s in pair_census.strings(q, qo)], [s.decode() for s in pair_census.strings(t, to)]


def _align(ctx, packed, max_ops=None):
    q, qo, t, to = packed
    return ctx.align_pairs(q, t, max_ops, query_offsets=qo, target_offsets=to)


@pytest.fixture(scope="module")
def census_short():
    return _census(11, 200_000, 72, 160)


@pytest.fixture(scope="module")
def census_short_result(census_short):
    with Context(0) as ctx:
        return _align(ctx, census_short[0])


def test_census_pairs_equal_the_oracle(census_short, census_short_result):
    _, qs, ts = census_short
    res = census_short_result
    assert len(res) == 200_000 and res.stats.n_aligned == 200_000 and res.stats.n_oversize == 0
    # the census's wildcard letters send these pairs to the generic kernel (found by the packed kernels on the way)
    assert (res.records["flags"] & api.R_GENERIC != 0).sum() > 1000
    _check(res, _oracle(qs, ts))
    sub = list(range(0, 200_000, 10))
    for lanes in (8, 16):
        _check(res, _oracle([qs[k] for k in sub], [ts[k] for k in sub], lanes=lanes), sub)


def test_read_sized_census_pairs_equal_the_oracle():
    packed, qs, ts = _census(41, 20_000, 260, 1000)
    with Context(0) as ctx:
        res = _align(ctx, packed)
    assert res.ops.shape[1] == 3 * max(len(x) for x in qs)
    assert not (res.records["flags"] & api.R_OPS_TRUNC).any()
    _check(res, _oracle(qs, ts))
    sub = list(range(0, 20_000, 10))
    for lanes in (8, 16):
        _check(res, _oracle([qs[k] for k in sub], [ts[k] for k in sub], lanes=lanes), sub)


@pytest.mark.parametrize("scoring", CHEAP_GAPS + [(10, 2, 9, -3), (10, 2, 2, -9)])
def test_other_scorings_equal_the_oracle(scoring):
    """the cheap-gap scorings of the striped census, match 9 (the fp16 score-only step does not apply) and mismatch -9
    (outside the tagged trace encoding)"""
    o, e, m, x = scoring
    packed, qs, ts = _census(21, 20_000, 72, 160)
    with Context(0, default_params(gap_open=o, gap_extend=e, match=m, mismatch=x)) as ctx:
        res = _align(ctx, packed)
    _check(res, _oracle(qs, ts, params=orc.default_params(gap_open=o, gap_extend=e, match=m, mismatch=x)))


def test_the_generic_kernel_gives_identical_records(census_short, census_short_result):
    with Context(0, default_params(flags=api.F_FORCE_GENERIC)) as ctx:
        res = _align(ctx, census_short[0])
    assert res.stats.n_generic == 200_000 and (res.records["flags"] & api.R_GENERIC).all()
    a, b = census_short_result.records.copy(), res.records.copy()
    a["flags"] &= ~np.uint32(api.R_GENERIC)
    b["flags"] &= ~np.uint32(api.R_GENERIC)
    assert np.array_equal(a, b) and np.array_equal(census_short_result.ops, res.ops)


def test_annotate_alignments_through_the_pair_call():
    """C1's aligned reads as (RC(read), window) pairs give what the annotate path gave them, and the batch's results
    and a replay of its kernels are unaffected by the pair call"""
    names, contigs, cfg, n = sim.config_c1()
    rd = sim.make_reads(cfg, 0, n, contigs)
    ref = contigs[0].tobytes()
    with Context(0) as ctx:
        ctx.load_reference(names, [c.tobytes() for c in contigs])
        b = ctx.alloc_batch(rd.n, int(rd.seq_off[rd.n]))
        b.fill(rd.seq4, rd.seq_off, rd.l_qseq, rd.tid, rd.pos, rd.aligned_len, rd.clip_left, rd.clip_right).run()
        rec0, ws0, ri0 = (x.copy() for x in b.results())
        al = np.nonzero(b.flags[:rd.n] & api.R_ALIGNED)[0]
        assert len(al) > 1000
        W = ctx.params.window_size
        qs, ts = [], []
        for r in al:
            so = int(rd.seq_off[r])
            qs.append(orc.revcomp_nt16(rd.seq4[so:so + (int(rd.l_qseq[r]) + 1) // 2], int(rd.l_qseq[r])))
            end = min(int(rd.pos[r]) + int(rd.aligned_len[r]) + W, len(ref))
            ts.append(ref[int(b.win_start[r]):end])
        res = ctx.align_pairs(qs, ts)
        for f in FIELDS:
            assert np.array_equal(res.records[f], getattr(b, f)[al]), f
        k = np.minimum(res.records["n_ops"], api.MAX_OPS)
        m = np.arange(api.MAX_OPS)[None, :] < k[:, None]
        assert np.array_equal(np.where(m, res.ops[:, :api.MAX_OPS], 0), np.where(m, b.ops[al], 0))
        rec1, ws1, ri1 = b.results()
        assert np.array_equal(rec0, rec1) and np.array_equal(ws0, ws1) and np.array_equal(ri0, ri1)
        assert b.replay_kernels(2) > 0
        rec2, _, _ = b.results()
        assert np.array_equal(rec0, rec2)
        b.close()


def _planted(rng, qlen, tlen):
    q = readsets.random_ref(rng, qlen).decode()
    t = list(readsets.random_ref(rng, tlen).decode())
    if qlen and tlen:
        piece = [c if rng.random() > 0.05 else rng.choice("ACGT") for c in q[:min(qlen, tlen)]]
        if qlen > 40 and rng.random() < 0.5:                       # an indel in the planted copy
            cut = rng.randrange(10, len(piece) - 10)
            piece = piece[:cut] + list("ACG") + piece[cut:] if rng.random() < 0.5 else piece[:cut] + piece[cut + 3:]
        at = rng.randrange(0, max(1, tlen - len(piece) + 1))
        t[at:at + len(piece)] = piece
        t = t[:tlen]
    return q, "".join(t)


def test_sizes_across_every_kernel():
    rng = random.Random(5)
    qs, ts = [], []
    for ql in list(range(1, 305, 3)) + [104, 105, 152, 153, 200, 201, 256, 257, 304]:   # the five row classes
        q, t = _planted(rng, ql, rng.randrange(max(8, ql // 2), 4000)); qs.append(q); ts.append(t)
    for ql in range(305, 601, 15):                                                        # generic kernel
        q, t = _planted(rng, ql, rng.randrange(300, 2000)); qs.append(q); ts.append(t)
    for tl in (5_000, 9_999, 33_000, 70_000):                                             # restaged target chunks
        q, t = _planted(rng, rng.choice((100, 250, 300)), tl); qs.append(q); ts.append(t)
    q, t = _planted(rng, 60, 1_200_000); qs.append(q); ts.append(t)                     # beyond the packed kernels
    n_checked = len(qs)
    qs += ["ACGT" * 250, "", "ACGT", ""]                                                  # oversize, empty q / t / both
    ts += ["A" * 2_200_000, "ACGT", "", ""]
    with Context(0) as ctx:
        res = ctx.align_pairs(qs, ts)
    _check(res, _oracle(qs[:n_checked], ts[:n_checked]), range(n_checked))
    assert res.stats.n_generic >= 21 and res.records["flags"][n_checked - 1] & api.R_GENERIC
    assert res.records[n_checked].tolist() == (0,) * 6 + (api.R_OVERSIZE, 0) and res.stats.n_oversize == 1
    for k in range(n_checked + 1, n_checked + 4):
        assert res.records[k].tolist() == (0,) * 8
    assert res.stats.n_aligned == n_checked


def test_contract():
    with Context(0) as ctx:
        with pytest.raises(FadeGpuError) as e:
            ctx.align_pairs(["ACGT", "ACGT", "ACGT", "AC-T"], ["ACGT"] * 4)
        assert e.value.code == -1 and "pair 3" in str(e.value)
        with pytest.raises(FadeGpuError) as e:
            ctx.align_pairs(["ACGT", "ACXT"], ["ACGT"] * 2)
        assert "pair 1" in str(e.value)
        # a submitted batch blocks the call until it is waited for
        names, contigs, cfg, n = sim.config_c1()
        ctx.load_reference(names, [c.tobytes() for c in contigs])
        rd = sim.make_reads(cfg, 0, 2000, contigs)
        b = ctx.alloc_batch(rd.n, int(rd.seq_off[rd.n]))
        b.fill(rd.seq4, rd.seq_off, rd.l_qseq, rd.tid, rd.pos, rd.aligned_len, rd.clip_left, rd.clip_right)
        b.submit()
        with pytest.raises(FadeGpuError) as e:
            ctx.align_pairs(["ACGT"], ["ACGT"])
        assert e.value.code == -4
        b.wait()
        assert ctx.align_pairs(["ACGTACGT"], ["TTACGTACGTTT"]).cigar(0) == "8="
        b.close()
    packed, qs, ts = _census(23, 5_000, 72, 160)
    with Context(0) as ctx:
        full = _align(ctx, packed)
        cut = _align(ctx, packed, max_ops=3)
    with Context(0, default_params(flags=api.F_TAGS_ONLY)) as ctx:      # tags-only does not apply: all traced back
        tags = _align(ctx, packed)
    assert np.array_equal(tags.records, full.records) and np.array_equal(tags.ops, full.ops)
    assert not (tags.records["flags"] & api.R_SCORE_ONLY).any()
    long = full.records["n_ops"] > 3
    assert long.sum() > 100
    assert np.array_equal(cut.records["n_ops"], full.records["n_ops"])
    assert np.array_equal((cut.records["flags"] & api.R_OPS_TRUNC) != 0, long)
    assert not (full.records["flags"] & api.R_OPS_TRUNC).any()
    assert np.array_equal(cut.ops, full.ops[:, :3])


def test_many_launches_give_the_same_results():
    packed, _, _ = _census(51, 200_000, 160, 700)
    with Context(0) as ctx:
        a = _align(ctx, packed)
    with Context(0, default_params(scratch_bytes=4 << 20)) as ctx:
        b = _align(ctx, packed)
    assert b.stats.kernel_launches > 3 * a.stats.kernel_launches
    assert np.array_equal(a.records, b.records) and np.array_equal(a.ops, b.ops)
