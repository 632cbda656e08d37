"""The packed kernels at the full query height of every row class, at scorings on both sides of each number domain's
bound (tests/test_score_range.py): match 7, whose top scores (7 * 304 = 2128) do not fit the tagged trace recorder's
16 * H in int16, next to match 6, mismatch -8 / -9, match 9 and 100, mismatch 0 and the largest gap penalties.
align_pairs against the scalar oracle (every record field, the full CIGAR), F_NO_SHORTCUT and F_FORCE_GENERIC against
the default rounds, the score-only calls against the traced ones, regions on both strands against pairs, and the
annotate path at match 7.  Run with `pytest -m gpu` on a B200."""
import functools
import random

import numpy as np
import pytest

from fade_b200 import Context, api, default_params, sim
from oracle import oracle as orc
from parity_util import compare, oracle_params, run_gpu
from test_gpu_pairs import _check, _oracle
from test_gpu_regions import _rc
from test_gpu_score_only import _same_as_traced
from test_score_range import EDGE_SCORINGS, R_CLASSES, ROWS, full_height_cases

pytestmark = pytest.mark.gpu


def _params(scoring, **kw):
    o, e, m, x = scoring
    return default_params(gap_open=o, gap_extend=e, match=m, mismatch=x, **kw)


def _row_class(qlen):
    return next(r for r in R_CLASSES if 8 * r >= qlen)


@functools.lru_cache(maxsize=None)
def _cases(scoring):
    """420 pairs: six draws of the CPU file's full-height cases per row class (queries of 8R, 8R - 1 and 7R + 1 rows,
    planted exactly, with an insertion, with a deletion, 10 % substituted), and one draw behind 1,024-5,000 random
    target columns, so that the best cells lie in a later restaged target chunk; with their oracle results"""
    rng = random.Random(f"gpu {scoring}")
    qs, ts = [], []
    for _ in range(6):
        for R in R_CLASSES:
            for q, t in full_height_cases(rng, R):
                qs.append(q); ts.append(t)
    for R in R_CLASSES:
        for q, t in full_height_cases(rng, R):
            qs.append(q); ts.append("".join(rng.choice("ACGT") for _ in range(rng.randint(1024, 5000))) + t)
    o, e, m, x = scoring
    return qs, ts, _oracle(qs, ts, params=orc.default_params(gap_open=o, gap_extend=e, match=m, mismatch=x))


@functools.lru_cache(maxsize=None)
def _traced(scoring, flags=0):
    qs, ts, _ = _cases(scoring)
    with Context(0, _params(scoring, flags=flags)) as ctx:
        return ctx.align_pairs(qs, ts)


@pytest.mark.parametrize("scoring", EDGE_SCORINGS)
def test_pairs_equal_the_oracle(scoring):
    qs, ts, ref = _cases(scoring)
    res = _traced(scoring)
    assert res.stats.n_aligned == len(qs) and res.stats.n_generic == 0
    _check(res, ref)
    # the cases reach the edge: every row class, and for match 7 scores past the tagged recorder's 2047
    assert {_row_class(len(q)) for q in qs} == set(R_CLASSES) and sum(len(t) > 1024 for t in ts) == 60
    assert res.records["score"].max() == scoring[2] * ROWS
    if scoring[2] * ROWS > 2047:
        assert (res.records["score"] > 2047).sum() >= 30


@pytest.mark.parametrize("flags", [api.F_NO_SHORTCUT, api.F_FORCE_GENERIC])
@pytest.mark.parametrize("scoring", EDGE_SCORINGS)
def test_no_shortcut_and_generic_give_identical_results(scoring, flags):
    """F_NO_SHORTCUT traces round 0 (and the tagged recorder replays every block it walks); F_FORCE_GENERIC serves every
    pair from the exact int32 kernel"""
    base, res = _traced(scoring), _traced(scoring, flags)
    a, b = base.records.copy(), res.records.copy()
    if flags == api.F_FORCE_GENERIC:
        assert (b["flags"] & api.R_GENERIC).all()
        a["flags"] &= ~np.uint32(api.R_GENERIC)
        b["flags"] &= ~np.uint32(api.R_GENERIC)
    assert np.array_equal(a, b), np.nonzero(a != b)[0][:10]
    assert np.array_equal(base.ops, res.ops)


@pytest.mark.parametrize("scoring", EDGE_SCORINGS)
def test_score_pairs_equal_the_traced_call(scoring):
    qs, ts, _ = _cases(scoring)
    with Context(0, _params(scoring)) as ctx:
        s = ctx.score_pairs(qs, ts)
    _same_as_traced(s, _traced(scoring))


@pytest.mark.parametrize("scoring", EDGE_SCORINGS)
def test_regions_on_both_strands_equal_the_pairs(scoring):
    """the targets as contigs; each query on strand 0, and its nt16 reverse complement on strand 1 (which the call
    reverse-complements back): records and CIGARs of the pair call, twice"""
    qs, ts, _ = _cases(scoring)
    n = len(qs)
    args = (qs + [_rc(q) for q in qs], list(range(n)) * 2, [0] * 2 * n, [len(t) for t in ts] * 2, [0] * n + [1] * n)
    with Context(0, _params(scoring)) as ctx:
        ctx.load_reference([f"t{k}" for k in range(n)], [t.encode() for t in ts])
        res, s = ctx.align_regions(*args), ctx.score_regions(*args)
        sp = ctx.score_pairs(qs, ts)
    pairs = _traced(scoring)
    assert np.array_equal(res.records, np.concatenate([pairs.records] * 2))
    assert np.array_equal(res.ops, np.concatenate([pairs.ops] * 2))
    _same_as_traced(s, res)
    assert np.array_equal(s.records, np.concatenate([sp.records] * 2))


@pytest.mark.parametrize("flags", [0, api.F_NO_SHORTCUT])
@pytest.mark.parametrize("long_clips", [False, True])
def test_annotate_batch_at_match_7(long_clips, flags):
    """2x300 reads with indels on a C1-sized contig at (10, 2, 7, -3) against the oracle (records, CIGAR, art_left /
    art_right).  The annotate path aligns the reverse complement of the whole read, which only its artifact clip
    matches, so artifact clips of 270-295 bases are what take the scores past 2047."""
    names, contigs, _, _ = sim.config_c1()
    kw = dict(read_len=300, p_indel=0.3)
    if long_clips:
        kw.update(p_artifact=0.9, p_random_clip=0.0, p_both=0.0, clip_min_art=270, clip_max=295)
    rd = sim.make_reads(sim.default_cfg(read_seed=2001, **kw), 0, 3000, contigs)
    with Context(0, _params((10, 2, 7, -3), flags=flags)) as ctx:
        ctx.load_reference(names, [c.tobytes() for c in contigs])
        b = run_gpu(ctx, rd)
        n_al = compare(b, rd, contigs, oracle_params(ctx.params))
        high = int((b.score[:rd.n][(b.flags[:rd.n] & api.R_ALIGNED) != 0] > 2047).sum())
        b.close()
    assert n_al > 400
    if long_clips:
        assert high > 100
