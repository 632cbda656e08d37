"""Score range of the packed kernels' number domains, at the full query height of every row class.

The packed kernels hold scores in three narrow domains: int16x2 (every fill step, the plain trace recorder, the
checkpoints), fp16 subnormals (fill_step_f16 / fill_step_f16x2, exact up to 2047) and the tagged domain 16*score + tag
in an int16 lane (the tagged trace recorder).  Which domain holds depends on the scoring and on the query height
together; fadegpu_create accepts match 1..100, mismatch -100..0, open up to 1000 and 1 <= extend <= open, and the
packed kernels take up to FG * 38 = 304 query rows.  This file checks make_consts' choices against the extreme values
of each domain, derived here from the recurrences, and runs the host emulation of one group (csrc/emu, the same
sw_core.cuh code as the kernels) against fo_sw_trace at scorings on both sides of every bound, with queries as tall as
each row class takes."""
import ctypes as C
import random

import numpy as np
import pytest

import emu_util as E
from oracle import oracle as orc
from test_emu_core import expect, got
from test_score_only import score_pair

ROWS = 8 * 38                       # tallest packed query (FG * 38)
R_CLASSES = (13, 19, 25, 32, 38)
I16 = (-32768, 32767)
I8 = (-128, 127)
FULL_CAP = 1024                     # op words of the full-CIGAR spill: more than any CIGAR of these cases

# (open, extend, match, mismatch) on both sides of the bounds: match 7 (16 * 7 * 304 wraps int16; the tagged recorder
# must not take it) next to match 6 (the largest it takes), mismatch -8 / -9 (the tagged LUT byte), match 9 and 100
# (beyond the fp16 steps), mismatch 0, and the largest gap penalties
EDGE_SCORINGS = [(10, 2, 2, -3), (10, 2, 6, -3), (10, 2, 7, -3), (10, 2, 7, -8), (3, 1, 8, -8), (12, 3, 9, -9),
                 (1000, 1000, 100, -100), (2, 1, 100, -100), (1, 1, 1, 0), (1000, 1000, 6, -8)]


def _emu():
    L = E.lib()
    L.fadeemu_align_pair_ops.argtypes = [C.c_int] + [C.c_void_p, C.c_int] * 4 + [C.c_int] * 6 + \
        [C.POINTER(E.AlnOut), C.POINTER(E.AlnOut), C.c_void_p, C.c_void_p]
    L.fadeemu_align_pair_ops.restype = C.c_int
    return L


def _fits(lo, hi, rng):
    return rng[0] <= lo and hi <= rng[1]


def _domains(open_, extend, match, mismatch):
    """Does each domain hold every value its steps form for this scoring at up to ROWS query rows?
    H lies in [0, match * ROWS] (the best ungapped run); a diagonal candidate Hdiag + s in [mismatch, match * ROWS]
    (Hdiag <= match * (rows above)); E and F start at -open and each step forms max(H - open, E - extend) from E >= -open,
    so the sums reach -open - extend."""
    hmax = match * ROWS
    plain = (_fits(mismatch, match, I8)                                 # PRMT LUT bytes, sign-extended
             and _fits(mismatch, hmax, I16) and _fits(-open_ - extend, hmax, I16))
    # fp16 steps: H + s must be an exact fp16 subnormal / first-binade integer (E and F stay int16 as in `plain`)
    f16 = plain and hmax <= 2047
    # tagged: LUT bytes 16 s + 8; H with its tag 16 H + 15; diagonal candidates 16 (Hdiag + s) + 8; the gap sums
    # 16 (E - extend) + 1 and 16 (F - extend) + 2 from E, F >= -16 open, and the packed -16 open
    tagged = (_fits(16 * mismatch + 8, 16 * match + 8, I8)
              and _fits(16 * mismatch + 8, 16 * hmax + 15, I16)
              and _fits(16 * (-open_ - extend) + 1, 16 * hmax + 15, I16)
              and _fits(-16 * open_, 0, I16))
    return plain, f16, tagged


def _contract_scorings():
    for open_, extend in ((1, 1), (10, 2), (1000, 1), (1000, 1000)):
        for match in range(1, 101):
            for mismatch in (0, -1, -3, -8, -9, -100):
                yield open_, extend, match, mismatch


def test_make_consts_picks_only_domains_that_hold_the_scores():
    L = E.lib()
    for fn in ("fadeemu_tagged_ok", "fadeemu_f16_ok"):
        getattr(L, fn).argtypes = [C.c_int] * 4
        getattr(L, fn).restype = C.c_int
    L.fadeemu_f16_pair.argtypes = [C.c_int] * 4 + [C.c_void_p]
    L.fadeemu_f16_pair.restype = None
    pair = np.zeros(4, np.uint32)
    n = tagged_n = f16_n = 0
    for sc in _contract_scorings():
        plain, f16, tagged = _domains(*sc)
        assert plain, sc                         # every validated scoring fits the int16 steps and checkpoints
        L.fadeemu_f16_pair(*sc, pair.ctypes.data)
        f16_ok, f16_pair_ok, tagged_ok = L.fadeemu_f16_ok(*sc), int(pair[0]), L.fadeemu_tagged_ok(*sc)
        assert not (f16_ok or f16_pair_ok) or f16, sc
        # the tagged recorder takes exactly the scorings it can hold (where it cannot, the plain recorder is exact)
        assert tagged_ok == tagged, sc
        n += 1
        tagged_n += tagged_ok
        f16_n += f16_ok
    assert n == 2400 and tagged_n == 4 * 6 * 4 and f16_n > 0    # tagged: match 1..6, mismatch >= -8
    # the bound sits between match 6 (6 * 304 = 1824) and match 7 (2128: 16 * 2128 wraps int16)
    assert L.fadeemu_tagged_ok(10, 2, 7, -3) == 0 and L.fadeemu_tagged_ok(10, 2, 6, -3) == 1
    assert L.fadeemu_tagged_ok(10, 2, 2, -3) == 1 and L.fadeemu_tagged_ok(10, 2, 2, -9) == 0


def _rnd(rng, n):
    return "".join(rng.choice("ACGT") for _ in range(n))


def full_height_cases(rng, R):
    """(query, target) pairs at the full height of row class R: queries of 8R, 8R - 1 and 7R + 1 rows planted exactly,
    with a 1-5-base insertion, with a 1-5-base deletion and with 10 % substitutions, between random flanks of 0-60
    bases"""
    out = []
    for ql in (8 * R, 8 * R - 1, 7 * R + 1):
        q = _rnd(rng, ql)
        cut, n = rng.randint(ql // 4, 3 * ql // 4), rng.randint(1, 5)
        noisy = "".join(c if rng.random() > 0.1 else rng.choice("ACGT") for c in q)
        for body, query in ((q, q), (q[:cut] + q[cut + n:], q), (q[:cut] + _rnd(rng, n) + q[cut:], q), (q, noisy)):
            out.append((query, _rnd(rng, rng.randint(0, 60)) + body + _rnd(rng, rng.randint(0, 60))))
    return out


def _ops_call(R, qa, ta, qb, tb, scoring, tagged):
    a, b = E.AlnOut(), E.AlnOut()
    ca, cta, cb, ctb = E.codes(qa), E.codes(ta), E.codes(qb), E.codes(tb)
    oa, ob = np.zeros(FULL_CAP, np.uint32), np.zeros(FULL_CAP, np.uint32)
    rc = _emu().fadeemu_align_pair_ops(R, ca.ctypes.data, len(ca), cta.ctypes.data, len(cta), cb.ctypes.data, len(cb),
                                       ctb.ctypes.data, len(ctb), *scoring, tagged, FULL_CAP, C.byref(a), C.byref(b),
                                       oa.ctypes.data, ob.ctypes.data)
    assert rc == 0, (R, scoring, tagged, rc)
    return (a, oa), (b, ob)


@pytest.mark.parametrize("scoring", EDGE_SCORINGS)
def test_full_height_emulation_equals_the_oracle(scoring):
    """every row class at its full height, in every emulation mode (bit 0: tagged recorder where make_consts allows it,
    bit 1: no diagonal shortcut, bit 2: scan-only first replay as round 0 on the device), the score-only calls, and the
    full CIGAR of the pair call's op spill"""
    o, e, m, x = scoring
    p = orc.default_params(gap_open=o, gap_extend=e, match=m, mismatch=x)
    rng = random.Random(str(scoring))
    top = 0
    for R in R_CLASSES:
        cases = full_height_cases(rng, R)
        want = {}
        for q, t in cases:
            r = orc.sw_trace(q, t, p, ops_cap=4096)
            want[q, t] = r
            top = max(top, r.score)
        for (qa, ta), (qb, tb) in zip(cases[0::2], cases[1::2]):
            for tagged in (1, 0, 3, 5):
                try:
                    xa, xb = E.align_pair(R, qa, ta, qb, tb, scoring=scoring, tagged=tagged)
                except RuntimeError as ex:          # a candidate that never finds its end cell (rc -3)
                    pytest.fail(f"R {R} tagged {tagged} qlen {len(qa)}/{len(qb)}: {ex}")
                assert got(xa) == expect(qa, ta, p), (R, tagged, qa, ta)
                assert got(xb) == expect(qb, tb, p), (R, tagged, qb, tb)
            for tagged in (5, 3):                   # the device's default rounds, and F_NO_SHORTCUT's
                for (x_, ops), q, t in zip(_ops_call(R, qa, ta, qb, tb, scoring, tagged), (qa, qb), (ta, tb)):
                    r = want[q, t]
                    assert (x_.score, x_.n_ops) == (r.score, r.n_ops), (R, tagged, q, t)
                    assert orc.cigar_string(ops[:x_.n_ops]) == orc.cigar_string(r.ops), (R, tagged, q, t)
                    assert not ops[x_.n_ops:].any()
            sa, sb, _ = score_pair(R, qa, ta, qb, tb, scoring=scoring)
            for x_, q, t in ((sa, qa, ta), (sb, qb, tb)):
                r = want[q, t]
                assert (x_.score, x_.end_query, x_.end_ref) == (r.score, r.end_query, r.end_ref), (R, q, t)
    # the exact 304-row plant reaches match * 304: for match 7 past 2047, the tagged domain's bound
    assert top == m * ROWS
