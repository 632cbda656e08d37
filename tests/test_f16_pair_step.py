"""The row-pair fp16 score-only step (fill_step_f16x2 in fade_b200/csrc/sw_core.cuh): one substitution lookup forms the
score words of two query rows, the second by an IMAD (w * 256 + c), so a word's low byte is one of the LUT bytes or
the addend c instead of the sign of its high byte.  Checks make_consts' choice of bytes against numpy float16 over that
low-byte domain, that the exactness check rejects a choice with a tie, the f16_pair_ok decision, and the emulated group
with the pair step against the oracle and against the single-row and integer steps."""
import ctypes as C
import random

import numpy as np
import pytest

import emu_util as E
import test_emu_core as T
from oracle import oracle as orc

# (scoring, f16_ok, f16_pair_ok): (10, 2, 2, -8) passes the single-row check (0xC7FF = -7.996) but no pair of high
# bytes holds -8 within half a unit below both LUT bytes (its candidates need a low byte < 64 or > 128, and 2.0's
# candidates are 0x3E..0x40); the last two exceed the fp16 integer range (max score * 304 > 2047)
SCORINGS = [((10, 2, 2, -3), 1, 1), ((6, 1, 1, -4), 1, 1), ((10, 2, 2, -8), 1, 0), ((12, 3, 9, -9), 0, 0),
            ((10, 2, 7, -3), 0, 0)]


def _emu():
    L = E.lib()
    L.fadeemu_f16_ok.argtypes = [C.c_int] * 4
    L.fadeemu_f16_ok.restype = C.c_int
    L.fadeemu_f16_pair.argtypes = [C.c_int] * 4 + [C.c_void_p]
    L.fadeemu_f16_pair.restype = None
    L.fadeemu_f16_pair_exact.argtypes = [C.c_int] * 4 + [C.c_uint32] * 3
    L.fadeemu_f16_pair_exact.restype = C.c_int
    return L


def pair_choice(scoring):
    out = np.zeros(4, dtype=np.uint32)
    _emu().fadeemu_f16_pair(*scoring, out.ctypes.data)
    return [int(v) for v in out]   # ok, high byte of match, of mismatch, addend c


def f16_value(words):
    return np.asarray(words, dtype=np.uint16).view(np.float16).astype(np.float64)


@pytest.mark.parametrize("scoring,ok,pair_ok", SCORINGS)
def test_f16_pair_ok(scoring, ok, pair_ok):
    assert _emu().fadeemu_f16_ok(*scoring) == ok
    assert pair_choice(scoring)[0] == pair_ok


@pytest.mark.parametrize("scoring", [s for s, _, p in SCORINGS if p])
def test_pair_words_give_exact_integer_sums(scoring):
    """every word the pair step forms (high byte pm / px, low byte pm, px or c) added to every H the packed kernels
    reach, in numpy float16 arithmetic: H + s exactly where it is positive, a word not positive as int16 elsewhere"""
    _, _, match, mismatch = scoring
    _, pm, px, c = pair_choice(scoring)
    top = max(match, mismatch) * 8 * 38
    n = np.arange(top + 1, dtype=np.float64)
    for hb, s in ((pm, match), (px, mismatch)):
        for lb in (pm, px, c):
            w = f16_value([(hb << 8) | lb])[0]
            d = (w * 2.0 ** -24 + n * 2.0 ** -24).astype(np.float16).view(np.int16)
            want = n.astype(np.int64) + s
            assert np.array_equal(d[want > 0], want[want > 0]), (hex(hb), hex(lb))
            assert (d[want <= 0] <= 0).all(), (hex(hb), hex(lb))


def test_pair_exactness_check_rejects_ties():
    """0xC1 with the addend 0 forms 0xC100 = -2.5, which rounds H - 2.5 to even: not exact.  The same bytes with a non-zero
    addend are exact, and so is 0xC2 with addend 0 (0xC2xx = -3.0 .. -3.498)."""
    L = _emu()
    assert L.fadeemu_f16_pair_exact(10, 2, 2, -3, 0x40, 0xC1, 0) == 0
    assert L.fadeemu_f16_pair_exact(10, 2, 2, -3, 0x40, 0xC1, 0xFF) == 1
    assert L.fadeemu_f16_pair_exact(10, 2, 2, -3, 0x40, 0xC2, 0) == 1
    assert L.fadeemu_f16_pair_exact(6, 1, 1, -4, 0x3C, 0xC4, 0) == 0     # 0xC4C4 = -4.77 rounds to -5


@pytest.mark.parametrize("scoring", [(10, 2, 2, -3), (6, 1, 1, -4), (10, 2, 2, -8)])
@pytest.mark.parametrize("tagged", [1, 0, 5])
@pytest.mark.parametrize("R,maxq,maxt,iters", [(1, 8, 40, 100), (2, 16, 60, 60), (5, 40, 200, 40), (19, 152, 400, 12),
                                               (38, 304, 500, 4)])
def test_group_emulation_with_pair_step_matches_oracle(R, maxq, maxt, iters, tagged, scoring):
    """the emulated group with the step make_consts chose (the pair step for the first two scorings, the single-row fp16
    step for the third), with bit 4 of `tagged` forcing the single-row fp16 step and with bit 3 the integer step: the
    same records, equal to the oracle's (odd R pairs its last row with a padding code)"""
    o, e, m, x = scoring
    p = orc.default_params(gap_open=o, gap_extend=e, match=m, mismatch=x)
    rng = random.Random(91 * R + tagged - x)
    for _ in range(iters):
        qa, ta = T.case(rng, maxq, maxt)
        qb, tb = T.case(rng, maxq, maxt)
        extra = rng.randint(0, 1)
        xa, xb = E.align_pair(R, qa, ta, qb, tb, scoring=scoring, extra_blocks=extra, tagged=tagged)
        ya, yb = E.align_pair(R, qa, ta, qb, tb, scoring=scoring, extra_blocks=extra, tagged=tagged | 16)
        za, zb = E.align_pair(R, qa, ta, qb, tb, scoring=scoring, extra_blocks=extra, tagged=tagged | 8)
        assert T.got(xa) == T.got(ya) == T.got(za) == T.expect(qa, ta, p), (R, qa, ta)
        assert T.got(xb) == T.got(yb) == T.got(zb) == T.expect(qb, tb, p), (R, qb, tb)
