"""CPU check of the shared kernel core (fade_b200/csrc/sw_core.cuh) through the host lock-step
emulation of one 8-thread group (csrc/emu/emu.cu): packed DPX-style DP step, skewed checkpoints,
block replay with plain and tagged trace recording, end-cell rule, traceback walker -- against
the oracle, bit-exact, on random / planted / gapped / N-containing / tie-heavy inputs."""
import random

import pytest

import emu_util as E
from oracle import oracle as orc


def rnd(rng, n, alpha="ACGT"):
    return "".join(rng.choice(alpha) for _ in range(n))


def mutate(rng, frag, alpha):
    frag = list(frag)
    for _ in range(rng.randint(0, 4)):
        if frag:
            k = rng.randrange(len(frag))
            r = rng.random()
            if r < 0.4:
                frag[k] = rng.choice(alpha)
            elif r < 0.7:
                del frag[k:k + rng.randint(1, 3)]
            else:
                frag[k:k] = list(rnd(rng, rng.randint(1, 3), alpha))
    return "".join(frag)


def case(rng, maxq, maxt):
    alpha = rng.choice(["ACGT", "ACGTN", "AC", "A"])
    m = rng.randint(1, maxt)
    t = rnd(rng, m, alpha)
    if rng.random() < 0.7 and m > 3:
        a = rng.randint(0, m - 2)
        b = rng.randint(a + 1, min(m, a + maxq))
        core = mutate(rng, t[a:b], alpha)
        pre = rnd(rng, rng.randint(0, max(0, maxq - len(core)) // 2), alpha)
        q = pre + core
        q = q + rnd(rng, rng.randint(0, max(0, maxq - len(q))), alpha)
        q = q[:maxq] or "A"
    else:
        q = rnd(rng, rng.randint(1, maxq), alpha)
    return q, t


def expect(q, t, params=None):
    r = orc.sw_trace(q, t, params)
    if r.score == 0:
        return (0, 0, 0, 0, 0, 0, [])
    return (r.score, r.end_query, r.end_ref, r.beg_query, r.beg_ref, r.n_ops, r.ops[:E.OPS_CAP])


def got(x):
    return (x.score, x.end_query, x.end_ref, x.beg_query, x.beg_ref, x.n_ops,
            [x.ops[k] for k in range(min(x.n_ops, E.OPS_CAP))])


# bit 0: tagged trace, 1: no diagonal shortcut, 2: the first replay scans with the score-only step and records no trace
# (round 0 on the device)
@pytest.mark.parametrize("tagged", [1, 0, 3, 2, 5])
@pytest.mark.parametrize("R,maxq,maxt,iters", [(1, 8, 40, 300), (2, 16, 90, 300), (3, 24, 120, 200),
                                               (5, 40, 200, 120), (13, 104, 300, 40), (19, 152, 400, 40),
                                               (25, 200, 400, 10), (32, 256, 500, 12), (38, 304, 500, 8)])
def test_group_emulation_matches_oracle(R, maxq, maxt, iters, tagged):
    rng = random.Random(1000 * R + (tagged & 1))
    for _ in range(iters):
        qa, ta = case(rng, maxq, maxt)
        qb, tb = case(rng, maxq, maxt)
        xa, xb = E.align_pair(R, qa, ta, qb, tb, extra_blocks=rng.randint(0, 1), tagged=tagged)
        assert got(xa) == expect(qa, ta), (R, qa, ta)
        assert got(xb) == expect(qb, tb), (R, qb, tb)


@pytest.mark.parametrize("tagged", [1, 3, 5])
def test_long_gaps_and_long_alignments(tagged):
    """gap runs longer than one checkpoint block and full-length alignments across many blocks,
    with and without the ungapped-diagonal shortcut of the traceback."""
    rng = random.Random(5)
    for _ in range(30):
        core = rnd(rng, 150)
        gap = rng.randint(5, 60)
        cut = rng.randint(40, 110)
        t = rnd(rng, rng.randint(0, 200)) + core[:cut] + rnd(rng, gap) + core[cut:] + rnd(rng, rng.randint(0, 200))
        q2 = core[:cut] + core[cut + rng.randint(1, 30):]      # deletion from the query side
        xa, xb = E.align_pair(19, core, t, q2 or "A", t, tagged=tagged)
        assert got(xa) == expect(core, t)
        assert got(xb) == expect(q2 or "A", t)


def test_other_scoring_uses_plain_trace():
    """scoring outside the tagged encoding (|16*s+8| > 127) must fall back to the plain recorder."""
    rng = random.Random(9)
    p = orc.default_params(gap_open=12, gap_extend=3, match=9, mismatch=-9)
    for _ in range(60):
        qa, ta = case(rng, 40, 150)
        qb, tb = case(rng, 40, 150)
        xa, xb = E.align_pair(5, qa, ta, qb, tb, scoring=(12, 3, 9, -9))
        assert got(xa) == expect(qa, ta, p)
        assert got(xb) == expect(qb, tb, p)


def test_accept_predicates_in_result_flags():
    # K1 of SURVEY 8c: 10S10=, score 20: left accepted for clip_len <= 11 (5*20 > 9*n), not 12
    q, t = "AAAAAAAAAACATTAGCCAT", "GGGGGCATTAGCCATGGGGG"
    a, b = E.align_pair(3, q, t, q, t, clips=(11, 0, 12, 0))
    assert a.flags & 2 and not (b.flags & 2)
    # right side needs a trailing S and first op '=': 3=5S (K4)
    a, b = E.align_pair(1, "ACGCCACG", "TTACGTT", "ACGCCACG", "TTACGTT", clips=(0, 3, 0, 4), min_length=2)
    assert a.flags & 4 and not (b.flags & 4)      # 5*6 > 9*3 but not > 9*4
    # below the length floor nothing is accepted
    a, b = E.align_pair(1, "ACGCCACG", "TTACGTT", "ACGCCACG", "TTACGTT", clips=(0, 3, 0, 3), min_length=5)
    assert not (a.flags & 6)


def test_prmt_emulation_matches_ptx_semantics():
    L = E.lib()
    assert L.fadeemu_prmt(0xFDFDFD02, 0xFDFDFDFD, 0x8080) == 0x00020002      # both lanes match (+2)
    assert L.fadeemu_prmt(0xFDFDFD02, 0xFDFDFDFD, 0x8091) == 0x0002FFFD      # lane a mismatch (-3)
    for nib, code in {1: 2, 2: 3, 4: 1, 8: 0, 15: 4, 0: 5, 3: 5, 5: 5}.items():
        assert L.fadeemu_comp_code_of_nt16(nib) == code


@pytest.mark.parametrize("tagged", [1, 3, 5])
def test_diagonal_shortcut_edge_cases(tagged):
    """paths that start exactly at query row 0 / target column 0, long mismatch-rich diagonals and
    competing gapped alternatives: the proof-based shortcut must agree with the replayed traceback."""
    rng = random.Random(77)
    for _ in range(150):
        n = rng.randint(40, 150)
        core = rnd(rng, n)
        noisy = "".join(c if rng.random() > 0.08 else rng.choice("ACGT") for c in core)
        kind = rng.randrange(4)
        if kind == 0:      # alignment begins at target column 0 and query row 0
            q, t = noisy, core + rnd(rng, rng.randint(0, 150))
        elif kind == 1:    # begins at target column 0, query has a prefix
            q, t = rnd(rng, rng.randint(1, 40))[: 152 - n] + noisy, core + rnd(rng, rng.randint(0, 100))
        elif kind == 2:    # begins at query row 0 deep inside the target
            q, t = noisy, rnd(rng, rng.randint(33, 300)) + core + rnd(rng, rng.randint(0, 60))
        else:              # a gap in the middle: the diagonal proof must fail and the replay take over
            cut = rng.randint(15, n - 15)
            q, t = noisy, rnd(rng, rng.randint(0, 200)) + core[:cut] + rnd(rng, rng.randint(1, 6)) + core[cut:]
        q = q[:152]
        xa, xb = E.align_pair(19, q, t, q[::-1], t, tagged=tagged, extra_blocks=rng.randint(0, 1))
        assert got(xa) == expect(q, t), (q, t)
        assert got(xb) == expect(q[::-1], t)
