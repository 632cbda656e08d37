"""fadegpu_score_pairs / fadegpu_score_regions without a GPU: the ABI surface (symbols in the header, in ABI_SYMBOLS, in
the D binding; loud failure without a ctx or a device), the Python packing and validation shared with align_pairs /
align_regions, and the end-only traceback of the shared kernel core (csrc/emu, the host lock-step emulation of one
group) against the oracle's fo_sw_trace: score and end cell, whether the end cell is in the first candidate block or
in a later one."""
import ctypes as C
import os
import random
import re

import numpy as np
import pytest

import emu_util as E
from fade_b200 import _lib, api
from oracle import oracle as orc
from test_emu_core import case

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SCORE_FNS = ("fadegpu_score_pairs", "fadegpu_score_regions")


def test_score_symbols_are_declared_exported_and_bound():
    L = _lib.lib()
    hdr = open(os.path.join(ROOT, "include", "fadegpu.h")).read()
    d = open(os.path.join(ROOT, "integration", "fadegpu.d")).read()
    for fn in SCORE_FNS + ("fadegpu_align_regions",):
        assert re.search(rf"\bint {fn}\s*\(", hdr) and re.search(rf"\bint {fn}\s*\(", d), fn
        assert fn in _lib.ABI_SYMBOLS and hasattr(L, fn), fn
    assert L.fadegpu_score_pairs.argtypes[2] == C.POINTER(_lib.PairsIn)
    assert L.fadegpu_score_regions.argtypes[2] == C.POINTER(_lib.RegionsIn)
    assert len(L.fadegpu_score_pairs.argtypes) == len(L.fadegpu_score_regions.argtypes) == 5   # no max_ops, no ops
    # the D binding pins fadegpu_regions at the header's 48 bytes, with the header's fields in order
    body = re.search(r"struct fadegpu_regions\s*\{(.*?)\}", d, re.S).group(1)
    assert re.findall(r"\*\s*(\w+);", body) == [f[0] for f in _lib.RegionsIn._fields_]
    assert "static assert(fadegpu_regions.sizeof == 48 && fadegpu_regions.strand.offsetof == 40, " in d


def test_score_calls_fail_loudly_without_ctx_or_device():
    L = _lib.lib()
    out = (_lib.PairResult * 1)()
    assert L.fadegpu_score_pairs(None, 1, C.byref(_lib.PairsIn()), out, None) == -1          # FADEGPU_E_ARG
    assert b"fadegpu_score_pairs" in L.fadegpu_last_error(None)
    assert L.fadegpu_score_regions(None, 1, C.byref(_lib.RegionsIn()), out, None) == -1
    assert b"fadegpu_score_regions" in L.fadegpu_last_error(None)
    try:
        n = api.device_count()
    except _lib.FadeGpuError:
        n = 0
    if n > 0:
        pytest.skip("a GPU is present: the device side is covered by tests/test_gpu_score_only.py")
    for call in (lambda c: c.score_pairs(["ACGT"], ["ACGT"]), lambda c: c.score_regions(["ACGT"], [0], [0], [4])):
        with pytest.raises(_lib.FadeGpuError) as e:
            call(api.Context(0))
        assert e.value.code in (-5, -2)                                                     # no device, no fallback


class _NoLib(Exception):
    pass


@pytest.mark.parametrize("args,kw", [
    ((["ACGT", "AC"], ["ACGT"]), {}),                                                     # 2 queries, 1 target
    ((b"ACGTAC", b"ACGT"), dict(query_offsets=[0, 4, 6], target_offsets=[0, 4])),
    ((b"ACGT", b"ACGT"), dict(query_offsets=[0, 8], target_offsets=[0, 4])),              # beyond the buffer
    ((b"ACGT", b"ACGT"), dict(query_offsets=[[0, 4]], target_offsets=[0, 4])),            # not 1-d
])
def test_pair_inputs_raise_as_align_pairs_does(args, kw, monkeypatch):
    """score_pairs packs and validates through pack_pairs: the same ValueErrors as align_pairs, before any call"""
    def no_lib():
        raise _NoLib()
    monkeypatch.setattr(api, "lib", no_lib)
    ctx = object.__new__(api.Context)
    errs = []
    for call in (ctx.align_pairs, ctx.score_pairs):
        with pytest.raises(ValueError) as e:
            call(*args, **kw)
        errs.append(str(e.value))
    assert errs[0] == errs[1]


@pytest.mark.parametrize("bad", [
    dict(tids=[0, 1]),
    dict(ends=[[4], [4], [4]]),
    dict(strands=[0, 1]),
    dict(tids=[0, 2 ** 31, 0]),
    dict(strands=[0, 256, 0]),
    dict(starts=[0.5, 0, 0]),
])
def test_region_inputs_raise_as_align_regions_does(bad, monkeypatch):
    def no_lib():
        raise _NoLib()
    monkeypatch.setattr(api, "lib", no_lib)
    ctx = object.__new__(api.Context)
    kw = dict(tids=[0, 0, 0], starts=[0, 0, 0], ends=[4, 4, 4], strands=[0, 1, 0])
    kw.update(bad)
    errs = []
    for call in (ctx.align_regions, ctx.score_regions):
        with pytest.raises(ValueError) as e:
            call(["ACGT"] * 3, kw["tids"], kw["starts"], kw["ends"], kw["strands"])
        errs.append(str(e.value))
    assert errs[0] == errs[1]


def test_valid_inputs_reach_the_library(monkeypatch):
    """valid inputs pass the packing and arrive at the C call with the ABI layout (stopped there)"""
    seen = {}

    class Fake:
        def fadegpu_score_pairs(self, h, n, pin, rec, st):
            seen["pairs"] = (n, pin._obj.query_off)
            raise _NoLib()

        def fadegpu_score_regions(self, h, n, rin, rec, st):
            seen["regions"] = n
            raise _NoLib()
    monkeypatch.setattr(api, "lib", lambda: Fake())
    ctx = object.__new__(api.Context)
    ctx._h = None
    with pytest.raises(_NoLib):
        ctx.score_pairs(["ACGT", "", "acg"], ["ACGTT", "A", ""])
    with pytest.raises(_NoLib):
        ctx.score_regions(b"ACGTAC", [0, 1], [0, 5], [4, 9], [1, 0], query_offsets=[0, 4, 6])
    assert seen["pairs"][0] == 3 and seen["regions"] == 2


# ---- the end-only traceback of the shared core, on the host emulation ----

def _emu():
    L = E.lib()
    if not getattr(L, "_score_bound", False):
        L.fadeemu_score_pair.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int,
                                         C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                         C.POINTER(E.AlnOut), C.POINTER(E.AlnOut), C.c_void_p]
        L.fadeemu_score_pair.restype = C.c_int
        L._score_bound = True
    return L


def score_pair(R, qa, ta, qb, tb, scoring=(10, 2, 2, -3), extra_blocks=0, tagged=0):
    """(record a, record b, [scans a, first candidate block a, scans b, first candidate block b])"""
    a, b = E.AlnOut(), E.AlnOut()
    ca, cta, cb, ctb = E.codes(qa), E.codes(ta), E.codes(qb), E.codes(tb)
    info = np.zeros(4, np.int32)
    rc = _emu().fadeemu_score_pair(R, ca.ctypes.data, len(ca), cta.ctypes.data, len(cta), cb.ctypes.data, len(cb),
                                   ctb.ctypes.data, len(ctb), *scoring, extra_blocks, tagged, C.byref(a), C.byref(b),
                                   info.ctypes.data)
    if rc:
        raise RuntimeError(f"fadeemu_score_pair rc={rc}")
    return a, b, info.tolist()


def _check(R, q, t, x, params=None):
    """x against fo_sw_trace: score and end cell; no begin cell, no CIGAR; returns the end cell's block"""
    r = orc.sw_trace(q, t, params)
    want = (r.score, r.end_query, r.end_ref) if r.score > 0 else (0, 0, 0)
    assert (x.score, x.end_query, x.end_ref) == want, (R, q, t)
    assert (x.beg_query, x.beg_ref, x.n_ops, x.flags) == (0, 0, 0, 1) and not any(x.ops)
    return (x.end_ref + x.end_query // R) // 32      # the skewed block (t = j + g) that holds the end cell


def _tie_case(rng, maxq, maxt):
    """repeats of one motif: many cells tie at the maximum, in several candidate blocks of several threads"""
    motif = "".join(rng.choice("ACGT") for _ in range(rng.randint(1, 6)))
    q = (motif * maxq)[:rng.randint(1, maxq)]
    t = "".join(rng.choice((motif, motif, motif[::-1], "A", "GT")) for _ in range(maxt))[:rng.randint(1, maxt)]
    return q, t


@pytest.mark.parametrize("tagged", [0, 2, 8, 16])   # bit 1: no diagonal shortcut (must change nothing); 3 / 4: steps
@pytest.mark.parametrize("R,maxq,maxt,iters", [(1, 8, 60, 400), (2, 16, 90, 400), (3, 24, 160, 300),
                                               (5, 40, 220, 200), (13, 104, 400, 60), (19, 152, 500, 60),
                                               (25, 200, 500, 16), (32, 256, 600, 16), (38, 304, 600, 12)])
def test_end_only_matches_the_oracle(R, maxq, maxt, iters, tagged):
    rng = random.Random(4000 + 10 * R + tagged)
    for it in range(iters):
        gen = _tie_case if it % 3 == 2 else case
        qa, ta = gen(rng, maxq, maxt)
        qb, tb = gen(rng, maxq, maxt)
        xa, xb, _ = score_pair(R, qa, ta, qb, tb, extra_blocks=rng.randint(0, 1), tagged=tagged)
        _check(R, qa, ta, xa)
        _check(R, qb, tb, xb)


def test_end_only_other_scorings():
    rng = random.Random(12)
    for scoring in ((12, 3, 9, -9), (5, 1, 1, -1), (10, 2, 2, -8), (3, 3, 4, -2)):
        p = orc.default_params(gap_open=scoring[0], gap_extend=scoring[1], match=scoring[2], mismatch=scoring[3])
        for _ in range(80):
            qa, ta = case(rng, 40, 200)
            qb, tb = _tie_case(rng, 40, 200)
            xa, xb, _ = score_pair(5, qa, ta, qb, tb, scoring=scoring)
            _check(5, qa, ta, xa, p)
            _check(5, qb, tb, xb, p)


def _late_end_case(rng, R):
    """an end cell in a later candidate block: thread g1 reaches S first at skewed step t1 = 32 b + 31 (the last of
    block b), with an A-run ending at (i1, j1); thread g2 >= g1 + 2 reaches S with a G-run ending at an earlier column
    j2 = j1 - d, whose step j2 + g2 lies in block b + 1.  P3 takes the first column: (i2, j2)."""
    g1 = rng.randint(0, 5)
    g2 = rng.randint(g1 + 2, 7)
    d = rng.randint(1, g2 - g1 - 1)
    i1, i2 = g1 * R + rng.randrange(R), g2 * R + rng.randrange(R)
    L = min(rng.randint(1, d), i1 + 1)
    j1 = 32 * rng.randint(0, 3) + 31 - g1
    j2 = j1 - d
    q = ["C"] * rng.randint(i2 + 1, 8 * R)
    t = ["T"] * (j1 + 1 + rng.randint(0, 40))
    for k in range(L):
        q[i1 - k], t[j1 - k] = "A", "A"
        q[i2 - k], t[j2 - k] = "G", "G"
    return "".join(q), "".join(t), (j1 + g1) // 32


def test_both_scan_outcomes_are_covered():
    """random, planted, gapped and tie-heavy cases put the end cell in the first candidate block (after one scan or
    several); constructed ones put it in a later block, which the scan reaches in a later round"""
    rng = random.Random(21)
    first = multi = 0
    for it in range(3000):
        R = rng.choice((1, 2, 3, 5))
        gen = (case, _tie_case)[it & 1]
        qa, ta = gen(rng, 8 * R, 40 * R)
        qb, tb = gen(rng, 8 * R, 40 * R)
        xa, xb, info = score_pair(R, qa, ta, qb, tb, extra_blocks=rng.randint(0, 1))
        for q, t, x, (scans, fb) in ((qa, ta, xa, info[:2]), (qb, tb, xb, info[2:])):
            blk = _check(R, q, t, x)
            if scans == 0:
                assert x.score == 0 and fb == -1
                continue
            assert 1 <= scans <= 8 and blk >= fb             # at most one scan per candidate thread (FG = 8)
            multi += scans > 1
            first += blk == fb
    assert first > 4000 and multi > 50, (first, multi)
    for _ in range(400):
        R = rng.choice((1, 2, 3, 5, 13, 19, 38))
        qa, ta, b0 = _late_end_case(rng, R)
        qb, tb = case(rng, 8 * R, 200)
        xa, xb, info = score_pair(R, qa, ta, qb, tb)
        assert _check(R, qa, ta, xa) == b0 + 1 and info[:2] == [2, b0], (R, qa, ta, info)
        _check(R, qb, tb, xb)
