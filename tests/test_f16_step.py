"""The fp16x2 score-only step (fill_step_f16 in fade_b200/csrc/sw_core.cuh): the diagonal add runs as HFMA2 on
integer scores held as fp16 subnormals.  Checks the host emulation of fma.rn.f16x2 against numpy float16 over the
operand domain the step uses, the f16_ok decision of make_consts, the emulated group
with the fp16 step against the oracle, and (on a GPU) the device instructions against the host emulation."""
import ctypes as C
import os
import random
import subprocess

import numpy as np
import pytest

import emu_util as E
import test_emu_core as T
from oracle import oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
UNIT = 0x00010001          # packed fp16 2^-24: one unit of the score grid


def _emu():
    L = E.lib()
    L.fadeemu_fma_f16x2.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64]
    L.fadeemu_fma_f16x2.restype = None
    L.fadeemu_f16_ok.argtypes = [C.c_int] * 4
    L.fadeemu_f16_ok.restype = C.c_int
    return L


def _u32(x):
    return np.ascontiguousarray(x, dtype=np.uint32)


def emu_fma(a, b, c):
    a, b, c = _u32(a), _u32(b), _u32(c)
    out = np.empty_like(a)
    _emu().fadeemu_fma_f16x2(a.ctypes.data, b.ctypes.data, c.ctypes.data, out.ctypes.data, len(a))
    return out


def numpy_fma(a, b, c):
    """a * b + c per fp16 lane, formed exactly in float64 and rounded once to float16 (exact for the operands below:
    every value is a multiple of 2^-48 below 2^4)."""
    def lane(x, sh):
        return ((x >> sh) & 0xFFFF).astype(np.uint16).view(np.float16).astype(np.float64)

    out = np.zeros(len(a), dtype=np.uint32)
    for sh in (0, 16):
        r = (lane(a, sh) * lane(b, sh) + lane(c, sh)).astype(np.float16).view(np.uint16).astype(np.uint32)
        out |= r << sh
    return out


def lut_words():
    """every word the fp16 score LUT can produce: high byte b, low byte the sign of b replicated (finite only)"""
    b = np.arange(256, dtype=np.uint32)
    w = np.where(b < 0x80, b << 8, (b << 8) | 0xFF)
    return w[(w & 0x7C00) != 0x7C00]


def pack(lo, hi):
    return _u32(lo) | (_u32(hi) << 16)


def fma_domain():
    """score word x every H in 0..2047, both lanes, lanes shuffled against each other"""
    w, n = np.meshgrid(lut_words(), np.arange(2048, dtype=np.uint32))
    w, n = w.ravel(), n.ravel()
    return pack(w, np.roll(w, 7919)), np.full(len(w), UNIT, dtype=np.uint32), pack(n, np.roll(n, 104729))


def test_fma_emulation_matches_numpy_float16():
    a, b, c = fma_domain()
    assert np.array_equal(emu_fma(a, b, c), numpy_fma(a, b, c))
    # general operands: random finite words below 2.0 (exponent field < 16), any signs
    rng = np.random.default_rng(3)
    a, b, c = (rng.integers(0, 1 << 32, size=1 << 20, dtype=np.uint64).astype(np.uint32) & 0xBFFFBFFF for _ in range(3))
    assert np.array_equal(emu_fma(a, b, c), numpy_fma(a, b, c))


def test_score_words_give_exact_integer_sums():
    """the step's view of the fp16 results: H + s exactly, a word negative as int16 where H + s < 0"""
    for sel, s in ((0x40, 2), (0xC1, -3)):     # default LUT bytes: 2.0 and -2.998
        w = (sel << 8) | (0xFF if sel & 0x80 else 0)
        n = np.arange(2048 - 2, dtype=np.uint32)
        d = emu_fma(np.full(len(n), w * 0x10001, dtype=np.uint32), np.full(len(n), UNIT, dtype=np.uint32), n * 0x10001)
        lo = (d & 0xFFFF).astype(np.uint16).view(np.int16).astype(np.int64)
        want = n.astype(np.int64) + s
        assert np.array_equal(lo[want >= 0], want[want >= 0])
        assert (lo[want < 0] <= 0).all()
        assert np.array_equal(d >> 16, d & 0xFFFF)


@pytest.mark.parametrize("scoring,ok", [((10, 2, 2, -3), 1), ((6, 1, 1, -4), 1), ((12, 3, 9, -9), 0),
                                        ((10, 2, 7, -3), 0)])
def test_f16_ok(scoring, ok):
    """the fp16 step is used only where make_consts has checked it exact (H up to max score * 304 below 2048)"""
    assert _emu().fadeemu_f16_ok(*scoring) == ok


@pytest.mark.parametrize("scoring", [(10, 2, 2, -3), (6, 1, 1, -4), (12, 3, 9, -9)])
@pytest.mark.parametrize("tagged", [1, 0, 5])
@pytest.mark.parametrize("R,maxq,maxt,iters", [(1, 8, 40, 100), (5, 40, 200, 40), (19, 152, 400, 12), (38, 304, 500, 4)])
def test_group_emulation_with_f16_step_matches_oracle(R, maxq, maxt, iters, tagged, scoring):
    """the emulated group with the fp16 fill step where f16_ok (the first two scorings) and the integer step where not
    (the third), and with bit 3 of `tagged` forcing the integer step: the same records, equal to the oracle's"""
    o, e, m, x = scoring
    p = orc.default_params(gap_open=o, gap_extend=e, match=m, mismatch=x)
    rng = random.Random(77 * R + tagged + m)
    for _ in range(iters):
        qa, ta = T.case(rng, maxq, maxt)
        qb, tb = T.case(rng, maxq, maxt)
        xa, xb = E.align_pair(R, qa, ta, qb, tb, scoring=scoring, extra_blocks=rng.randint(0, 1), tagged=tagged)
        ya, yb = E.align_pair(R, qa, ta, qb, tb, scoring=scoring, extra_blocks=rng.randint(0, 1), tagged=tagged | 8)
        assert T.got(xa) == T.got(ya) == T.expect(qa, ta, p), (R, qa, ta)
        assert T.got(xb) == T.got(yb) == T.expect(qb, tb, p), (R, qb, tb)


@pytest.fixture(scope="module")
def device_f16x2(tmp_path_factory):
    so = tmp_path_factory.mktemp("f16x2") / "libf16x2_device.so"
    subprocess.check_call(["nvcc", "-O2", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC",
                           "-shared", "-o", str(so), os.path.join(ROOT, "tests", "native", "f16x2_device.cu")])
    L = C.CDLL(str(so))
    L.f16x2_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64]
    L.f16x2_device.restype = C.c_int

    def run(a, b, c):
        a, b, c = _u32(a), _u32(b), _u32(c)
        out = np.empty_like(a)
        rc = L.f16x2_device(a.ctypes.data, b.ctypes.data, c.ctypes.data, out.ctypes.data, len(a))
        assert rc == 0, f"cudaError {rc}"
        return out
    return run


@pytest.mark.gpu
def test_device_f16x2_matches_host_emulation(device_f16x2):
    """fma.rn.f16x2 on the GPU (no flush of the subnormal scores) equals the host emulation over the whole operand
    domain of the step, and on general operands"""
    a, b, c = fma_domain()
    assert np.array_equal(device_f16x2(a, b, c), emu_fma(a, b, c))
    rng = np.random.default_rng(4)
    a, b, c = (rng.integers(0, 1 << 32, size=1 << 20, dtype=np.uint64).astype(np.uint32) & 0x7BFF7BFF |
               (rng.integers(0, 2, size=1 << 20, dtype=np.uint64).astype(np.uint32) * 0x80008000) for _ in range(3))
    assert np.array_equal(device_f16x2(a, b, c), emu_fma(a, b, c))
