"""fadegpu_align_pairs without a GPU: the ABI surface (symbols, struct sizes in ctypes and in the D binding, loud
failure without a ctx or device), the full-CIGAR op spill of the shared walker in the host emulation, and the input
packing of Context.align_pairs."""
import ctypes as C
import functools
import os
import re

import numpy as np
import pytest

import emu_util
import pair_census
from fade_b200 import _lib, api
from oracle import oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_pair_symbols_are_declared_exported_and_bound():
    L = _lib.lib()
    hdr = open(os.path.join(ROOT, "include", "fadegpu.h")).read()
    assert re.search(r"\bint fadegpu_align_pairs\s*\(", hdr)
    assert "fadegpu_align_pairs" in _lib.ABI_SYMBOLS and hasattr(L, "fadegpu_align_pairs")
    assert C.sizeof(_lib.PairsIn) == 32 and C.sizeof(_lib.PairResult) == 32
    assert api.PAIR_RESULT_DTYPE.itemsize == 32
    assert [f[0] for f in _lib.PairResult._fields_] == list(api.PAIR_RESULT_DTYPE.names)
    d = open(os.path.join(ROOT, "integration", "fadegpu.d")).read()
    pins = {k: int(v) for k, v in re.findall(r'static assert\((\w+)\.sizeof == (\d+), "', d)}
    assert pins == {"fadegpu_pairs": 32, "fadegpu_pair_result": 32}
    assert re.search(r"\bint fadegpu_align_pairs\s*\(", d)


def test_align_pairs_fails_loudly_without_ctx_or_device():
    L = _lib.lib()
    out = (_lib.PairResult * 1)()
    pin = _lib.PairsIn()
    assert L.fadegpu_align_pairs(None, 1, C.byref(pin), 0, out, None, None) == -1   # FADEGPU_E_ARG
    assert L.fadegpu_last_error(None)
    try:
        n = api.device_count()
    except _lib.FadeGpuError:
        n = 0
    if n > 0:
        pytest.skip("a GPU is present: the device side is covered by tests/test_gpu_pairs.py")
    with pytest.raises(_lib.FadeGpuError) as e:
        api.Context(0).align_pairs(["ACGT"], ["ACGT"])
    assert e.value.code in (-5, -2)                                               # no device, no fallback


def _row_class(qlen):
    return next(r for r in (13, 19, 25, 32, 38) if 8 * r >= qlen)


def _emu_ops(q, t, cap, scoring=(10, 2, 2, -3)):
    lib = emu_util.lib()
    lib.fadeemu_align_pair_ops.restype = C.c_int
    a, b = emu_util.AlnOut(), emu_util.AlnOut()
    cq, ct = emu_util.codes(q), emu_util.codes(t)
    oa, ob = np.zeros(cap, np.uint32), np.zeros(cap, np.uint32)
    rc = lib.fadeemu_align_pair_ops(_row_class(len(q)), cq.ctypes.data_as(C.c_void_p), len(cq),
                                    ct.ctypes.data_as(C.c_void_p), len(ct), cq.ctypes.data_as(C.c_void_p), len(cq),
                                    ct.ctypes.data_as(C.c_void_p), len(ct), *scoring, 1, cap, C.byref(a), C.byref(b),
                                    oa.ctypes.data_as(C.c_void_p), ob.ctypes.data_as(C.c_void_p))
    assert rc == 0
    assert a.n_ops == b.n_ops and np.array_equal(oa, ob)
    return a, oa


@functools.lru_cache(maxsize=None)
def _long_cigar_pairs(n_want=40):
    """census pairs (gapped and low-complexity modes, read-sized) of ACGTN letters with more than 10 CIGAR ops"""
    q, qo, t, to = pair_census.gen_pairs(77, 0, 4000, 260, 1000)
    out = []
    for qs, ts in zip(pair_census.strings(q, qo), pair_census.strings(t, to)):
        qs, ts = qs.decode().upper(), ts.decode().upper()
        if set(qs + ts) - set("ACGTN"):
            continue
        r = orc.sw_trace(qs, ts, ops_cap=4096)
        if r.n_ops > 10:
            out.append((qs, ts, r))
        if len(out) == n_want:
            break
    return out


def test_op_spill_in_the_emulation_gives_the_full_forward_cigar():
    pairs = _long_cigar_pairs()
    assert len(pairs) == 40 and max(r.n_ops for _, _, r in pairs) > 20
    for qs, ts, r in pairs:
        o, ops = _emu_ops(qs, ts, 4096)
        assert (o.score, o.end_query, o.end_ref, o.beg_query, o.beg_ref, o.n_ops) == \
            (r.score, r.end_query, r.end_ref, r.beg_query, r.beg_ref, r.n_ops)
        assert list(ops[:r.n_ops]) == r.ops and not ops[r.n_ops:].any()
        assert o.flags & 8                                         # the 10-op record says R_OPS_TRUNC
        # capacity 10: exactly today's ring output; capacity c < n_ops: the first c forward ops
        _, ops10 = _emu_ops(qs, ts, 10)
        assert list(ops10) == list(o.ops)
        for cap in (1, 3, 7, r.n_ops - 1):
            _, opsc = _emu_ops(qs, ts, cap)
            assert list(opsc) == r.ops[:cap]


def test_op_spill_leaves_short_cigars_and_zero_scores_alone():
    for qs, ts in (("ACGTACGTAC", "TTACGTACGTACTT"), ("AAAA", "CCCC"), ("ACGCCACG", "TTACGTT")):
        r = orc.sw_trace(qs, ts, ops_cap=64)
        o, ops = _emu_ops(qs, ts, 64)
        assert o.n_ops == r.n_ops and list(ops[:r.n_ops]) == r.ops and not ops[r.n_ops:].any()
        assert list(o.ops[:min(10, r.n_ops)]) == r.ops[:10]


def test_pair_inputs_pack_the_same_from_lists_and_from_buffers():
    qs = ["ACGT", "", "nacgtRYKM", "=ACMGRSVTWYHKDBN"]
    ts = [b"TTGCA", b"ACGT", b"", b"xyzACGT"]
    q1, qo1, t1, to1 = api.pack_pairs(qs, ts)
    assert qo1.tolist() == [0, 4, 4, 13, 29] and to1.tolist() == [0, 5, 9, 9, 16]
    assert q1.tobytes() == "".join(qs).encode() and t1.tobytes() == b"".join(ts)
    # one buffer per side plus offsets: bytes or uint8 arrays, offsets need not start at 0
    for qb, tb in ((q1.tobytes(), t1.tobytes()), (q1, t1)):
        q2, qo2, t2, to2 = api.pack_pairs(qb, tb, query_offsets=qo1, target_offsets=to1)
        assert np.array_equal(q2, q1) and np.array_equal(qo2, qo1) and np.array_equal(t2, t1) and np.array_equal(to2, to1)
        assert qo2.dtype == np.int64 and q2.dtype == np.uint8 and q2.flags["C_CONTIGUOUS"]
    pad = np.frombuffer(b"ZZ" + q1.tobytes(), np.uint8)
    q3, qo3, _, _ = api.pack_pairs(pad, t1, query_offsets=qo1 + 2, target_offsets=to1)
    assert np.array_equal(qo3, qo1 + 2) and np.array_equal(q3, pad)
    with pytest.raises(ValueError):
        api.pack_pairs(["A", "C"], ["A"])
    with pytest.raises(ValueError):
        api.pack_pairs(q1, t1, query_offsets=qo1 + 100, target_offsets=to1)


def test_default_max_ops_cannot_truncate():
    _, qo, _, _ = api.pack_pairs(["A" * 7, "ACG", "A" * 150], ["A", "A", "A"])
    assert api.default_max_ops(qo) == 450
    assert api.default_max_ops(np.zeros(1, np.int64)) == 0
    # the bound 3 * qlen holds with room on the longest CIGARs the census produces
    for qs, _, r in _long_cigar_pairs():
        assert r.n_ops <= 3 * len(qs)
