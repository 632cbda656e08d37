"""fadegpu_align_regions without a GPU: the ABI surface (symbol, the 48-byte fadegpu_regions in ctypes and in the
header, loud failure without a ctx or device) and the input packing and validation of Context.align_regions."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from fade_b200 import _lib, api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_region_symbol_is_declared_exported_and_bound():
    L = _lib.lib()
    hdr = open(os.path.join(ROOT, "include", "fadegpu.h")).read()
    assert re.search(r"\bint fadegpu_align_regions\s*\(", hdr)
    assert "fadegpu_align_regions" in _lib.ABI_SYMBOLS and hasattr(L, "fadegpu_align_regions")
    assert L.fadegpu_align_regions.argtypes[2] == C.POINTER(_lib.RegionsIn)


def test_regions_struct_matches_the_header():
    assert C.sizeof(_lib.RegionsIn) == 48
    hdr = open(os.path.join(ROOT, "include", "fadegpu.h")).read()
    body = re.search(r"typedef struct fadegpu_regions \{(.*?)\} fadegpu_regions;\s*/\* (\d+) bytes", hdr, re.S)
    assert body and int(body.group(2)) == 48
    names = re.findall(r"\*\s*(\w+)", re.sub(r"/\*.*?\*/", "", body.group(1)))
    assert names == [f[0] for f in _lib.RegionsIn._fields_]


def test_align_regions_fails_loudly_without_ctx_or_device():
    L = _lib.lib()
    out = (_lib.PairResult * 1)()
    rin = _lib.RegionsIn()
    assert L.fadegpu_align_regions(None, 1, C.byref(rin), 0, out, None, None) == -1   # FADEGPU_E_ARG
    assert b"fadegpu_align_regions" in L.fadegpu_last_error(None)
    try:
        n = api.device_count()
    except _lib.FadeGpuError:
        n = 0
    if n > 0:
        pytest.skip("a GPU is present: the device side is covered by tests/test_gpu_regions.py")
    with pytest.raises(_lib.FadeGpuError) as e:
        api.Context(0).align_regions(["ACGT"], [0], [0], [4])
    assert e.value.code in (-5, -2)                                               # no device, no fallback


def test_region_inputs_pack_to_the_abi_dtypes():
    q, qo, tid, start, end, strand = api.pack_regions(["ACGT", "", "nRYK"], [0, 2, 1], [0, 10, 5], [4, 10, 9])
    assert qo.tolist() == [0, 4, 4, 8] and q.tobytes() == b"ACGTnRYK"
    assert tid.dtype == np.int32 and start.dtype == np.int64 and end.dtype == np.int64 and strand.dtype == np.uint8
    assert tid.tolist() == [0, 2, 1] and start.tolist() == [0, 10, 5] and end.tolist() == [4, 10, 9]
    assert strand.tolist() == [0, 0, 0]                                           # strands=None: the queries as given
    for a in (tid, start, end, strand):
        assert a.flags["C_CONTIGUOUS"]
    # a buffer plus offsets, and numpy inputs of other dtypes
    q2, qo2, tid2, start2, end2, strand2 = api.pack_regions(
        q.tobytes(), np.array([0, 2, 1], np.int64), np.array([0, 10, 5], np.int32), [4, 10, 9],
        np.array([1, 0, 1], np.int64), query_offsets=qo)
    assert np.array_equal(q2, q) and np.array_equal(qo2, qo) and tid2.dtype == np.int32 and start2.dtype == np.int64
    assert strand2.tolist() == [1, 0, 1] and strand2.dtype == np.uint8


@pytest.mark.parametrize("bad", [
    dict(tids=[0, 1]),                      # lengths differ from the queries
    dict(starts=[0, 0, 0, 0]),
    dict(ends=[[4], [4], [4]]),             # not 1-d
    dict(strands=[0, 1]),
    dict(tids=[0, 2 ** 31, 0]),             # does not fit int32
    dict(strands=[0, 256, 0]),              # does not fit uint8
    dict(strands=[0, -1, 0]),
    dict(starts=[0.5, 0, 0]),               # not an integer
])
def test_region_inputs_that_do_not_fit_raise_value_error(bad):
    kw = dict(tids=[0, 0, 0], starts=[0, 0, 0], ends=[4, 4, 4], strands=[0, 1, 0])
    kw.update(bad)
    with pytest.raises(ValueError):
        api.pack_regions(["ACGT"] * 3, kw["tids"], kw["starts"], kw["ends"], kw["strands"])
