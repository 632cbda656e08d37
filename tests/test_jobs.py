"""Jobs (fadegpu_submit_pairs / fadegpu_submit_regions / fadegpu_job_wait) without a GPU: the ABI surface (symbols in
the header, in ABI_SYMBOLS and in the D binding, the results view against the header), loud failure without a ctx, a
job or a device, and the Python packing and validation at submit, shared with align_* / score_*."""
import ctypes as C
import os
import re

import pytest

from fade_b200 import _lib, api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
JOB_FNS = ("fadegpu_job_create", "fadegpu_job_destroy", "fadegpu_submit_pairs", "fadegpu_submit_regions",
           "fadegpu_job_wait", "fadegpu_job_results_view")
E_ARG = -1


def test_job_symbols_are_declared_exported_and_bound():
    L = _lib.lib()
    hdr = open(os.path.join(ROOT, "include", "fadegpu.h")).read()
    d = open(os.path.join(ROOT, "integration", "fadegpu.d")).read()
    for fn in JOB_FNS:
        assert re.search(rf"\b(int|void) {fn}\s*\(", hdr) and re.search(rf"\b(int|void) {fn}\s*\(", d), fn
        assert fn in _lib.ABI_SYMBOLS and hasattr(L, fn), fn
    assert "#define FADEGPU_JOB_SCORE_ONLY 1u" in hdr and "FADEGPU_JOB_SCORE_ONLY = 1;" in d
    assert api.JOB_SCORE_ONLY == 1
    assert L.fadegpu_submit_pairs.argtypes[3] == C.POINTER(_lib.PairsIn)
    assert L.fadegpu_submit_regions.argtypes[3] == C.POINTER(_lib.RegionsIn)


def test_results_view_matches_the_header():
    hdr = open(os.path.join(ROOT, "include", "fadegpu.h")).read()
    body = re.search(r"typedef struct fadegpu_job_results \{(.*?)\} fadegpu_job_results;", hdr, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = re.findall(r"(\w+)\s*[;,]", body)
    assert names == [f[0] for f in _lib.JobResults._fields_] == ["n", "records", "ops", "max_ops", "reserved"]
    assert C.sizeof(_lib.JobResults) == 32 and _lib.JobResults.max_ops.offset == 24
    d = open(os.path.join(ROOT, "integration", "fadegpu.d")).read()
    assert "static assert(fadegpu_job_results.sizeof == 32 && fadegpu_job_results.max_ops.offsetof == 24," in d


def test_job_calls_fail_loudly_without_ctx_job_or_device():
    L = _lib.lib()
    out = C.c_void_p()
    assert L.fadegpu_job_create(None, C.byref(out)) == E_ARG and not out.value
    assert b"fadegpu_job_create" in L.fadegpu_last_error(None)
    assert L.fadegpu_submit_pairs(None, None, 1, C.byref(_lib.PairsIn()), 0, 0) == E_ARG
    assert b"fadegpu_submit_pairs" in L.fadegpu_last_error(None)
    assert L.fadegpu_submit_regions(None, None, 1, C.byref(_lib.RegionsIn()), 0, 1) == E_ARG
    assert b"fadegpu_submit_regions" in L.fadegpu_last_error(None)
    assert L.fadegpu_job_wait(None, None, None) == E_ARG
    assert b"fadegpu_job_wait" in L.fadegpu_last_error(None)
    assert L.fadegpu_job_results_view(None, C.byref(_lib.JobResults())) == E_ARG
    L.fadegpu_job_destroy(None)                                                  # a no-op, as fadegpu_destroy(NULL)
    try:
        n = api.device_count()
    except _lib.FadeGpuError:
        n = 0
    if n > 0:
        pytest.skip("a GPU is present: the device side is covered by tests/test_gpu_jobs.py")
    with pytest.raises(_lib.FadeGpuError) as e:
        api.Context(0)
    assert e.value.code in (-5, -2)                                              # no device, no fallback


class _NoLib(Exception):
    pass


def _no_lib_ctx(monkeypatch):
    def no_lib():
        raise _NoLib()
    monkeypatch.setattr(api, "lib", no_lib)
    return object.__new__(api.Context)


@pytest.mark.parametrize("args,kw", [
    ((["ACGT", "AC"], ["ACGT"]), {}),                                                     # 2 queries, 1 target
    ((b"ACGT", b"ACGT"), dict(query_offsets=[0, 8], target_offsets=[0, 4])),              # beyond the buffer
    ((b"ACGT", b"ACGT"), dict(query_offsets=[[0, 4]], target_offsets=[0, 4])),            # not 1-d
])
def test_pair_inputs_raise_at_submit_as_align_pairs_does(args, kw, monkeypatch):
    ctx = _no_lib_ctx(monkeypatch)
    errs = []
    for call in (ctx.align_pairs, ctx.submit_pairs, lambda *a, **k: ctx.submit_pairs(*a, score_only=True, **k)):
        with pytest.raises(ValueError) as e:
            call(*args, **kw)
        errs.append(str(e.value))
    assert errs[0] == errs[1] == errs[2]


@pytest.mark.parametrize("bad", [dict(tids=[0, 1]), dict(strands=[0, 256, 0]), dict(starts=[0.5, 0, 0])])
def test_region_inputs_raise_at_submit_as_align_regions_does(bad, monkeypatch):
    ctx = _no_lib_ctx(monkeypatch)
    kw = dict(tids=[0, 0, 0], starts=[0, 0, 0], ends=[4, 4, 4], strands=[0, 1, 0])
    kw.update(bad)
    errs = []
    for call in (ctx.align_regions, ctx.submit_regions):
        with pytest.raises(ValueError) as e:
            call(["ACGT"] * 3, kw["tids"], kw["starts"], kw["ends"], kw["strands"])
        errs.append(str(e.value))
    assert errs[0] == errs[1]


def test_score_only_jobs_take_no_max_ops(monkeypatch):
    ctx = _no_lib_ctx(monkeypatch)
    with pytest.raises(ValueError, match="max_ops"):
        ctx.submit_pairs(["ACGT"], ["ACGT"], 4, score_only=True)
    with pytest.raises(ValueError, match="max_ops"):
        ctx.submit_regions(["ACGT"], [0], [0], [4], None, 1, score_only=True)


def test_valid_inputs_reach_the_library(monkeypatch):
    """valid inputs pass the packing and arrive at the submit with the ABI layout, the default max_ops and the job
    flags; a refused submit frees its job"""
    seen = {}

    class Fake:
        def fadegpu_job_create(self, h, out):
            out._obj.value = 1234
            return 0

        def fadegpu_job_destroy(self, j):
            seen.setdefault("destroyed", []).append(j.value)

        def fadegpu_submit_pairs(self, h, j, n, pin, max_ops, flags):
            seen["pairs"] = (n, max_ops, flags)
            return E_ARG

        def fadegpu_submit_regions(self, h, j, n, rin, max_ops, flags):
            seen["regions"] = (n, max_ops, flags)
            return E_ARG

        def fadegpu_last_error(self, h):
            return b"refused"
    monkeypatch.setattr(api, "lib", lambda: Fake())
    ctx = object.__new__(api.Context)
    ctx._h = C.c_void_p(1)
    ctx._jobs = set()
    with pytest.raises(_lib.FadeGpuError):
        ctx.submit_pairs(["ACGT", "", "acg"], ["ACGTT", "A", ""])
    assert seen["pairs"] == (3, 12, 0)
    with pytest.raises(_lib.FadeGpuError):
        ctx.submit_regions(b"ACGTAC", [0, 1], [0, 5], [4, 9], [1, 0], query_offsets=[0, 4, 6], score_only=True)
    assert seen["regions"] == (2, 0, api.JOB_SCORE_ONLY)
    assert seen["destroyed"] == [1234, 1234]
    ctx._h = C.c_void_p()
