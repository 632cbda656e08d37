"""Loader of libfadegpu.so -- fails loudly when the CUDA extension is missing."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libfadegpu.so")
_lib = None


class FadeGpuError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"fadegpu error {code}: {msg}")
        self.code = code


def lib_path() -> str:
    return _SO


def build(force: bool = False) -> str:
    """Compile libfadegpu.so (and the CPU-test emulation) for sm_100a with nvcc, in-tree."""
    args = ["make", "-C", os.path.join(_HERE, "csrc"), "-s"]
    if force:
        args.append("-B")
    subprocess.check_call(args)
    return _SO


class Params(C.Structure):
    _fields_ = [("window_size", C.c_int32), ("min_length", C.c_int32), ("gap_open", C.c_int32),
                ("gap_extend", C.c_int32), ("match", C.c_int32), ("mismatch", C.c_int32),
                ("flags", C.c_uint32), ("scratch_bytes", C.c_int64), ("host_threads", C.c_int32),
                ("reserved", C.c_int32)]


class BatchView(C.Structure):
    _fields_ = [("max_reads", C.c_int64), ("max_seq_bytes", C.c_int64),
                ("seq4", C.POINTER(C.c_uint8)), ("seq_off", C.POINTER(C.c_int64)),
                ("l_qseq", C.POINTER(C.c_int32)), ("tid", C.POINTER(C.c_int32)), ("pos", C.POINTER(C.c_int64)),
                ("aligned_len", C.POINTER(C.c_int32)), ("clip_left", C.POINTER(C.c_int32)),
                ("clip_right", C.POINTER(C.c_int32)),
                ("flags", C.POINTER(C.c_uint8)), ("score", C.POINTER(C.c_int32)),
                ("beg_query", C.POINTER(C.c_int32)), ("end_query", C.POINTER(C.c_int32)),
                ("beg_ref", C.POINTER(C.c_int32)), ("end_ref", C.POINTER(C.c_int32)),
                ("win_start", C.POINTER(C.c_int64)), ("n_ops", C.POINTER(C.c_int32)),
                ("ops", C.POINTER(C.c_uint32)),
                ("gate", C.POINTER(C.c_uint8)), ("meta", C.c_void_p)]


class Inputs(C.Structure):
    _fields_ = [("seq4", C.c_void_p), ("seq_off", C.c_void_p), ("l_qseq", C.c_void_p), ("tid", C.c_void_p),
                ("pos", C.c_void_p), ("aligned_len", C.c_void_p), ("clip_left", C.c_void_p),
                ("clip_right", C.c_void_p)]


class Result(C.Structure):
    _fields_ = [("score", C.c_int32), ("end_query", C.c_int32), ("end_ref", C.c_int32), ("beg_query", C.c_int32),
                ("beg_ref", C.c_int32), ("n_ops", C.c_int32), ("flags", C.c_uint32), ("read", C.c_int32),
                ("ops", C.c_uint32 * 10)]   # FADEGPU_MAX_OPS


class ResultsView(C.Structure):
    _fields_ = [("n_results", C.c_int64), ("results", C.POINTER(Result)), ("win_start", C.POINTER(C.c_int64)),
                ("result_index", C.POINTER(C.c_int32))]


class Stats(C.Structure):
    _fields_ = [("n_reads", C.c_int64), ("n_aligned", C.c_int64), ("n_generic", C.c_int64), ("cells", C.c_int64),
                ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64), ("kernel_launches", C.c_int32),
                ("kernel_ms", C.c_float), ("fill_ms", C.c_float), ("trace_ms", C.c_float),
                ("generic_ms", C.c_float), ("total_ms", C.c_float), ("scratch_bytes", C.c_int64),
                ("host_submit_ms", C.c_float), ("host_wait_ms", C.c_float), ("host_classify_ms", C.c_float),
                ("host_sort_ms", C.c_float), ("host_gather_ms", C.c_float), ("host_threads", C.c_int32),
                ("reserved", C.c_int32), ("n_oversize", C.c_int64)]


class PairsIn(C.Structure):
    """fadegpu_pairs: host arrays of one fadegpu_align_pairs / fadegpu_score_pairs call"""
    _fields_ = [("query", C.c_void_p), ("query_off", C.c_void_p), ("target", C.c_void_p), ("target_off", C.c_void_p)]


class RegionsIn(C.Structure):
    """fadegpu_regions: host arrays of one fadegpu_align_regions / fadegpu_score_regions call"""
    _fields_ = [("query", C.c_void_p), ("query_off", C.c_void_p), ("tid", C.c_void_p), ("start", C.c_void_p),
                ("end", C.c_void_p), ("strand", C.c_void_p)]


class PairResult(C.Structure):
    _fields_ = [("score", C.c_int32), ("end_query", C.c_int32), ("end_ref", C.c_int32), ("beg_query", C.c_int32),
                ("beg_ref", C.c_int32), ("n_ops", C.c_int32), ("flags", C.c_uint32), ("reserved", C.c_int32)]


class JobResults(C.Structure):
    """fadegpu_job_results: the records and ops of a waited job, in pinned memory the job owns"""
    _fields_ = [("n", C.c_int64), ("records", C.c_void_p), ("ops", C.c_void_p), ("max_ops", C.c_int32),
                ("reserved", C.c_int32)]


class HostRecord(C.Structure):
    _fields_ = [("flag", C.c_int32), ("has_sa", C.c_int32), ("cigar", C.POINTER(C.c_uint32)),
                ("n_cigar", C.c_int32), ("seq4", C.POINTER(C.c_uint8)), ("qual", C.POINTER(C.c_uint8)),
                ("l_qseq", C.c_int32), ("tid", C.c_int32), ("pos", C.c_int64)]


# every symbol include/fadegpu.h and include/fadehost.h declare
ABI_SYMBOLS = [
    "fadegpu_abi_version", "fadegpu_device_count", "fadegpu_default_params", "fadegpu_create",
    "fadegpu_destroy", "fadegpu_last_error", "fadegpu_load_reference", "fadegpu_share_reference",
    "fadegpu_reference_info", "fadegpu_alloc_batch", "fadegpu_get_batch_view", "fadegpu_free_batch",
    "fadegpu_submit", "fadegpu_submit_compact", "fadegpu_submit_inputs", "fadegpu_wait", "fadegpu_get_results", "fadegpu_get_stats", "fadegpu_get_timeline", "fadegpu_replay_kernels", "fadegpu_replay_batches",
    "fadegpu_align_pairs", "fadegpu_align_regions", "fadegpu_score_pairs", "fadegpu_score_regions",
    "fadegpu_job_create", "fadegpu_job_destroy", "fadegpu_submit_pairs", "fadegpu_submit_regions", "fadegpu_job_wait",
    "fadegpu_job_results_view",
    "fadegpu_measure_alu_peak",
    "fadehost_parse_clips", "fadehost_aligned_length", "fadehost_prepare", "fadehost_finish",
]


def lib():
    """The loaded C ABI.  Raises if libfadegpu.so has not been built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_SO):
        raise FadeGpuError(-100, f"{_SO} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                                 "(nvcc, sm_100a); fade_b200 has no CPU fallback")
    L = C.CDLL(_SO)
    vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    L.fadegpu_abi_version.restype = C.c_int
    L.fadegpu_device_count.argtypes = [C.POINTER(C.c_int)]
    L.fadegpu_default_params.argtypes = [C.POINTER(Params)]
    L.fadegpu_create.argtypes = [C.c_int, C.POINTER(Params), C.POINTER(vp)]
    L.fadegpu_destroy.argtypes = [vp]
    L.fadegpu_destroy.restype = None
    L.fadegpu_last_error.argtypes = [vp]
    L.fadegpu_last_error.restype = C.c_char_p
    L.fadegpu_load_reference.argtypes = [vp, i32, C.POINTER(C.c_char_p), C.POINTER(i64), C.POINTER(C.c_char_p)]
    L.fadegpu_share_reference.argtypes = [vp, vp]
    L.fadegpu_reference_info.argtypes = [vp, C.POINTER(i32), C.POINTER(i64), C.POINTER(i64)]
    L.fadegpu_alloc_batch.argtypes = [vp, i64, i64, C.POINTER(vp)]
    L.fadegpu_get_batch_view.argtypes = [vp, C.POINTER(BatchView)]
    L.fadegpu_free_batch.argtypes = [vp]
    L.fadegpu_free_batch.restype = None
    L.fadegpu_submit.argtypes = [vp, vp, i64]
    L.fadegpu_submit_compact.argtypes = [vp, vp, i64, i64]
    L.fadegpu_submit_inputs.argtypes = [vp, vp, i64, C.POINTER(Inputs)]
    L.fadegpu_wait.argtypes = [vp, vp]
    L.fadegpu_get_results.argtypes = [vp, C.POINTER(ResultsView)]
    L.fadegpu_get_stats.argtypes = [vp, C.POINTER(Stats)]
    L.fadegpu_get_timeline.argtypes = [vp, vp, C.POINTER(C.c_float)]
    L.fadegpu_replay_kernels.argtypes = [vp, vp, i32, C.POINTER(C.c_float)]
    L.fadegpu_replay_batches.argtypes = [vp, C.POINTER(vp), i32, i32, C.POINTER(C.c_float)]
    L.fadegpu_align_pairs.argtypes = [vp, i64, C.POINTER(PairsIn), i32, vp, vp, C.POINTER(Stats)]
    L.fadegpu_align_regions.argtypes = [vp, i64, C.POINTER(RegionsIn), i32, vp, vp, C.POINTER(Stats)]
    L.fadegpu_score_pairs.argtypes = [vp, i64, C.POINTER(PairsIn), vp, C.POINTER(Stats)]
    L.fadegpu_score_regions.argtypes = [vp, i64, C.POINTER(RegionsIn), vp, C.POINTER(Stats)]
    L.fadegpu_job_create.argtypes = [vp, C.POINTER(vp)]
    L.fadegpu_job_destroy.argtypes = [vp]
    L.fadegpu_job_destroy.restype = None
    L.fadegpu_submit_pairs.argtypes = [vp, vp, i64, C.POINTER(PairsIn), i32, C.c_uint32]
    L.fadegpu_submit_regions.argtypes = [vp, vp, i64, C.POINTER(RegionsIn), i32, C.c_uint32]
    L.fadegpu_job_wait.argtypes = [vp, vp, C.POINTER(Stats)]
    L.fadegpu_job_results_view.argtypes = [vp, C.POINTER(JobResults)]
    L.fadegpu_measure_alu_peak.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    L.fadehost_parse_clips.argtypes = [C.POINTER(C.c_uint32), i32, C.POINTER(C.c_uint32)]
    L.fadehost_parse_clips.restype = None
    L.fadehost_aligned_length.argtypes = [C.POINTER(C.c_uint32), i32]
    L.fadehost_aligned_length.restype = i64
    L.fadehost_prepare.argtypes = [C.POINTER(HostRecord), C.POINTER(i32), C.POINTER(i32), C.POINTER(i32),
                                   C.POINTER(C.c_uint8)]
    L.fadehost_finish.argtypes = [C.POINTER(HostRecord), C.c_char_p, C.c_uint8, i32, i32, i32, C.c_uint8, i64, i32,
                                  i32, C.POINTER(C.c_uint32), C.POINTER(C.c_uint8), C.c_char_p, C.c_char_p,
                                  C.c_char_p, C.c_char_p, C.c_size_t]
    if L.fadegpu_abi_version() != 2:
        raise FadeGpuError(-101, "libfadegpu.so ABI version mismatch")
    _lib = L
    return L
