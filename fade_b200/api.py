"""Python host layer over the C ABI: Context / Batch wrappers and an `annotate_records` loop that
mirrors source/anno.d:44-50 + annotateTask (source/anno.d:55-110) in batched form."""
from __future__ import annotations

import ctypes as C
import weakref
from dataclasses import dataclass, field

import numpy as np

from ._lib import (BatchView, FadeGpuError, HostRecord, Inputs, JobResults, PairResult, PairsIn, Params, RegionsIn,
                   Result, ResultsView, Stats, lib)

MAX_OPS = 10
R_ALIGNED, R_ART_LEFT, R_ART_RIGHT, R_OPS_TRUNC, R_GENERIC, R_OVERSIZE, R_SCORE_ONLY = 1, 2, 4, 8, 16, 32, 64
F_FORCE_GENERIC = 1
F_NO_SCATTER = 2
F_TAGS_ONLY = 4
F_NO_SHORTCUT = 8
F_HOST_BINNING = 16
F_SYNC_SUBMIT = 32
JOB_SCORE_ONLY = 1
RESULT_DTYPE = np.dtype([("score", "<i4"), ("end_query", "<i4"), ("end_ref", "<i4"), ("beg_query", "<i4"),
                         ("beg_ref", "<i4"), ("n_ops", "<i4"), ("flags", "<u4"), ("read", "<i4"),
                         ("ops", "<u4", (MAX_OPS,))])
# fadegpu_read_meta: one read of the compact input layout (fadegpu_submit_compact)
META_DTYPE = np.dtype([("pos", "<i8"), ("seq_off", "<u4"), ("l_qseq", "<i4"), ("tid", "<i4"), ("aligned_len", "<i4"),
                       ("clip_left", "<u4"), ("clip_right", "<u4")])
assert META_DTYPE.itemsize == 32
OPCHARS = "MIDNSHP=XB"
# fadegpu_pair_result: one record of Context.align_pairs, in pair order
PAIR_RESULT_DTYPE = np.dtype([("score", "<i4"), ("end_query", "<i4"), ("end_ref", "<i4"), ("beg_query", "<i4"),
                              ("beg_ref", "<i4"), ("n_ops", "<i4"), ("flags", "<u4"), ("reserved", "<i4")])
assert PAIR_RESULT_DTYPE.itemsize == 32


def _pack_side(seqs, offsets=None):
    """One side of a pair call as (uint8 buffer, int64 offsets[n+1]): a list of str / bytes, or one bytes / uint8 buffer
    plus its offsets."""
    if offsets is not None:
        buf = np.frombuffer(seqs, dtype=np.uint8) if isinstance(seqs, (bytes, bytearray)) else np.asarray(seqs)
        if buf.dtype != np.uint8 or buf.ndim != 1:
            raise TypeError("a sequence buffer must be bytes or a 1-d uint8 array")
        off = np.ascontiguousarray(offsets, dtype=np.int64)
        if off.ndim != 1 or len(off) < 1:
            raise ValueError("offsets must be a 1-d array of n+1 entries")
        if len(off) > 1 and (off[0] < 0 or off[-1] > len(buf)):
            raise ValueError("offsets exceed the sequence buffer")
        return np.ascontiguousarray(buf), off
    parts = [s.encode() if isinstance(s, str) else bytes(s) for s in seqs]
    off = np.zeros(len(parts) + 1, dtype=np.int64)
    if parts:
        np.cumsum([len(p) for p in parts], out=off[1:])
    return np.frombuffer(b"".join(parts), dtype=np.uint8).copy(), off


def pack_pairs(queries, targets, query_offsets=None, target_offsets=None):
    """(query buffer, query offsets, target buffer, target offsets) as fadegpu_align_pairs reads them"""
    q, qo = _pack_side(queries, query_offsets)
    t, to = _pack_side(targets, target_offsets)
    if len(qo) != len(to):
        raise ValueError(f"{len(qo) - 1} queries but {len(to) - 1} targets")
    return q, qo, t, to


def _region_array(x, dtype, n, name):
    """one per-region array of Context.align_regions in its ABI dtype: n entries whose values survive the conversion"""
    a = np.asarray(x)
    if a.ndim != 1 or len(a) != n:
        raise ValueError(f"{name} must be a 1-d array of {n} entries (one per query), not of shape {a.shape}")
    out = np.ascontiguousarray(a, dtype=dtype)
    if n and not np.array_equal(out, a):
        raise ValueError(f"{name} holds values outside {np.dtype(dtype).name}")
    return out


def pack_regions(queries, tids, starts, ends, strands=None, query_offsets=None):
    """(query buffer, query offsets, tid int32, start int64, end int64, strand uint8) as fadegpu_align_regions reads
    them; strands None means all 0 (the queries as given)"""
    q, qo = _pack_side(queries, query_offsets)
    n = len(qo) - 1
    strands = np.zeros(n, np.uint8) if strands is None else strands
    return (q, qo, _region_array(tids, np.int32, n, "tids"), _region_array(starts, np.int64, n, "starts"),
            _region_array(ends, np.int64, n, "ends"), _region_array(strands, np.uint8, n, "strands"))


def default_max_ops(query_offsets) -> int:
    """3 * the longest query: no CIGAR of a local alignment can be longer (see fadegpu_align_pairs in fadegpu.h)"""
    qo = np.asarray(query_offsets, dtype=np.int64)
    return int(3 * np.diff(qo).max()) if len(qo) > 1 else 0


@dataclass
class PairResults:
    """Context.align_pairs / align_regions: records[n] (PAIR_RESULT_DTYPE) and ops[n, max_ops] in pair / region order,
    and the call's stats."""
    records: np.ndarray
    ops: np.ndarray
    stats: Stats

    def __len__(self):
        return len(self.records)

    def cigar(self, k: int) -> str:
        """forward CIGAR of pair k (its first max_ops ops when the record has R_OPS_TRUNC)"""
        n = min(int(self.records["n_ops"][k]), self.ops.shape[1])
        return "".join(f"{int(o) >> 4}{OPCHARS[int(o) & 0xf]}" for o in self.ops[k, :n])


@dataclass
class ScoreResults:
    """Context.score_pairs / score_regions: records[n] (PAIR_RESULT_DTYPE) in pair / region order -- score, end_query,
    end_ref and flags; beg_query, beg_ref and n_ops are 0, there is no CIGAR -- and the call's stats."""
    records: np.ndarray
    stats: Stats

    def __len__(self):
        return len(self.records)


def default_params(**kw) -> Params:
    p = Params()
    rc = lib().fadegpu_default_params(C.byref(p))
    if rc:
        raise FadeGpuError(rc, "fadegpu_default_params")
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def device_count() -> int:
    n = C.c_int(0)
    rc = lib().fadegpu_device_count(C.byref(n))
    if rc:
        raise FadeGpuError(rc, lib().fadegpu_last_error(None).decode())
    return n.value


def _np_view(ptr, n, dtype):
    if n == 0:
        return np.zeros(0, dtype=dtype)
    addr = C.cast(ptr, C.c_void_p).value
    buf = (C.c_char * (n * np.dtype(dtype).itemsize)).from_address(addr)
    return np.frombuffer(buf, dtype=dtype, count=n)


class Context:
    """One per (host thread, GPU): scoring profile + device-resident packed reference.
    Replaces Parasail("ACTGN",10,2,2,-3) (anno.d:36) and IndexedFastaFile (anno.d:23)."""

    def __init__(self, device: int = 0, params: Params | None = None):
        self._h = C.c_void_p()
        self.params = params or default_params()
        rc = lib().fadegpu_create(device, C.byref(self.params), C.byref(self._h))
        if rc:
            raise FadeGpuError(rc, lib().fadegpu_last_error(None).decode())
        self.device = device
        self.contig_names: list[str] = []
        self._batches = weakref.WeakSet()      # freed before the ctx: a batch must not outlive it
        self._jobs = weakref.WeakSet()         # the same for jobs

    def _check(self, rc: int):
        if rc:
            raise FadeGpuError(rc, lib().fadegpu_last_error(self._h).decode())

    def load_reference(self, names: list[str], seqs: list):
        """seqs: ASCII contigs as bytes or as C-contiguous uint8 numpy arrays (passed without a copy)."""
        n = len(seqs)
        cn = (C.c_char_p * n)(*[s.encode() for s in names])
        cs = (C.c_char_p * n)()
        for k, s in enumerate(seqs):
            if isinstance(s, np.ndarray):
                assert s.dtype == np.uint8 and s.flags["C_CONTIGUOUS"]
                C.cast(cs, C.POINTER(C.c_void_p))[k] = s.ctypes.data
            else:
                cs[k] = s
        ln = (C.c_int64 * n)(*[len(s) for s in seqs])
        self._check(lib().fadegpu_load_reference(self._h, n, cn, ln, cs))
        self.contig_names = list(names)

    def share_reference_from(self, other: "Context"):
        self._check(lib().fadegpu_share_reference(self._h, other._h))
        self.contig_names = list(other.contig_names)

    def reference_info(self):
        a, b, c = C.c_int32(), C.c_int64(), C.c_int64()
        self._check(lib().fadegpu_reference_info(self._h, C.byref(a), C.byref(b), C.byref(c)))
        return a.value, b.value, c.value

    def measure_alu_peak(self):
        ops, mhz = C.c_double(), C.c_double()
        self._check(lib().fadegpu_measure_alu_peak(self._h, C.byref(ops), C.byref(mhz)))
        return ops.value, mhz.value

    def replay_batches(self, batches, iters: int = 1) -> float:
        """fadegpu_replay_batches: device ms of `iters` passes of only the kernels over resident batches,
        queued back to back as consecutive submits queue them."""
        arr = (C.c_void_p * len(batches))(*[b._h.value for b in batches])
        ms = C.c_float()
        self._check(lib().fadegpu_replay_batches(self._h, arr, len(batches), iters, C.byref(ms)))
        return ms.value

    def align_pairs(self, queries, targets, max_ops: int | None = None, *, query_offsets=None,
                    target_offsets=None) -> PairResults:
        """fadegpu_align_pairs: Smith-Waterman with traceback of query k against target k, with the ctx's scoring.

        queries / targets: lists of str or bytes, or one bytes / uint8 buffer each with query_offsets /
        target_offsets (n+1 int64 entries).  Queries are taken as given (no reverse complement) and must use the
        nt16 letters =ACMGRSVTWYHKDBN; targets may hold any letter.  max_ops defaults to 3 * the longest query,
        which never truncates a CIGAR."""
        q, qo, t, to = pack_pairs(queries, targets, query_offsets, target_offsets)
        n = len(qo) - 1
        if max_ops is None:
            max_ops = default_max_ops(qo)
        rec = np.zeros(n, dtype=PAIR_RESULT_DTYPE)
        ops = np.zeros((n, max_ops), dtype=np.uint32)
        st = Stats()
        pin = PairsIn(q.ctypes.data, qo.ctypes.data, t.ctypes.data, to.ctypes.data)
        self._check(lib().fadegpu_align_pairs(self._h, n, C.byref(pin), max_ops, rec.ctypes.data,
                                              ops.ctypes.data if max_ops > 0 else None, C.byref(st)))
        return PairResults(rec, ops, st)

    def align_regions(self, queries, tids, starts, ends, strands=None, max_ops: int | None = None, *,
                      query_offsets=None) -> PairResults:
        """fadegpu_align_regions: Smith-Waterman with traceback of query k against [starts[k], ends[k]) of the loaded
        contig tids[k], with the ctx's scoring.

        queries: as in align_pairs (nt16 letters).  strands[k] = 1 aligns the reverse complement of query k (its
        beg_query / end_query then index the reverse complement); None means all 0.  beg_ref / end_ref are relative to
        starts[k].  max_ops defaults to 3 * the longest query, which never truncates a CIGAR."""
        q, qo, tid, start, end, strand = pack_regions(queries, tids, starts, ends, strands, query_offsets)
        n = len(qo) - 1
        if max_ops is None:
            max_ops = default_max_ops(qo)
        rec = np.zeros(n, dtype=PAIR_RESULT_DTYPE)
        ops = np.zeros((n, max_ops), dtype=np.uint32)
        st = Stats()
        rin = RegionsIn(q.ctypes.data, qo.ctypes.data, tid.ctypes.data, start.ctypes.data, end.ctypes.data,
                        strand.ctypes.data)
        self._check(lib().fadegpu_align_regions(self._h, n, C.byref(rin), max_ops, rec.ctypes.data,
                                                ops.ctypes.data if max_ops > 0 else None, C.byref(st)))
        return PairResults(rec, ops, st)

    def score_pairs(self, queries, targets, *, query_offsets=None, target_offsets=None) -> ScoreResults:
        """fadegpu_score_pairs: score and end cell of query k against target k, without traceback.  Inputs as in
        align_pairs; score, end_query and end_ref equal align_pairs' on the same inputs."""
        q, qo, t, to = pack_pairs(queries, targets, query_offsets, target_offsets)
        n = len(qo) - 1
        rec = np.zeros(n, dtype=PAIR_RESULT_DTYPE)
        st = Stats()
        pin = PairsIn(q.ctypes.data, qo.ctypes.data, t.ctypes.data, to.ctypes.data)
        self._check(lib().fadegpu_score_pairs(self._h, n, C.byref(pin), rec.ctypes.data, C.byref(st)))
        return ScoreResults(rec, st)

    def score_regions(self, queries, tids, starts, ends, strands=None, *, query_offsets=None) -> ScoreResults:
        """fadegpu_score_regions: score and end cell of query k against [starts[k], ends[k]) of contig tids[k], without
        traceback.  Inputs as in align_regions; score, end_query and end_ref equal align_regions' on the same inputs."""
        q, qo, tid, start, end, strand = pack_regions(queries, tids, starts, ends, strands, query_offsets)
        n = len(qo) - 1
        rec = np.zeros(n, dtype=PAIR_RESULT_DTYPE)
        st = Stats()
        rin = RegionsIn(q.ctypes.data, qo.ctypes.data, tid.ctypes.data, start.ctypes.data, end.ctypes.data,
                        strand.ctypes.data)
        self._check(lib().fadegpu_score_regions(self._h, n, C.byref(rin), rec.ctypes.data, C.byref(st)))
        return ScoreResults(rec, st)

    def submit_pairs(self, queries, targets, max_ops: int | None = None, *, score_only: bool = False,
                     query_offsets=None, target_offsets=None) -> "Job":
        """fadegpu_submit_pairs on a new job: align_pairs (score_pairs with score_only=True) that returns once the
        inputs are copied; the kernels run while the caller goes on, and Job.wait() gives the call's results"""
        return self._new_job(_pairs_job(queries, targets, max_ops, score_only, query_offsets, target_offsets))

    def submit_regions(self, queries, tids, starts, ends, strands=None, max_ops: int | None = None, *,
                       score_only: bool = False, query_offsets=None) -> "Job":
        """fadegpu_submit_regions on a new job: align_regions (score_regions with score_only=True); see submit_pairs"""
        return self._new_job(_regions_job(queries, tids, starts, ends, strands, max_ops, score_only, query_offsets))

    def _new_job(self, call) -> "Job":
        job = Job(self)
        try:
            return job._submit(call)
        except BaseException:
            job.close()
            raise

    def alloc_batch(self, max_reads: int, max_seq_bytes: int) -> "Batch":
        return Batch(self, max_reads, max_seq_bytes)

    def close(self):
        if self._h:
            for b in list(self._batches):
                b.close()
            for j in list(self._jobs):
                j.close()
            lib().fadegpu_destroy(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _job_max_ops(qo, max_ops, score_only: bool) -> int:
    if score_only:
        if max_ops:
            raise ValueError("a score-only job has no CIGAR: max_ops must be 0 or None")
        return 0
    return default_max_ops(qo) if max_ops is None else max_ops


def _pairs_job(queries, targets, max_ops, score_only, query_offsets, target_offsets):
    """the packed and validated arguments of fadegpu_submit_pairs (and the arrays they point into)"""
    q, qo, t, to = pack_pairs(queries, targets, query_offsets, target_offsets)
    max_ops = _job_max_ops(qo, max_ops, score_only)
    pin = PairsIn(q.ctypes.data, qo.ctypes.data, t.ctypes.data, to.ctypes.data)
    return "fadegpu_submit_pairs", len(qo) - 1, pin, max_ops, score_only, (q, qo, t, to)


def _regions_job(queries, tids, starts, ends, strands, max_ops, score_only, query_offsets):
    q, qo, tid, start, end, strand = pack_regions(queries, tids, starts, ends, strands, query_offsets)
    max_ops = _job_max_ops(qo, max_ops, score_only)
    rin = RegionsIn(q.ctypes.data, qo.ctypes.data, tid.ctypes.data, start.ctypes.data, end.ctypes.data,
                    strand.ctypes.data)
    return "fadegpu_submit_regions", len(qo) - 1, rin, max_ops, score_only, (q, qo, tid, start, end, strand)


class Job:
    """One pair or region call in flight (Context.submit_pairs / submit_regions).  wait() gives what the synchronous
    call would have returned: PairResults, or ScoreResults for a score-only job.  A job can be closed before it is
    waited for (close waits for it); the ctx closes its jobs when it is closed."""

    def __init__(self, ctx: Context):
        self.ctx = ctx
        self._h = C.c_void_p()
        ctx._check(lib().fadegpu_job_create(ctx._h, C.byref(self._h)))
        ctx._jobs.add(self)
        self.score_only = False

    def submit_pairs(self, queries, targets, max_ops: int | None = None, *, score_only: bool = False,
                     query_offsets=None, target_offsets=None) -> "Job":
        """fadegpu_submit_pairs: inputs and max_ops as in Context.align_pairs (max_ops defaults to 3 * the longest
        query, and must be 0 or None with score_only).  A job is reused once waited for: its buffers grow with use."""
        return self._submit(_pairs_job(queries, targets, max_ops, score_only, query_offsets, target_offsets))

    def submit_regions(self, queries, tids, starts, ends, strands=None, max_ops: int | None = None, *,
                       score_only: bool = False, query_offsets=None) -> "Job":
        """fadegpu_submit_regions: inputs and max_ops as in Context.align_regions; see submit_pairs"""
        return self._submit(_regions_job(queries, tids, starts, ends, strands, max_ops, score_only, query_offsets))

    def _submit(self, call) -> "Job":
        fn, n, inp, max_ops, score_only, _arrays = call     # (the arrays are read during the call only)
        self.ctx._check(getattr(lib(), fn)(self.ctx._h, self._h, n, C.byref(inp), max_ops,
                                           JOB_SCORE_ONLY if score_only else 0))
        self.score_only = score_only
        return self

    def wait(self):
        st = Stats()
        self.ctx._check(lib().fadegpu_job_wait(self.ctx._h, self._h, C.byref(st)))
        v = JobResults()
        self.ctx._check(lib().fadegpu_job_results_view(self._h, C.byref(v)))
        n, m = int(v.n), int(v.max_ops)
        rec = _np_view(C.cast(v.records, C.POINTER(C.c_uint8)), n * PAIR_RESULT_DTYPE.itemsize, np.uint8)
        rec = rec.view(PAIR_RESULT_DTYPE).copy()
        if self.score_only:
            return ScoreResults(rec, st)
        ops = _np_view(C.cast(v.ops, C.POINTER(C.c_uint32)), n * m, np.uint32).reshape(n, m).copy()
        return PairResults(rec, ops, st)

    def close(self):
        if self._h:
            lib().fadegpu_job_destroy(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Batch:
    """Pinned struct-of-arrays buffers (numpy views) + device mirrors, owned by the library."""

    def __init__(self, ctx: Context, max_reads: int, max_seq_bytes: int):
        self.ctx = ctx
        self._h = C.c_void_p()
        ctx._check(lib().fadegpu_alloc_batch(ctx._h, max_reads, max_seq_bytes, C.byref(self._h)))
        ctx._batches.add(self)
        v = BatchView()
        ctx._check(lib().fadegpu_get_batch_view(self._h, C.byref(v)))
        self.max_reads, self.max_seq_bytes = max_reads, max_seq_bytes
        n = max_reads
        self.seq4 = _np_view(v.seq4, max_seq_bytes, np.uint8)
        self.seq_off = _np_view(v.seq_off, n + 1, np.int64)
        self.l_qseq = _np_view(v.l_qseq, n, np.int32)
        self.tid = _np_view(v.tid, n, np.int32)
        self.pos = _np_view(v.pos, n, np.int64)
        self.aligned_len = _np_view(v.aligned_len, n, np.int32)
        self.clip_left = _np_view(v.clip_left, n, np.int32)
        self.clip_right = _np_view(v.clip_right, n, np.int32)
        self.flags = _np_view(v.flags, n, np.uint8)
        self.gate = _np_view(v.gate, n, np.uint8)
        self.meta = _np_view(C.cast(v.meta, C.POINTER(C.c_uint8)), n * META_DTYPE.itemsize, np.uint8).view(META_DTYPE)
        self.seq_bytes = 0
        if v.score:     # per-read output arrays exist unless the ctx has F_NO_SCATTER
            self.score = _np_view(v.score, n, np.int32)
            self.beg_query = _np_view(v.beg_query, n, np.int32)
            self.end_query = _np_view(v.end_query, n, np.int32)
            self.beg_ref = _np_view(v.beg_ref, n, np.int32)
            self.end_ref = _np_view(v.end_ref, n, np.int32)
            self.win_start = _np_view(v.win_start, n, np.int64)
            self.n_ops = _np_view(v.n_ops, n, np.int32)
            self.ops = _np_view(v.ops, n * MAX_OPS, np.uint32).reshape(n, MAX_OPS)
        else:
            self.score = self.beg_query = self.end_query = self.beg_ref = self.end_ref = None
            self.win_start = self.n_ops = self.ops = None
        self.n = 0

    def fill(self, seq4, seq_off, l_qseq, tid, pos, aligned_len, clip_left, clip_right):
        n = len(l_qseq)
        if n > self.max_reads or int(seq_off[n]) > self.max_seq_bytes:
            raise ValueError("batch too small")
        self.seq4[:int(seq_off[n])] = seq4[:int(seq_off[n])]
        self.seq_off[:n + 1] = seq_off[:n + 1]
        self.l_qseq[:n] = l_qseq
        self.tid[:n] = tid
        self.pos[:n] = pos
        self.aligned_len[:n] = aligned_len
        self.clip_left[:n] = clip_left
        self.clip_right[:n] = clip_right
        self.n = n
        return self

    def fill_compact(self, seq4, seq_off, l_qseq, tid, pos, aligned_len, clip_left, clip_right):
        """the same reads in the compact layout: gate[] (one byte per read) + meta[] (32-byte records) + seq4"""
        n = len(l_qseq)
        nb = int(seq_off[n])
        if n > self.max_reads or nb > self.max_seq_bytes:
            raise ValueError("batch too small")
        self.seq4[:nb] = seq4[:nb]
        m = self.meta[:n]
        m["pos"] = pos
        m["seq_off"] = seq_off[:n]
        m["l_qseq"] = l_qseq
        m["tid"] = tid
        m["aligned_len"] = aligned_len
        m["clip_left"] = np.asarray(clip_left).astype(np.uint32)
        m["clip_right"] = np.asarray(clip_right).astype(np.uint32)
        np.minimum(np.maximum(m["clip_left"], m["clip_right"]), 255, out=self.gate[:n], casting="unsafe")
        self.n = n
        self.seq_bytes = nb
        return self

    def submit_compact(self, n: int | None = None, seq_bytes: int | None = None):
        if n is not None:
            self.n = n
        if seq_bytes is not None:
            self.seq_bytes = seq_bytes
        self.ctx._check(lib().fadegpu_submit_compact(self.ctx._h, self._h, self.n, self.seq_bytes))

    def submit(self, n: int | None = None):
        if n is not None:
            self.n = n
        self.ctx._check(lib().fadegpu_submit(self.ctx._h, self._h, self.n))

    def submit_arrays(self, n, seq4, seq_off, l_qseq, tid, pos, aligned_len, clip_left, clip_right):
        """fadegpu_submit_inputs: read the inputs straight from caller-owned (pageable) numpy arrays.
        seq_off may hold absolute offsets into seq4; arrays must be C-contiguous with the ABI dtypes."""
        def ptr(a, dt):
            assert a.dtype == dt and a.flags["C_CONTIGUOUS"], (a.dtype, dt)
            return a.ctypes.data
        inp = Inputs(ptr(seq4, np.uint8), ptr(seq_off, np.int64), ptr(l_qseq, np.int32), ptr(tid, np.int32),
                     ptr(pos, np.int64), ptr(aligned_len, np.int32), ptr(clip_left, np.int32),
                     ptr(clip_right, np.int32))
        self.n = n
        self.ctx._check(lib().fadegpu_submit_inputs(self.ctx._h, self._h, n, C.byref(inp)))

    def wait(self):
        self.ctx._check(lib().fadegpu_wait(self.ctx._h, self._h))

    def run(self, n: int | None = None):
        self.submit(n)
        self.wait()
        return self

    def results(self):
        """fadegpu_get_results: (records[n_results] structured array, win_start[n_results], result_index[n])
        as zero-copy numpy views valid until the next submit."""
        rv = ResultsView()
        self.ctx._check(lib().fadegpu_get_results(self._h, C.byref(rv)))
        k = int(rv.n_results)
        assert RESULT_DTYPE.itemsize == C.sizeof(Result)
        if k == 0:
            rec = np.zeros(0, dtype=RESULT_DTYPE)
            ws = np.zeros(0, dtype=np.int64)
        else:
            addr = C.cast(rv.results, C.c_void_p).value
            rec = np.frombuffer((C.c_char * (k * RESULT_DTYPE.itemsize)).from_address(addr), dtype=RESULT_DTYPE, count=k)
            ws = _np_view(rv.win_start, k, np.int64)
        return rec, ws, _np_view(rv.result_index, self.n, np.int32)

    def stats(self) -> Stats:
        s = Stats()
        self.ctx._check(lib().fadegpu_get_stats(self._h, C.byref(s)))
        return s

    def timeline(self, origin: "Batch"):
        """device ms of (uploads start, first fill starts, kernels done, results home, inputs ready, last fill done) relative to origin's start"""
        ms = (C.c_float * 6)()
        self.ctx._check(lib().fadegpu_get_timeline(self._h, origin._h, ms))
        return [float(x) for x in ms]

    def replay_kernels(self, iters: int = 1) -> float:
        ms = C.c_float()
        self.ctx._check(lib().fadegpu_replay_kernels(self.ctx._h, self._h, iters, C.byref(ms)))
        return ms.value

    def cigar(self, r: int) -> str:
        k = min(int(self.n_ops[r]), MAX_OPS)
        return "".join(f"{int(o) >> 4}{OPCHARS[int(o) & 0xf]}" for o in self.ops[r, :k])

    def close(self):
        if self._h:
            lib().fadegpu_free_batch(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


@dataclass
class Record:
    """The fields of a SAM/BAM record that annotateTask reads (dhtslib SAMRecord subset)."""
    qname: str
    flag: int
    tid: int
    pos: int                 # 0-based
    cigar: np.ndarray        # uint32 BAM-encoded
    seq4: np.ndarray         # uint8 BAM packed bases
    qual: np.ndarray         # uint8 raw phred
    l_qseq: int
    has_sa: bool = False
    tags: dict = field(default_factory=dict)   # filled by annotate_records: rs, am, as, ar, ab


def _host_record(rec: Record):
    cg = np.ascontiguousarray(rec.cigar, dtype=np.uint32)
    s4 = np.ascontiguousarray(rec.seq4, dtype=np.uint8)
    ql = np.ascontiguousarray(rec.qual, dtype=np.uint8)
    hr = HostRecord(rec.flag, int(rec.has_sa), cg.ctypes.data_as(C.POINTER(C.c_uint32)), len(cg),
                    s4.ctypes.data_as(C.POINTER(C.c_uint8)), ql.ctypes.data_as(C.POINTER(C.c_uint8)),
                    rec.l_qseq, rec.tid, rec.pos)
    return hr, (cg, s4, ql)


def annotate_records(ctx: Context, records: list[Record], batch: Batch | None = None) -> list[Record]:
    """Batched equivalent of `foreach(rec; parallel(bam.allRecords)) annotateTask(...)`
    (source/anno.d:44-50): every record gets tags['rs'], artifact records also am/as/ar/ab."""
    L = lib()
    n = len(records)
    total_seq = sum((r.l_qseq + 1) // 2 for r in records)
    own = batch is None
    if own:
        batch = ctx.alloc_batch(max(n, 1), max(total_seq, 16))
    hrs, keep, prep = [], [], []
    off = 0
    for k, rec in enumerate(records):
        hr, refs = _host_record(rec)
        hrs.append(hr)
        keep.append(refs)
        al, cl, cr, rs = C.c_int32(), C.c_int32(), C.c_int32(), C.c_uint8()
        L.fadehost_prepare(C.byref(hr), C.byref(al), C.byref(cl), C.byref(cr), C.byref(rs))
        prep.append((al.value, cl.value, cr.value, rs.value))
        nb = (rec.l_qseq + 1) // 2
        batch.seq_off[k] = off
        batch.seq4[off:off + nb] = refs[1][:nb]
        off += nb
        batch.l_qseq[k] = rec.l_qseq
        batch.tid[k] = rec.tid
        batch.pos[k] = rec.pos
        batch.aligned_len[k] = al.value
        batch.clip_left[k] = cl.value
        batch.clip_right[k] = cr.value
    batch.seq_off[n] = off
    batch.run(n)
    for k, rec in enumerate(records):
        al, cl, cr, rs = prep[k]
        cap = 4 * rec.l_qseq + 256 + (len(ctx.contig_names[rec.tid]) if 0 <= rec.tid < len(ctx.contig_names) else 0)
        am, as_, ar, ab = (C.create_string_buffer(cap) for _ in range(4))
        rs_out = C.c_uint8()
        name = ctx.contig_names[rec.tid].encode() if 0 <= rec.tid < len(ctx.contig_names) else b""
        ops = np.ascontiguousarray(batch.ops[k])
        rc = L.fadehost_finish(C.byref(hrs[k]), name, rs, cl, cr, al, int(batch.flags[k]), int(batch.win_start[k]),
                               int(batch.beg_ref[k]), int(batch.n_ops[k]), ops.ctypes.data_as(C.POINTER(C.c_uint32)),
                               C.byref(rs_out), am, as_, ar, ab, cap)
        if rc < 0:
            raise FadeGpuError(rc, "fadehost_finish: buffer too small")
        rec.tags = {"rs": rs_out.value}
        if rc == 1:
            rec.tags.update(am=am.value.decode(), ar=ar.value.decode(), ab=ab.value.decode())
            rec.tags["as"] = as_.value.decode()
    if own:
        batch.close()
    return records
