"""bench.py --dump-outputs: the sampled reads' results land in the right rows whatever order the records come in
(CPU, with a stand-in batch), the sample is fixed and inside 64 MB, and on a B200 the dump of a small bench run
equals the oracle read for read."""
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
from fade_b200 import api, sim
from oracle import oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class _Batch:
    """what OutputSample reads of a Batch: n, flags and results(), the records shuffled as the library may order them"""

    def __init__(self, n, rng, first):
        self.n = n
        self.flags = np.zeros(n + 3, np.uint8)
        self.flags[:n] = np.where(rng.random(n) < 0.5, rng.integers(0, 8, n) | 1, 0)
        reads = rng.permutation(np.where(self.flags[:n] & 1)[0])
        g = reads + first
        self.rec = np.zeros(len(reads), api.RESULT_DTYPE)
        self.rec["read"] = reads
        for i, f in enumerate(bench.OutputSample.FIELDS):
            self.rec[f] = g * 10 + i
        self.rec["n_ops"] = g % 14
        self.rec["flags"] = self.flags[reads]
        self.rec["ops"] = g[:, None] * 16 + np.arange(api.MAX_OPS)
        self.ws = g.astype(np.int64) * 3_000_000
        self.ridx = np.full(n, -1, np.int32)
        self.ridx[reads] = np.arange(len(reads))

    def results(self):
        return self.rec, self.ws, self.ridx


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}


def test_dump_rows_follow_result_index(tmp_path):
    rng = np.random.default_rng(5)
    s = bench.OutputSample(2500, 100)
    for a in range(0, 2500, 700):
        s.take(_Batch(min(700, 2500 - a), rng, a), a)
    s.write(str(tmp_path))
    d = _load(tmp_path)
    g = d["read"].astype(np.int64) - 100
    assert np.array_equal(g, np.arange(2500)) and all(v.dtype == np.float64 for v in d.values())
    has = d["flags"] % 2 == 1
    assert 0 < has.sum() < 2500
    for i, f in enumerate(bench.OutputSample.FIELDS[:-1]):
        assert np.array_equal(d[f][has], g[has] * 10 + i) and not d[f][~has].any()
    assert np.array_equal(d["n_ops"][has], g[has] % 14)
    assert np.array_equal(d["win_start"][has], g[has] * 3_000_000.0)
    assert np.array_equal(d["result_flags"], d["flags"])
    n_ops = np.minimum(g % 14, api.MAX_OPS)[:, None]
    live = has[:, None] & (np.arange(api.MAX_OPS)[None, :] < n_ops)
    assert np.array_equal(d["ops"], np.where(live, g[:, None] * 16 + np.arange(api.MAX_OPS), 0))


def test_dump_sample_of_a_large_stream_is_fixed_and_bounded():
    a, b = bench.OutputSample(10_000_000, 0), bench.OutputSample(10_000_000, 0)
    assert np.array_equal(a.idx, b.idx) and len(a.idx) == bench.DUMP_READS
    assert (np.diff(a.idx) > 0).all() and a.idx[-1] < 10_000_000
    assert a.idx.nbytes + sum(v.nbytes for v in a.out.values()) <= 64 << 20


@pytest.mark.gpu
def test_bench_dump_equals_the_oracle(tmp_path):
    """two groups of three chunks, two timed steps: every read's dumped result against the oracle"""
    n, ref_len = 6000, 2_000_000
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1",
                        "--reads", str(n), "--ref-len", str(ref_len), "--chunk", "1000", "--group", "3", "--file-reads", "0",
                        "--cpu-sample", "1000", "--scalar-sample", "0", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True)
    assert p.returncode == 0, p.stderr[-3000:]
    d = _load(tmp_path)
    assert np.array_equal(d["read"], np.arange(n))
    ref = sim.make_contig(bench.REF_SEED, 0, ref_len, 0, 0, 0.0)
    rd = sim.make_reads(sim.default_cfg(read_seed=bench.READ_SEED), 0, n, [ref], with_records=False)
    res, ops = orc.align_batch(rd.seq4, rd.seq_off, rd.l_qseq, rd.tid, rd.pos, rd.aligned_len, rd.clip_left,
                               rd.clip_right, [ref.tobytes()], ops_cap=api.MAX_OPS)
    al = res["aligned"] == 1
    assert 100 < al.sum() < n
    flags = d["flags"].astype(np.int64)
    assert np.array_equal(flags & 1, res["aligned"]) and np.array_equal((flags >> 1) & 1, res["art_left"])
    assert np.array_equal((flags >> 2) & 1, res["art_right"])
    for f in bench.OutputSample.FIELDS + ("win_start",):
        assert np.array_equal(d[f][al], res[f][al]) and not d[f][~al].any(), f
    live = np.arange(api.MAX_OPS)[None, :] < np.minimum(res["n_ops"], api.MAX_OPS)[:, None]
    assert np.array_equal(d["ops"], np.where(live & al[:, None], ops[:, :api.MAX_OPS], 0))
