"""Throughput of queued region jobs (fadegpu_submit_regions / fadegpu_job_wait) against the synchronous calls
(fadegpu_align_regions, fadegpu_score_regions) on the same read-shaped regions.

The alignments are those of tools/regions_bench.py: the aligned reads of BASELINE configs[1] (c2)'s first --reads
simulated reads, each read's forward letters on strand 1 against its window of the resident 100 Mbp reference.  The
whole set is streamed --passes times in chunks of --chunks regions.  For each chunk size, traced (max_ops --max-ops)
and score-only, --rounds times in alternation:
  * sync: one synchronous call per chunk, back to back;
  * jobs depth d (d = 1..4): d jobs reused in turn, at most d in flight; chunk k is submitted once job k - d is
    waited for.
Each leg reports regions per second host to host (wall clock over all chunks), the SW-kernel time summed over its
calls or jobs (the stats' kernel_ms, which for jobs can include overlapped work of neighbouring jobs) as a share of the
wall time, and whether every job's records and ops are byte-equal to the synchronous call's on the same chunk.  The
card's name, power limit and SM clock are printed beside the numbers.

    python tools/jobs_bench.py [--reads 1000000] [--chunks 41211,164843] [--passes 4]
"""
from __future__ import annotations

import argparse
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from fade_b200 import Context, Job, api, sim  # noqa: E402
from pairs_bench import READ_SEED, REF_LEN, REF_SEED, card  # noqa: E402
from regions_bench import c2_alignments  # noqa: E402


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reads", type=int, default=1_000_000)
    ap.add_argument("--max-ops", type=int, default=32, help="CIGAR ops returned per alignment of the traced legs")
    ap.add_argument("--chunks", default="41211,164843", help="regions per call / job, comma-separated")
    ap.add_argument("--passes", type=int, default=4, help="times the whole set of regions is streamed per leg")
    ap.add_argument("--depths", default="1,2,3,4")
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()

    t0 = time.time()
    contig = sim.make_contig(REF_SEED, 0, REF_LEN, 0, 0, 0.0)
    rd = sim.make_reads(sim.default_cfg(read_seed=READ_SEED), 0, a.reads, [contig], with_records=False)
    ref = contig.tobytes()
    print(f"card: {card()}")
    print(f"workload: c2, first {a.reads} reads (seed {READ_SEED}) vs {REF_LEN} bp (seed {REF_SEED}); "
          f"generated in {time.time() - t0:.1f} s")
    depths = [int(x) for x in a.depths.split(",")]
    with Context(0) as ctx:
        ctx.load_reference(["chrS"], [ref])
        b, al, fwd, _, _, starts, ends = c2_alignments(ctx, rd, ref)
        b.close()
        n = len(al)
        rq, rqo, tids, starts, ends, strands = api.pack_regions(fwd, np.zeros(n), starts, ends, np.ones(n))
        print(f"alignments: {n} regions (the aligned reads), {len(rq)} query bases; streamed {a.passes} times per leg")
        for size in [int(x) for x in a.chunks.split(",")]:
            bounds = [(k, min(k + size, n)) for k in range(0, n, size)]
            chunks = [(rq, rqo[k0:k1 + 1], tids[k0:k1], starts[k0:k1], ends[k0:k1], strands[k0:k1])
                      for k0, k1 in bounds] * a.passes
            for score_only in (False, True):
                max_ops = 0 if score_only else a.max_ops
                call = ctx.score_regions if score_only else ctx.align_regions
                tag = f"chunk {size} {'score_regions' if score_only else 'align_regions'}"

                def sync():
                    if score_only:
                        return [call(q, t, s, e, st, query_offsets=qo) for q, qo, t, s, e, st in chunks]
                    return [call(q, t, s, e, st, max_ops, query_offsets=qo) for q, qo, t, s, e, st in chunks]

                def jobs(depth, pool):
                    out = [None] * len(chunks)
                    for k, (q, qo, t, s, e, st) in enumerate(chunks):
                        if k >= depth:
                            out[k - depth] = pool[k % depth].wait()
                        pool[k % depth].submit_regions(q, t, s, e, st, None if score_only else max_ops,
                                                       score_only=score_only, query_offsets=qo)
                    for k in range(max(0, len(chunks) - depth), len(chunks)):
                        out[k] = pool[k % depth].wait()
                    return out

                pools = {d: [Job(ctx) for _ in range(d)] for d in depths}
                want = sync()                                                   # warm-up of every leg
                for d in depths:
                    jobs(d, pools[d])
                for rnd in range(a.rounds):
                    legs = [("sync", sync)] + [(f"jobs depth {d}", lambda d=d: jobs(d, pools[d])) for d in depths]
                    for name, leg in legs:
                        t1 = time.perf_counter()
                        res = leg()
                        wall = time.perf_counter() - t1
                        kms = sum(r.stats.kernel_ms for r in res)
                        same = all(r.records.tobytes() == w.records.tobytes() and
                                   (score_only or r.ops.tobytes() == w.ops.tobytes()) for r, w in zip(res, want))
                        print(f"round {rnd} {tag} {name}: {n * a.passes / wall:.4g} regions/s ({wall * 1e3:.1f} ms "
                              f"wall for {len(chunks)} calls), SW kernels {kms:.1f} ms = {kms / (wall * 1e3):.0%} of "
                              f"wall; records equal to the synchronous call: {same}")
                for p in pools.values():
                    for j in p:
                        j.close()


if __name__ == "__main__":
    main()
