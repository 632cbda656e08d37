"""Throughput of fadegpu_align_regions on read-shaped regions, beside fadegpu_align_pairs, the score-only calls
(fadegpu_score_regions / fadegpu_score_pairs) and the annotate path on the same alignments.

The alignments are those of BASELINE configs[1] (c2), as in tools/pairs_bench.py: the first --reads simulated 2x150
reads against the synthetic 100 Mbp chromosome (seeds as bench.py), and for every read the annotate path aligns, its
forward letters on strand 1 against its window [win_start, window end) of the resident reference.  One annotate batch
of the same reads is submitted and waited for; then, --rounds times in alternation:
  * regions: one Context.align_regions call from host arrays to host results (wall clock), with its kernel ms (the SW
    kernels), total device ms, H2D / D2H bytes and launches from the call's stats;
  * score_regions: the same for one Context.score_regions call on the same inputs (score and end cell, no traceback);
  * pairs: the same for one Context.align_pairs call on (RC(read), window letters);
  * score_pairs: the same for one Context.score_pairs call on those pairs;
  * batch: fadegpu_replay_kernels of the annotate batch (binning + the same SW kernels, nothing copied).
Every round checks that the region and pair records equal each other and the annotate batch's, and that the score-only
legs' score, end_query and end_ref equal their traced legs'.  The card's name, power limit and SM clock are printed
beside the numbers.

    python tools/regions_bench.py [--reads 1000000] [--max-ops 32]
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

from fade_b200 import Context, api, sim  # noqa: E402
from oracle import oracle as orc  # noqa: E402
from pairs_bench import READ_SEED, REF_LEN, REF_SEED, card  # noqa: E402

FIELDS = ("score", "end_query", "end_ref", "beg_query", "beg_ref", "n_ops")


def line(name, rnd, n, wall, st):
    print(f"round {rnd} {name}: {n / wall:.4g} /s ({wall * 1e3:.2f} ms wall), kernel {st.kernel_ms:.3f} ms "
          f"({st.cells / (st.kernel_ms * 1e6):.1f} GCUPS, {st.cells} cells), device total {st.total_ms:.3f} ms, "
          f"h2d {st.h2d_bytes} B, d2h {st.d2h_bytes} B, {st.kernel_launches} launches, {st.n_generic} generic")


def c2_alignments(ctx, rd, ref):
    """one annotate batch of the reads rd on ctx (reference ref loaded), and every alignment it ran: (batch, read
    indices, forward letters, reverse-complement letters, window letters, window starts, window ends)"""
    b = ctx.alloc_batch(rd.n, int(rd.seq_off[rd.n]))
    b.fill(rd.seq4, rd.seq_off, rd.l_qseq, rd.tid, rd.pos, rd.aligned_len, rd.clip_left, rd.clip_right).run()
    al = np.nonzero(b.flags[:rd.n] & api.R_ALIGNED)[0]
    W = ctx.params.window_size
    fwd, rcs, ts = [], [], []
    starts = b.win_start[al].astype(np.int64)
    ends = np.minimum(rd.pos[al] + rd.aligned_len[al] + W, len(ref)).astype(np.int64)
    for r, s, e in zip(al, starts, ends):
        so, lq = int(rd.seq_off[r]), int(rd.l_qseq[r])
        fwd.append(orc.decode_nt16(rd.seq4[so:so + (lq + 1) // 2], lq))
        rcs.append(orc.revcomp_nt16(rd.seq4[so:so + (lq + 1) // 2], lq))
        ts.append(ref[int(s):int(e)])
    return b, al, fwd, rcs, ts, starts, ends


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reads", type=int, default=1_000_000)
    ap.add_argument("--max-ops", type=int, default=32, help="CIGAR ops returned per alignment (n_ops is always exact)")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--replay-iters", type=int, default=5)
    a = ap.parse_args()

    t0 = time.time()
    contig = sim.make_contig(REF_SEED, 0, REF_LEN, 0, 0, 0.0)
    rd = sim.make_reads(sim.default_cfg(read_seed=READ_SEED), 0, a.reads, [contig], with_records=False)
    ref = contig.tobytes()
    print(f"card: {card()}")
    print(f"workload: c2, first {a.reads} reads (seed {READ_SEED}) vs {REF_LEN} bp (seed {REF_SEED}); "
          f"generated in {time.time() - t0:.1f} s")
    with Context(0) as ctx:
        ctx.load_reference(["chrS"], [ref])
        b, al, fwd, rcs, ts, starts, ends = c2_alignments(ctx, rd, ref)
        rq, rqo, tids, starts, ends, strands = api.pack_regions(fwd, np.zeros(len(al)), starts, ends, np.ones(len(al)))
        q, qo, t, to = api.pack_pairs(rcs, ts)
        n = len(al)
        print(f"alignments: {n} (the aligned reads), {len(rq)} query bases, {len(t)} window bases, max_ops {a.max_ops}")

        def regions():
            return ctx.align_regions(rq, tids, starts, ends, strands, a.max_ops, query_offsets=rqo)

        def pairs():
            return ctx.align_pairs(q, t, a.max_ops, query_offsets=qo, target_offsets=to)

        def score_regions():
            return ctx.score_regions(rq, tids, starts, ends, strands, query_offsets=rqo)

        def score_pairs():
            return ctx.score_pairs(q, t, query_offsets=qo, target_offsets=to)

        def timed(name, rnd, call):
            t1 = time.perf_counter()
            res = call()
            line(name, rnd, n, time.perf_counter() - t1, res.stats)
            return res

        reg, pr, sreg, spr = regions(), pairs(), score_regions(), score_pairs()               # warm-up
        b.replay_kernels(1)
        for rnd in range(a.rounds):
            reg = timed("regions", rnd, regions)
            sreg = timed("score_regions", rnd, score_regions)
            pr = timed("pairs", rnd, pairs)
            spr = timed("score_pairs", rnd, score_pairs)
            ms = b.replay_kernels(a.replay_iters) / a.replay_iters
            bst = b.stats()
            print(f"round {rnd} batch: replay_kernels {ms:.3f} ms per pass ({bst.cells / (ms * 1e6):.1f} GCUPS, "
                  f"{bst.n_aligned} alignments)")
            same_pairs = np.array_equal(reg.records, pr.records) and np.array_equal(reg.ops, pr.ops)
            same_batch = all(np.array_equal(reg.records[f], getattr(b, f)[al]) for f in FIELDS)
            print(f"round {rnd} records: regions == pairs (records and ops): {same_pairs}; "
                  f"regions == annotate batch ({', '.join(FIELDS)}): {same_batch}")
            same_score = [all(np.array_equal(s.records[f], tr.records[f]) for f in ("score", "end_query", "end_ref"))
                          for s, tr in ((sreg, reg), (spr, pr))]
            print(f"round {rnd} score-only records (score, end_query, end_ref): score_regions == regions: "
                  f"{same_score[0]}; score_pairs == pairs: {same_score[1]}")
        b.close()


if __name__ == "__main__":
    main()
