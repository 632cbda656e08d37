"""Throughput of fadegpu_align_pairs on read-shaped pairs, beside the annotate path on the same alignments.

The pairs are those of BASELINE configs[1] (c2): the first --reads simulated 2x150 reads against the synthetic 100 Mbp
chromosome (seeds as bench.py), and for every read the annotate path aligns, the pair (RC(read), its window).  One
annotate batch of the same reads is submitted and waited for; then, three times in alternation:
  * pairs: one Context.align_pairs call from host arrays to host results (wall clock), with its kernel ms (the SW
    kernels), total device ms and H2D bytes from the call's stats;
  * batch: fadegpu_replay_kernels of the annotate batch (binning + the same SW kernels, nothing copied).
The card's name, power limit and SM clock are printed beside the numbers.

    python tools/pairs_bench.py [--reads 1000000] [--max-ops 32]
"""
from __future__ import annotations

import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from fade_b200 import Context, api, sim  # noqa: E402
from oracle import oracle as orc  # noqa: E402

REF_SEED, READ_SEED, REF_LEN = 1002, 2002, 100_000_000   # bench.py's c2


def card() -> str:
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader",
                               "-i", os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0]],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:   # the numbers still stand, without the card's settings
        return f"nvidia-smi unavailable ({e})"


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reads", type=int, default=1_000_000)
    ap.add_argument("--max-ops", type=int, default=32, help="CIGAR ops returned per pair (n_ops is always exact)")
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
        b = ctx.alloc_batch(rd.n, int(rd.seq_off[rd.n]))
        b.fill(rd.seq4, rd.seq_off, rd.l_qseq, rd.tid, rd.pos, rd.aligned_len, rd.clip_left, rd.clip_right).run()
        al = np.nonzero(b.flags[:rd.n] & api.R_ALIGNED)[0]
        W = ctx.params.window_size
        qs, ts = [], []
        for r in al:
            so = int(rd.seq_off[r])
            qs.append(orc.revcomp_nt16(rd.seq4[so:so + (int(rd.l_qseq[r]) + 1) // 2], int(rd.l_qseq[r])))
            end = min(int(rd.pos[r]) + int(rd.aligned_len[r]) + W, len(ref))
            ts.append(ref[int(b.win_start[r]):end])
        q, qo, t, to = api.pack_pairs(qs, ts)
        n = len(al)
        print(f"pairs: {n} (the aligned reads), {len(q)} query bases, {len(t)} target bases, max_ops {a.max_ops}")

        res = ctx.align_pairs(q, t, a.max_ops, query_offsets=qo, target_offsets=to)          # warm-up
        same = all(np.array_equal(res.records[f], getattr(b, f)[al]) for f in ("score", "end_ref", "beg_ref", "n_ops"))
        print(f"records equal the annotate batch's: {same}")
        b.replay_kernels(1)
        for rnd in range(a.rounds):
            t1 = time.perf_counter()
            res = ctx.align_pairs(q, t, a.max_ops, query_offsets=qo, target_offsets=to)
            wall = time.perf_counter() - t1
            st = res.stats
            print(f"round {rnd} pairs: {n / wall:.4g} pairs/s ({wall * 1e3:.2f} ms wall), kernel {st.kernel_ms:.3f} ms "
                  f"({st.cells / (st.kernel_ms * 1e6):.1f} GCUPS, {st.cells} cells, {st.kernel_launches} launches), "
                  f"device total {st.total_ms:.3f} ms, h2d {st.h2d_bytes} B, d2h {st.d2h_bytes} B, "
                  f"{st.n_generic} generic")
            ms = b.replay_kernels(a.replay_iters) / a.replay_iters
            bst = b.stats()
            print(f"round {rnd} batch: replay_kernels {ms:.3f} ms per pass ({bst.cells / (ms * 1e6):.1f} GCUPS, "
                  f"{bst.n_aligned} alignments)")
        b.close()


if __name__ == "__main__":
    main()
