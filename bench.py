#!/usr/bin/env python
"""bench.py -- headline benchmark of the `fade annotate` realignment hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload c2|c3|c4] [--dump-outputs DIR]

One "step" = one pass of the hot path over the whole workload, processed as chunks of --chunk reads
through the C ABI (libfadegpu.so).  Workloads (BASELINE.json `configs`):

  c2 (default, the bench line)  configs[1]: 10 M simulated 2x150 paired reads against a synthetic 100 Mbp
      chromosome, default window-size / min-length, PER GPU ("weak": every rank simulates its own reads).
  c3  configs[2]: 100 M reads against a 3.1 Gbp / 24-contig reference resident in every GPU's HBM; the read
      stream is SPLIT over the ranks ("strong").  Reads are generated group by group (--group chunks at a
      time, untimed) and every group is timed the same way as c2's single group; times add up.
  c4  configs[3]: 2x250 reads, --window-size 1000, clip law U{1..40} (use with --reads 2000000).

  value  reads/s with every chunk's inputs already resident in HBM: one CUDA-event interval around ALL
         kernel launches of the chunks (binning, fill, traceback rounds, generic kernel), queued back to
         back as consecutive submits queue them (fadegpu_replay_batches); no host work, no copies.
  e2e    reads/s through the public C ABI with HOST buffers, wall clock.  --e2e-path compact (default):
         every chunk's records sit in the pinned host view of its batch in the compact layout (one gate
         byte + one 32-byte record per read + the 4-bit bases, written there by the caller's BAM reader,
         INTEGRATION.md section 2); per chunk fadegpu_submit_compact copies the gate bytes, the GPU
         fetches the records and bases it needs, bins, aligns, and the result records come back;
         fadegpu_wait + fadegpu_get_results hand them to the host, which reads every flag byte and every
         record.  --e2e-path view: fadegpu_submit from the seven-array view (36 B / read uploaded).
         --e2e-path arrays: fadegpu_submit_inputs on pageable caller arrays.
  roofline  INT16x2 ALU roofline: cells/s against 2*R_alu/9 (SURVEY.md 8d) and against 2*R_alu/7.5 (the
         fill kernel's own instruction mix), R_alu measured live by fadegpu_measure_alu_peak.
  cpu_baseline  a CPU port of the path (oracle/fade_oracle_simd.c: AVX-512BW / AVX2, 32 / 16 alignments per vector, trace
         table + traceback, OpenMP on the host cores; validated against the scalar oracle) timed on a
         bounded sample of the same reads, and the scalar oracle beside it.  `--impl reference` prints
         that arm alone.

Multi-GPU: launched under torchrun, one rank per GPU, every rank with its own reference copy; no data-path
collective; value = all ranks' reads / max-over-ranks time.

--dump-outputs DIR: after the K timed steps, the results the last timed pass through the C ABI handed back (per-read
flags, and each read's record: score, begin / end cells, op count, ops, window start) for a fixed, seeded sample of
2^18 of rank 0's reads (all of them when there are fewer), one DIR/<name>.npy per field plus DIR/read.npy with the
sampled read numbers.  The workload is seeded, so the same arguments give the same inputs, and two builds can be
compared file for file.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

REF_LEN = 100_000_000
REF_SEED = 1002
READ_SEED = 2002
N_READS = 10_000_000
CHUNK = 1_000_000
C3_READS = 100_000_000
C3_BASES = 3.1e9
# --dump-outputs: 20 float64 values per sampled read, so 2^18 reads are 40 MiB (inside 64 MB)
DUMP_READS = 1 << 18
DUMP_SEED = 3003
# hg38 chr1-22,X,Y lengths; scaled to sum 3.1 Gbp (SURVEY.md 8d, C3)
HG38 = [248956422, 242193529, 198295559, 190214555, 181538259, 170805979, 159345973, 145138636, 138394717, 133797422,
        135086622, 133275309, 114364328, 107043718, 101991189, 90338345, 83257441, 80373285, 58617616, 64444167,
        46709983, 50818468, 156040895, 57227415]


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="fade_b200", choices=["fade_b200", "reference"])
    ap.add_argument("--reads", type=int, default=0,
                    help="reads per GPU per step (c2 / c4: default 10 M) or in total over all GPUs (c3: default 100 M)")
    ap.add_argument("--ref-len", type=int, default=REF_LEN)
    ap.add_argument("--chunk", type=int, default=CHUNK)
    ap.add_argument("--group", type=int, default=10, help="chunks resident (pinned host + HBM) at a time")
    ap.add_argument("--cpu-sample", type=int, default=4_000_000,
                    help="reads in the cpu_baseline sample (4 M reads = about 30 core-seconds of the SIMD port)")
    ap.add_argument("--scalar-sample", type=int, default=200_000, help="reads in the scalar-oracle sample (0 = skip)")
    ap.add_argument("--host-threads", type=int, default=0, help="host threads per rank (0 = cores / ranks)")
    ap.add_argument("--depth", type=int, default=3, help="chunks in flight in the e2e loop")
    ap.add_argument("--e2e-path", default="compact", choices=["compact", "view", "arrays"],
                    help="compact = fadegpu_submit_compact (gate byte + 32-byte record per read in the pinned view); "
                         "view = fadegpu_submit (seven arrays); arrays = fadegpu_submit_inputs from pageable arrays")
    ap.add_argument("--workload", default="c2", choices=["c2", "c3", "c4"])
    ap.add_argument("--tags-only", action="store_true",
                    help="FADEGPU_F_TAGS_ONLY: no traceback for alignments whose score already fails both accept predicates "
                         "(what the file drivers use; NOT the default bench line, which produces every record in full)")
    ap.add_argument("--file-reads", type=int, default=1_000_000,
                    help="records of the e2e_file leg (fade-b200 annotate BAM -> BAM on the first reads of the workload; 0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned for a fixed, seeded sample of rank 0's "
                         "reads as DIR/<name>.npy (float64), to compare two builds output for output")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if a.dump_outputs and (a.impl == "reference" or a.e2e_path == "arrays"):
        ap.error("--dump-outputs reads the results the GPU path leaves resident in its batches: "
                 "it needs --impl fade_b200 and --e2e-path compact or view")
    if a.reads <= 0:
        a.reads = C3_READS if a.workload == "c3" else N_READS
    return a


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed regions (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []
        self.windows = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "200"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append((time.time(), ln.strip()))

    def window(self, t0: float, t1: float):
        self.windows.append((t0, t1))

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, ln in self.lines:
            if self.windows and not any(a - 0.05 <= ts <= b + 0.15 for a, b in self.windows):
                continue          # a sample taken while the next group of reads was being generated
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for nm, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "power_w_max": max(pw),
                "samples": len(sm), "reasons": sorted(reasons)}


class Workload:
    """reference + this rank's slice of the read stream, generated group by group"""

    def __init__(self, args, rank: int, world: int):
        from fade_b200 import shard, sim
        self.args = args
        self.kind = args.workload
        self.window = 1000 if self.kind == "c4" else 300
        t0 = time.time()
        if self.kind == "c3":
            scale = C3_BASES / sum(HG38)
            lens = [int(x * scale) for x in HG38]
            self.names = [f"chr{i + 1}" for i in range(22)] + ["chrX", "chrY"]
            self.contigs = [sim.make_contig(1003, i, n, 1_000_000, 10_000, 0.0) for i, n in enumerate(lens)]
            self.cfg = sim.default_cfg(read_seed=2003)
            self.first, self.last = shard.shard_range(args.reads, rank, world)      # strong: the stream is split
            self.scaling = "strong"
        else:
            self.names = ["chrS"]
            self.contigs = [sim.make_contig(REF_SEED, 0, args.ref_len, 0, 0, 0.0)]
            if self.kind == "c4":
                self.cfg = sim.default_cfg(read_seed=2004, read_len=250, window=1000, frag_mean=600, frag_sd=80,
                                           short_clip_law=1)
            else:
                self.cfg = sim.default_cfg(read_seed=READ_SEED)
            self.first, self.last = shard.weak_range(args.reads, rank)              # weak: every rank its own reads
            self.scaling = "weak"
        self.n = self.last - self.first
        self.gen_s = time.time() - t0
        g = max(1, args.group) * args.chunk
        self.groups = [(a, min(self.last, a + g) - a) for a in range(self.first, self.last, g)] or [(self.first, 0)]

    def reads(self, first: int, n: int):
        from fade_b200 import sim
        t0 = time.time()
        rd = sim.make_reads(self.cfg, first, n, self.contigs, with_records=False)
        self.gen_s += time.time() - t0
        return rd

    def config(self) -> dict:
        a = self.args
        if self.kind == "c4":
            desc = (f"{a.reads} simulated 2x250 paired reads (seed 2004, clip lengths U(1..40)) vs synthetic "
                    f"{a.ref_len} bp chromosome (seed {REF_SEED}), window-size 1000, min-length 5, per GPU")
        elif self.kind == "c3":
            desc = (f"{a.reads} simulated 2x150 paired reads (seed 2003) split over the GPUs vs synthetic "
                    f"{sum(len(c) for c in self.contigs)} bp reference in 24 contigs (hg38 proportions, seed 1003, 1 % N runs) "
                    f"resident in every GPU's HBM, window-size 300, min-length 5")
        else:
            desc = (f"{a.reads} simulated 2x150 paired reads (seed {READ_SEED}) vs synthetic "
                    f"{a.ref_len} bp chromosome (seed {REF_SEED}), window-size 300, min-length 5, per GPU")
        if a.tags_only:
            desc += "; FADEGPU_F_TAGS_ONLY (no traceback where the score rules out both accept predicates)"
        return {"workload": desc, "chunk_reads": a.chunk, "resident_chunks": a.group,
                "l2": "inputs + checkpoint scratch per chunk (>2 GB) exceed the 126 MB L2; no explicit flush"}


class OutputSample:
    """What the path hands a caller (fadegpu_get_results after fadegpu_wait), kept for a fixed, seeded sample of the
    rank's reads, one row per read.  The records come in an unspecified order, so each is placed through result_index;
    a read without a record keeps zeros in the record fields, and ops past min(n_ops, MAX_OPS) are zeroed.  float64
    holds every int32 / uint32 / int64 field exactly."""
    FIELDS = ("score", "end_query", "end_ref", "beg_query", "beg_ref", "n_ops")

    def __init__(self, n_reads: int, first: int):
        from fade_b200 import api
        self.max_ops = api.MAX_OPS
        if n_reads > DUMP_READS:
            self.idx = np.sort(np.random.default_rng(DUMP_SEED).choice(n_reads, DUMP_READS, replace=False))
        else:
            self.idx = np.arange(n_reads)
        self.first = first
        n = len(self.idx)
        self.out = {k: np.zeros(n) for k in ("flags", *self.FIELDS, "result_flags", "win_start")}
        self.out["ops"] = np.zeros((n, self.max_ops))

    def take(self, b, first: int):
        """the sampled reads among [first, first + b.n) of the rank's stream, from batch b's last results"""
        lo, hi = np.searchsorted(self.idx, [first, first + b.n])
        k = self.idx[lo:hi] - first
        rec, ws, ridx = b.results()
        self.out["flags"][lo:hi] = b.flags[k]
        r = ridx[k]
        row = np.arange(lo, hi)[r >= 0]
        r = r[r >= 0]
        for f in self.FIELDS:
            self.out[f][row] = rec[f][r]
        self.out["result_flags"][row] = rec["flags"][r]
        self.out["win_start"][row] = ws[r]
        live = np.arange(self.max_ops)[None, :] < np.minimum(rec["n_ops"][r], self.max_ops)[:, None]
        self.out["ops"][row] = np.where(live, rec["ops"][r], 0)

    def write(self, d: str):
        os.makedirs(d, exist_ok=True)
        np.save(os.path.join(d, "read.npy"), (self.idx + self.first).astype(np.float64))
        for k, v in self.out.items():
            np.save(os.path.join(d, f"{k}.npy"), v)


def cpu_kind() -> str:
    """What the SIMD arm is on this host: the widest of AVX-512BW (32 int16 lanes) and AVX2 (16) the CPU runs."""
    from oracle import oracle as orc
    lanes = orc.simd_lanes()
    isa = {32: "AVX-512BW 32-lane", 16: "AVX2 16-lane"}.get(lanes, "scalar (no AVX2 on this host)")
    return (f"{isa} inter-sequence port of the path (oracle/fade_oracle_simd.c: SW fill with trace table, "
            "traceback, predicates; in-memory reference), validated against the scalar oracle")


def cpu_baseline(contigs, rd, n_sample: int, threads: int, window: int = 300, simd: bool = True):
    """CPU port of the path on the host cores over the first n_sample reads: reads/s, GCUPS."""
    from oracle import oracle as orc
    prm = orc.default_params(window_size=window)
    n = min(n_sample, rd.n)
    sl = slice(0, n)
    off = rd.seq_off[: n + 1]
    t0 = time.perf_counter()
    res, _ = orc.align_batch(rd.seq4[: int(off[n])], off, rd.l_qseq[sl], rd.tid[sl], rd.pos[sl], rd.aligned_len[sl],
                             rd.clip_left[sl], rd.clip_right[sl], contigs, params=prm, n_threads=threads, simd=simd,
                             ops_cap=10)
    dt = time.perf_counter() - t0
    al = res["aligned"] == 1
    cells = int((rd.l_qseq[sl][al].astype(np.int64) * res["tlen"][al]).sum())
    return n / dt, cells / dt / 1e9, n, dt


def run_reference(args, rank: int, world: int):
    """Reference arm: the reference's CPU implementation of the path.  The real `fade` binary cannot
    be built here (D + dparasail/parasail + dhtslib/htslib are absent), so this times the oracle
    port on all host cores (kind "port"), one bounded sample per step."""
    if rank != 0:
        return
    wl = Workload(args, 0, 1)
    rd = wl.reads(wl.first, min(max(args.cpu_sample, 1), wl.n))
    threads = os.cpu_count() or 1          # rank 0 alone runs this arm: it may use every host core
    from fade_b200 import sim as _sim
    _sim.set_threads(threads)
    vals, gc = [], []
    for i in range(args.warmup + args.steps):
        v, g, n, dt = cpu_baseline(wl.contigs, rd, args.cpu_sample, threads, wl.window)
        if i >= args.warmup:
            vals.append(v); gc.append(g)
    v = statistics.mean(vals)
    sample = f"first {rd.n} reads of the workload per step; {cpu_kind()}; OpenMP {threads} threads"
    # parasail 2.4.3 (what real fade links) has no AVX-512 kernels: when the arm above ran 32 lanes, one more pass
    # with the 16-lane AVX2 kernel says what the narrower ISA gives on the same cores
    from oracle import oracle as orc
    avx2 = None
    if orc.simd_lanes() == 32:
        os.environ["FADE_ORACLE_SIMD"] = "avx2"
        try:
            v2, g2, _, _ = cpu_baseline(wl.contigs, rd, args.cpu_sample, threads, wl.window)
            avx2 = {"value": v2, "unit": "reads/s", "gcups": g2,
                    "note": "same sample, 16-lane AVX2 kernel forced (FADE_ORACLE_SIMD=avx2): the widest ISA parasail 2.4.3 has kernels for"}
        finally:
            del os.environ["FADE_ORACLE_SIMD"]
    line = {
        "impl": "reference", "metric": "annotate_reads_per_sec", "value": v, "unit": "reads/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * rd.n / v,
        "higher_is_better": True, "scaling": wl.scaling, "vs_baseline": None, "dtype": "int16", "data": "synthetic",
        "config": wl.config(), "gcups": statistics.mean(gc),
        "cpu_baseline": {"value": v, "unit": "reads/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if avx2:
        line["cpu_baseline"]["avx2_16_lane"] = avx2
    print(json.dumps(line), file=args.out, flush=True)


def claim_stdout():
    """Keep stdout clean for the ONE JSON line: everything else that writes to fd 1 (NCCL's version
    banner, library chatter) goes to stderr; returns a writer bound to the real stdout."""
    sys.stdout.flush()
    real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    return real


def file_level_e2e(wl: Workload, n_reads: int, threads: int, device: int):
    """`fade-b200 annotate -b in.bam ref.fa > out.bam` (the repo's own C++ driver, fade_b200/csrc/host) on the first
    n_reads records of the workload: records/s of the whole process and of its record loop (FADE_TIMING)."""
    import tempfile
    from fade_b200 import sim
    exe = os.path.join(ROOT, "fade_b200", "bin", "fade-b200")
    if n_reads <= 0 or not os.path.exists(exe) or not hasattr(sim, "write_bam"):
        return None
    d = tempfile.mkdtemp(prefix="fade_bench_")
    try:
        rd = sim.make_reads(wl.cfg, wl.first, min(n_reads, wl.n), wl.contigs, with_records=True)
        fa, bam, out = (os.path.join(d, x) for x in ("ref.fa", "in.bam", "out.bam"))
        sim.write_fasta(fa, wl.names, wl.contigs)
        sim.write_bam(bam, wl.names, wl.contigs, rd)
        env = dict(os.environ, FADE_TIMING="1", OMP_NUM_THREADS=str(threads))

        def once(level):
            t0 = time.perf_counter()
            with open(out, "wb") as f:
                p = subprocess.run([exe, "annotate", "-b", "--level", str(level), "-t", str(threads), "--device", str(device), bam, fa],
                                   stdout=f, stderr=subprocess.PIPE, text=True, env=env)   # level "fast" = the driver's default
            wall = time.perf_counter() - t0
            if p.returncode != 0:
                return None, p.stderr[-300:]
            loop, phases = None, None
            for ln in p.stderr.splitlines():
                if "record loop" in ln:
                    loop = float(ln.split("record loop")[1].split("s:")[0])
                    phases = ln.split("record loop")[1].strip()
            return {"records_per_s": rd.n / wall, "wall_s": round(wall, 3), "record_loop_s": loop,
                    "record_loop_records_per_s": (rd.n / loop) if loop else None, "phases": phases,
                    "out_bytes": os.path.getsize(out)}, None
        once("fast")                      # untimed: page cache, CUDA module load
        rf, err = once("fast")
        if rf is None:
            return {"error": err}
        r6, _ = once(6)
        return {"value": rf["record_loop_records_per_s"], "unit": "records/s", "records": rd.n,
                "record_loop_s": rf["record_loop_s"], "whole_process_records_per_s": rf["records_per_s"], "wall_s": rf["wall_s"],
                "what": "fade-b200 annotate -b (BGZF BAM in, BGZF BAM out with the driver's built-in DEFLATE encoder). value = records/s of "
                        "its record loop (first record read to last record written: inflate, parse, submit, wait, tag, deflate, write); "
                        "the whole process adds a fixed start-up (CUDA context, FASTA load, reference upload, pinned buffers: wall_s - "
                        "record_loop_s) that 1 M records do not amortise (10 M records: profiles/r02_c5_chain.json)",
                "phases": rf["phases"], "zlib_level_6": r6,
                "in_bytes": os.path.getsize(bam), "out_bytes": rf["out_bytes"], "threads": threads}
    finally:
        import shutil
        shutil.rmtree(d, ignore_errors=True)


def main():
    args = parse_args()
    out = claim_stdout()
    # A ctx drives four streams (fills, traceback, uploads + binning, results) that must overlap.  With the default of 8
    # hardware queues per device they can end up sharing a queue with each other once NCCL has added its own streams
    # (N > 1), which serialises the binning of the next batch behind the running fill.  Must be set before the CUDA
    # context exists; fadegpu_create sets the same default for processes that have not created one yet.
    os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
    from fade_b200 import shard as _shard
    rank, local_rank, world = _shard.world()
    # torchrun exports OMP_NUM_THREADS=1; the host side of the path (gather / scatter) and the generators are
    # told their thread count explicitly instead: the node's cores split by ranks
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
    host_threads = args.host_threads or max(1, (os.cpu_count() or 1) // max(1, local_world))
    args.host_threads = host_threads
    args.out = out
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    from fade_b200 import sim as _sim
    _sim.set_threads(host_threads)

    import torch
    import torch.distributed as dist
    from fade_b200 import Context

    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        torch.cuda.synchronize(local_rank)
        if world > 1:
            dist.barrier()

    from fade_b200 import shard
    red = shard.Reducer(world, device=f"cuda:{local_rank}")
    max_over_ranks, sum_over_ranks = red.max, red.sum

    wl = Workload(args, rank, world)
    dump = OutputSample(wl.n, wl.first) if (args.dump_outputs and rank == 0) else None
    from fade_b200 import default_params
    from fade_b200 import api as _api
    # compact results (fadegpu_get_results): fadegpu_wait rebuilds only flags[] and the result index
    ctx = Context(local_rank, default_params(host_threads=host_threads, window_size=wl.window,
                                             flags=_api.F_NO_SCATTER | (_api.F_TAGS_ONLY if args.tags_only else 0)))
    ctx.load_reference(wl.names, wl.contigs)
    alu_ops, max_mhz = ctx.measure_alu_peak()

    chunk = max(1, min(args.chunk, max(g[1] for g in wl.groups)))
    stride = (wl.cfg.read_len + 1) // 2
    path = args.e2e_path
    n_batches = max(1, max((g[1] + chunk - 1) // chunk for g in wl.groups))
    batches = [ctx.alloc_batch(chunk, chunk * stride) for _ in range(n_batches if path != "arrays" else 2)]

    def load_chunk(b, rd, a, e):
        """the host side of a chunk: its records in the pinned view of its batch (untimed: the BAM reader's job)"""
        m = e - a
        args_ = (rd.seq4[a * stride: e * stride], rd.seq_off[a: e + 1] - rd.seq_off[a], rd.l_qseq[a:e], rd.tid[a:e],
                 rd.pos[a:e], rd.aligned_len[a:e], rd.clip_left[a:e], rd.clip_right[a:e])
        if path == "compact":
            b.fill_compact(*args_)
        else:
            b.fill(*args_)
        b.n = m

    def submit(b):
        if path == "compact":
            b.submit_compact()
        else:
            b.submit()

    agg = {"aligned": 0, "cells": 0, "launches": 0, "generic": 0, "art": 0, "oversize": 0}
    stage = {"fill": 0.0, "trace": 0.0, "gen": 0.0}
    copies = {"h2d": 0, "d2h": 0}
    host_ms = {}

    def collect_stats(b):
        st = b.stats()
        agg["aligned"] += st.n_aligned; agg["cells"] += st.cells; agg["launches"] += st.kernel_launches
        agg["generic"] += st.n_generic; agg["oversize"] += st.n_oversize
        agg["art"] += int(((b.flags[: b.n] & 6) != 0).sum())

    def note_copies(b):
        st = b.stats()
        copies["h2d"] += st.h2d_bytes; copies["d2h"] += st.d2h_bytes

    def note_host(b):
        st = b.stats()
        for kx in ("host_submit_ms", "host_wait_ms", "host_classify_ms", "host_sort_ms", "host_gather_ms"):
            host_ms[kx] = host_ms.get(kx, 0.0) + getattr(st, kx)

    def consume(b):
        """read the chunk's results on the host: the rs-relevant flags of every read + the compact records"""
        rec, ws, ridx = b.results()
        m8 = b.n & ~7                        # every flag byte, eight at a time
        return int(b.flags[:m8].view(np.uint64).sum(dtype=np.uint64) & 0xffff) + int(b.flags[m8: b.n].sum()) \
            + int(rec["score"].sum()) + len(ws)

    # rank 0 prints the line, so rank 0 samples its GPU; eight pollers of the driver on one box would only disturb
    # the other ranks' launches
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e2e_steps = []      # wall seconds of every e2e pass of this rank
    k_ms = 0.0          # device ms of the kernel-only passes, all groups, all steps
    e_s = 0.0           # wall seconds of the e2e passes
    cb = None
    scalar = None
    for gi, (gfirst, gn) in enumerate(wl.groups):
        rd = wl.reads(gfirst, gn)
        bounds = [(a, min(gn, a + chunk)) for a in range(0, gn, chunk)]
        live = batches[: len(bounds)] if path != "arrays" else batches

        # ---- make the group resident (untimed) and collect its statistics ----
        if path != "arrays":
            for b, (a, e) in zip(live, bounds):
                load_chunk(b, rd, a, e)
                submit(b)
                b.wait()
                collect_stats(b)
                b.replay_kernels(1)          # serialised per-stage timers (fill / traceback / generic)
                st = b.stats()
                stage["fill"] += st.fill_ms; stage["trace"] += st.trace_ms; stage["gen"] += st.generic_ms

        def kernel_step(collect: bool = False):
            """inputs resident: only the kernels, timed with CUDA events on the device"""
            if path != "arrays":
                return ctx.replay_batches(live, 1)
            ms = 0.0
            for (a, e) in bounds:
                b = batches[0]
                b.fill(rd.seq4[a * stride: e * stride], rd.seq_off[a: e + 1] - rd.seq_off[a], rd.l_qseq[a:e], rd.tid[a:e],
                       rd.pos[a:e], rd.aligned_len[a:e], rd.clip_left[a:e], rd.clip_right[a:e]).run()
                ms += b.replay_kernels(1)
                if collect:
                    collect_stats(b)
                    st = b.stats()
                    stage["fill"] += st.fill_ms; stage["trace"] += st.trace_ms; stage["gen"] += st.generic_ms
            return ms

        def e2e_step():
            """host buffers -> C ABI -> host results, several chunks in flight; wall clock around the whole pass"""
            t0 = time.perf_counter()
            acc = 0
            if path != "arrays":
                issued = 0
                for i in range(len(bounds)):
                    while issued < min(len(bounds), i + args.depth):
                        submit(live[issued])
                        issued += 1
                    live[i].wait()
                    acc += consume(live[i])
                    note_copies(live[i])
                return time.perf_counter() - t0, acc
            pending = None
            for i, (a, e) in enumerate(bounds):
                b = batches[i & 1]
                b.submit_arrays(e - a, rd.seq4, rd.seq_off[a:], rd.l_qseq[a:], rd.tid[a:], rd.pos[a:],
                                rd.aligned_len[a:], rd.clip_left[a:], rd.clip_right[a:])   # seq_off: absolute offsets
                if pending is not None:
                    pending.wait()
                    acc += consume(pending)
                    note_copies(pending)
                pending = b
            pending.wait()
            acc += consume(pending)
            note_copies(pending)
            return time.perf_counter() - t0, acc

        if path == "arrays":
            kernel_step(True)
        if gi == 0:
            for _ in range(args.warmup):
                kernel_step()
            e2e_step()
        # ---- timed: kernels with resident inputs ----
        barrier()
        t_w0 = time.time()
        for s in range(args.steps):
            k_ms += kernel_step()
        barrier()
        # ---- timed: end to end through the C ABI ----
        for s in range(args.steps):
            # The K timed passes are bracketed by a barrier + synchronize on both sides; no barrier BETWEEN passes: it
            # phase-locks the ranks, and eight GPUs pulling their bases over PCIe in the same microseconds cost every
            # pass 1.3 ms on the 8-GPU box (FADE_BENCH_STEP_BARRIER=1 restores it; with the ranks 0.7 ms out of phase,
            # FADE_BENCH_STAGGER_MS=0.7, a pass is another 1.3 ms shorter -- profiles/README.md).
            if s == 0 or os.environ.get("FADE_BENCH_STEP_BARRIER"):
                barrier()
            if os.environ.get("FADE_BENCH_STAGGER_MS"):      # diagnostics: ranks out of phase by a fixed offset
                time.sleep(1e-3 * float(os.environ["FADE_BENCH_STAGGER_MS"]) * rank)
            copies["h2d"] = copies["d2h"] = 0
            dt, _ = e2e_step()
            e_s += dt
            e2e_steps.append(dt)
            if s == 0:          # bytes over PCIe of ONE pass over this group
                agg["h2d"] = agg.get("h2d", 0) + copies["h2d"]
                agg["d2h"] = agg.get("d2h", 0) + copies["d2h"]
        barrier()
        sampler.window(t_w0, time.time())
        if dump:        # untimed: the group's last timed pass left every chunk's results in its batch
            for b, (a, _) in zip(live, bounds):
                dump.take(b, gfirst - wl.first + a)
        for b in (live if path != "arrays" else batches):
            note_host(b)
        if gi == 0 and rank == 0:
            cb = cpu_baseline(wl.contigs, rd, args.cpu_sample, host_threads, wl.window)
            if args.scalar_sample > 0:
                scalar = cpu_baseline(wl.contigs, rd, args.scalar_sample, host_threads, wl.window, simd=False)
    clocks = sampler.stop() if rank == 0 else None
    if dump:
        dump.write(args.dump_outputs)

    per_rank = None
    if world > 1:       # every rank's e2e passes (diagnostics of the scaling curve): mean and worst pass in ms
        mine = [1e3 * statistics.mean(e2e_steps), 1e3 * max(e2e_steps), 1e3 * min(e2e_steps)]
        gathered = [None] * world
        dist.all_gather_object(gathered, mine)
        per_rank = [[round(x, 2) for x in g] for g in gathered]
    k_ms_max = max_over_ranks(k_ms)
    e_s_max = max_over_ranks(e_s)
    total_reads = sum_over_ranks(float(wl.n))
    total_cells = sum_over_ranks(float(agg["cells"]))
    total_aligned = sum_over_ranks(float(agg["aligned"]))
    ms_per_step = k_ms_max / args.steps
    value = total_reads / (ms_per_step * 1e-3)
    e2e_value = total_reads / (e_s_max / args.steps)

    # the pinned batches and the ctx go first: the file-level leg below starts a process of its own on the same GPU
    for b in batches:
        b.close()
    ctx.close()
    if rank == 0:
        cells_rank = float(agg["cells"])
        achieved = cells_rank / (k_ms / args.steps * 1e-3) / 1e9            # GCUPS, all kernels of the path, this rank
        k_fill, k_trace, k_gen = stage["fill"], stage["trace"], stage["gen"]
        fill_gcups = cells_rank / (k_fill * 1e-3) / 1e9 if k_fill > 0 else None
        peak9 = 2.0 * alu_ops / 9.0 / 1e9                                   # SURVEY 8(d): 9 packed instr / 2 cells
        peak75 = 2.0 * alu_ops / 7.5 / 1e9                                  # the fill kernel's own mix: 7.5 / 2 cells
        # algorithmic HBM bytes per alignment (SURVEY 8d): window 2-bit + N mask, query, metadata, result
        n_al = max(agg["aligned"], 1)
        hbm_bytes = agg.get("h2d", 0) + agg.get("d2h", 0) + n_al * 270
        cb_v, cb_g, cb_n, cb_dt = cb
        cpu = {"value": cb_v, "unit": "reads/s", "cores": host_threads, "kind": "port", "gcups": cb_g,
               "sample": f"first {cb_n} reads of the workload; {cpu_kind()}; OpenMP {host_threads} threads, {cb_dt:.1f} s"}
        if scalar:
            cpu["scalar"] = {"value": scalar[0], "unit": "reads/s", "gcups": scalar[1], "cores": host_threads,
                             "sample": f"first {scalar[2]} reads; the scalar oracle (oracle/fade_oracle.c, the parity authority), "
                                       f"OpenMP {host_threads} threads, {scalar[3]:.1f} s"}
        file_leg = file_level_e2e(wl, args.file_reads, host_threads, local_rank) if world == 1 else None
        line = {
            "metric": "annotate_reads_per_sec", "value": value, "unit": "reads/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": wl.scaling, "vs_baseline": None, "dtype": "int16",
            "data": "synthetic", "config": wl.config(),
            "gcups": total_cells / (ms_per_step * 1e-3) / 1e9,
            "aligned_reads_per_step": total_aligned, "artifact_reads_rank0": agg["art"],
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "reads/s", "h2d_bytes_per_step": agg.get("h2d", 0),
                    "d2h_bytes_per_step": agg.get("d2h", 0), "ms_per_step": 1e3 * e_s_max / args.steps,
                    "bytes_per_read": round((agg.get("h2d", 0) + agg.get("d2h", 0)) / max(wl.n, 1), 2),
                    "host_threads_per_rank": host_threads, "path": path,
                    "pass_ms_mean_max_min_per_rank": per_rank,
                    "host_ms_last_pass": {kx: round(v, 3) for kx, v in host_ms.items()}},
            "gpu_launches": agg["launches"] * args.steps,
            "roofline": {"bound": "int_alu", "achieved": achieved, "peak": peak9, "unit": "GCUPS",
                         "frac": achieved / peak9 if peak9 > 0 else None,
                         "peak_9instr": peak9, "peak_own_mix": peak75,
                         "frac_own_mix": achieved / peak75 if peak75 > 0 else None,
                         "fill_only_frac_own_mix": (fill_gcups / peak75) if (fill_gcups and peak75 > 0) else None,
                         "note": "peak / frac: SURVEY 8(d)'s 9 packed INT16x2 instructions per 2 cells; the score-only fill needs 7.5 "
                                 "(LOP3, PRMT, VIADDMNMX.RELU, VIMNMX, VIADD, 2 VIADDMNMX, half a VIMNMX3), so it can exceed that "
                                 "denominator; peak_own_mix / frac_own_mix use 7.5",
                         # dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel (sw_fill_kernel<19>) per
                         # launch, ncu --set full on a 1 M-read chunk of c2 (profiles/): only meaningful for that configuration
                         "traffic": FILL_TRAFFIC if (wl.kind == "c2" and chunk == 1_000_000) else None,
                         "kernel": "dominant: sw_fill_kernel<19>; achieved = cells / time of ALL kernels of the path "
                                   "(binning + fill + traceback rounds + generic)",
                         "fill_only_gcups": fill_gcups,
                         "fill_ms": k_fill, "trace_ms": k_trace, "generic_ms": k_gen,
                         "r_alu_thread_instr_per_s": alu_ops, "peak_source": "measured live (fadegpu_measure_alu_peak)",
                         "hbm": {"algorithmic_gbs": hbm_bytes / (k_ms / args.steps * 1e-3) / 1e9,
                                 "peak_gbs": peak_hbm()}},
            "cpu_baseline": cpu,
            "gen_seconds": wl.gen_s,
        }
        if agg["oversize"]:
            line["oversize_reads"] = agg["oversize"]
        if file_leg:
            line["e2e_file"] = file_leg
        print(json.dumps(line), file=out, flush=True)
    if world > 1:
        dist.destroy_process_group()


FILL_TRAFFIC = 2.455e9   # profiles/r02_prof_fill_raw.csv: 0.160 GB read + 2.295 GB written per launch (ncu --set full)


def peak_hbm():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f).get("hbm_gbs")
    except Exception:
        return 6650.0


if __name__ == "__main__":
    main()
