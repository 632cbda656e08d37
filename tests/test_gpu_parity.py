"""GPU parity tests proper: libfadegpu (through the C ABI) against the oracle, bit-exact.
Run with `pytest -m gpu` on a B200."""
import numpy as np
import pytest

from fade_b200 import Context, default_params, sim
from parity_util import compare, oracle_params, run_gpu

pytestmark = pytest.mark.gpu


def test_c1_config_bit_exact(gpu_ctx):
    """BASELINE.json configs[0]: 1 Mbp reference, 10k simulated 2x150 reads, defaults."""
    names, contigs, cfg, n = sim.config_c1()
    gpu_ctx.load_reference(names, [c.tobytes() for c in contigs])
    rd = sim.make_reads(cfg, 0, n, contigs)
    b = run_gpu(gpu_ctx, rd)
    n_al = compare(b, rd, contigs, oracle_params(gpu_ctx.params))
    assert n_al > 1000
    st = b.stats()
    assert st.n_aligned == n_al and st.kernel_launches >= 2 and st.n_generic == 0
    b.close()


def test_empty_and_no_clip_batches(gpu_ctx):
    names, contigs, cfg, n = sim.config_c1()
    gpu_ctx.load_reference(names, [c.tobytes() for c in contigs])
    rd = sim.make_reads(cfg, 0, 64, contigs)
    b = gpu_ctx.alloc_batch(64, 64 * 75)
    b.run(0)                                     # empty batch
    rd.clip_left[:] = 0
    rd.clip_right[:] = 0
    b.fill(rd.seq4, rd.seq_off, rd.l_qseq, rd.tid, rd.pos, rd.aligned_len, rd.clip_left, rd.clip_right).run()
    assert not b.flags[:64].any() and b.stats().n_aligned == 0
    b.close()


# ---- edge cases -----------------------------------------------------------------------------------
import random  # noqa: E402

import readsets  # noqa: E402
from fade_b200 import api  # noqa: E402
from oracle import oracle as orc  # noqa: E402


def _ctx(**kw):
    return Context(0, default_params(**kw))


def test_ragged_lengths_contig_ends_and_short_clips():
    """query lengths 20..320 (all five packed instantiations + the generic kernel above 304),
    windows clamped at contig starts and ends, clips at / below the length floor, several contigs."""
    rng = random.Random(11)
    contigs = [readsets.random_ref(rng, n) for n in (5000, 1200, 700, 330)]
    reads = readsets.ragged_reads(rng, contigs, 3000, max_len=320)
    rd = readsets.build(reads)
    with _ctx() as ctx:
        ctx.load_reference([f"c{i}" for i in range(4)], contigs)
        b = run_gpu(ctx, rd)
        n_al = compare(b, rd, contigs, oracle_params(ctx.params))
        assert n_al > 500 and 0 < b.stats().n_generic < 200
        b.close()


def test_wildcard_letters_go_through_generic_kernel():
    """IUPAC letters in reads and reference, lower case, N runs: P1 wildcard row/column (score 0,
    '=' by byte equality) -- served by the generic kernel on the device."""
    rng = random.Random(12)
    base = bytearray(readsets.random_ref(rng, 6000))
    for _ in range(40):
        p = rng.randrange(len(base))
        base[p] = ord(rng.choice("RYKMSWBDHVryn"))
    base[3000:3100] = b"N" * 100
    base[1000:1400] = bytes(base[1000:1400]).lower()
    contigs = [bytes(base)]
    reads = readsets.ragged_reads(rng, contigs, 1500, wild_read_rate=0.002, alpha="ACGTN")
    rd = readsets.build(reads)
    with _ctx() as ctx:
        ctx.load_reference(["w"], contigs)
        b = run_gpu(ctx, rd)
        n_al = compare(b, rd, contigs, oracle_params(ctx.params))
        st = b.stats()
        assert n_al > 300
        assert (b.flags[: rd.n] & api.R_GENERIC).any(), "some alignments must have met a wildcard letter"
        b.close()


def test_force_generic_equals_packed():
    names, contigs, cfg, n = sim.config_c1()
    rd = sim.make_reads(cfg, 0, 1500, contigs)
    with _ctx(flags=api.F_FORCE_GENERIC) as ctx:
        ctx.load_reference(names, [c.tobytes() for c in contigs])
        b = run_gpu(ctx, rd)
        n_al = compare(b, rd, contigs, oracle_params(ctx.params))
        assert b.stats().n_generic == n_al > 100
        b.close()


def test_both_kernel_families_against_the_striped_restatement():
    """The generic kernel and the scalar oracle are written alike, so agreeing with each other says little.  Here the
    packed kernels AND the generic kernel are compared with the structurally different restatement of parasail's
    striped lazy-F kernel (oracle/parasail_striped.c, 16 and 8 lanes) on every aligned read of a ragged read set."""
    rng = random.Random(91)
    contigs = [readsets.random_ref(rng, n) for n in (6000, 1500)]
    reads = readsets.ragged_reads(rng, contigs, 700, max_len=200)
    rd = readsets.build(reads)
    for flags in (0, api.F_FORCE_GENERIC):
        with _ctx(flags=flags) as ctx:
            ctx.load_reference(["a", "b"], contigs)
            b = run_gpu(ctx, rd)
            W = ctx.params.window_size
            n_checked = 0
            for k in np.flatnonzero(b.flags[: rd.n] & 1):
                r = reads[k]
                ref = contigs[r["tid"]].decode().upper()
                start = max(0, r["pos"] - W)
                end = min(len(ref), r["pos"] + r["aligned_len"] + W)
                assert int(b.win_start[k]) == start
                q = readsets.revcomp(r["seq"])
                for lanes in (16, 8):
                    s = orc.sw_trace_striped(q, ref[start:end], lanes)
                    assert (s.score, s.n_ops) == (int(b.score[k]), int(b.n_ops[k])), (k, lanes)
                    if s.score > 0:
                        assert (s.end_query, s.end_ref, s.beg_query, s.beg_ref) == \
                            (int(b.end_query[k]), int(b.end_ref[k]), int(b.beg_query[k]), int(b.beg_ref[k])), (k, lanes)
                        assert s.ops[: api.MAX_OPS] == [int(x) for x in b.ops[k, : min(s.n_ops, api.MAX_OPS)]], (k, lanes, s.cigar)
                n_checked += 1
            assert n_checked > 200
            assert (b.stats().n_generic > 0) == bool(flags)
            b.close()


@pytest.mark.parametrize("extra", [0, api.F_FORCE_GENERIC, api.F_HOST_BINNING])
def test_tags_only_skips_hopeless_tracebacks_and_changes_no_tag(extra):
    """FADEGPU_F_TAGS_ONLY: an alignment whose score fails `score > clip_len*0.9*2` (analysis.d:43,76,100) for both
    clips gets no traceback (record: score, FADEGPU_R_SCORE_ONLY); art_left / art_right of every read and the full
    record of every other alignment equal the oracle."""
    names, contigs, cfg, n = sim.config_c1()
    rd = sim.make_reads(cfg, 0, 6000, contigs)
    with _ctx(flags=api.F_TAGS_ONLY | extra) as ctx:
        ctx.load_reference(names, contigs)
        b = run_gpu(ctx, rd)
        res, ops = orc.align_batch(rd.seq4, rd.seq_off, rd.l_qseq, rd.tid, rd.pos, rd.aligned_len, rd.clip_left, rd.clip_right,
                                   contigs, params=oracle_params(ctx.params), ops_cap=api.MAX_OPS)
        fl = b.flags[: rd.n]
        assert np.array_equal((fl & 1).astype(np.int32), res["aligned"])
        assert np.array_equal(((fl >> 1) & 1).astype(np.int32), res["art_left"])
        assert np.array_equal(((fl >> 2) & 1).astype(np.int32), res["art_right"])
        al = res["aligned"] == 1
        so = (fl & api.R_SCORE_ONLY) != 0
        assert 0.15 < so[al].mean() < 0.6 and not so[~al].any()
        assert np.array_equal(b.score[: rd.n][al], res["score"][al])
        # a skipped alignment can indeed not be accepted: 5 * score <= 9 * clip for both clips past the floor
        S, cl, cr = res["score"], rd.clip_left, rd.clip_right
        may = ((cl > 5) & (5 * S > 9 * cl)) | ((cr > 5) & (5 * S > 9 * cr))
        assert np.array_equal(so[al], ~may[al])
        full = al & ~so
        for f in ("beg_query", "end_query", "beg_ref", "end_ref", "n_ops"):
            assert np.array_equal(getattr(b, f)[: rd.n][full], res[f][full]), f
        k = np.minimum(res["n_ops"], api.MAX_OPS)
        m = np.arange(api.MAX_OPS)[None, :] < k[:, None]
        assert np.array_equal(np.where(m, b.ops[: rd.n], 0)[full], np.where(m, ops, 0)[full])
        assert (b.n_ops[: rd.n][al & so] == 0).all()
        b.close()


def test_stress_config_long_windows_short_clips():
    """BASELINE.json configs[3]: --window-size 1000, --min-length 5, 2x250 reads, clip law U{1..40}."""
    ref = sim.make_contig(1002, 0, 400_000, 50_000, 300, 0.02)
    cfg = sim.default_cfg(read_seed=2004, read_len=250, window=1000, frag_mean=600, frag_sd=80, short_clip_law=1)
    rd = sim.make_reads(cfg, 0, 3000, [ref])
    with _ctx(window_size=1000, min_length=5) as ctx:
        ctx.load_reference(["chrS"], [ref.tobytes()])
        b = run_gpu(ctx, rd)
        n_al = compare(b, rd, [ref], oracle_params(ctx.params))
        assert n_al > 300
        b.close()


@pytest.mark.parametrize("min_length,window", [(0, 300), (20, 50), (59, 10), (-1, 300)])
def test_flag_variants(min_length, window):
    """--min-length / --window-size variants, incl. the negative floor that wraps (uint <= int)."""
    names, contigs, cfg, n = sim.config_c1()
    rd = sim.make_reads(cfg, 0, 2500, contigs)
    with _ctx(min_length=min_length, window_size=window) as ctx:
        ctx.load_reference(names, [c.tobytes() for c in contigs])
        b = run_gpu(ctx, rd)
        n_al = compare(b, rd, contigs, oracle_params(ctx.params))
        if min_length < 0:
            assert n_al == 0
        b.close()


def test_other_scoring_plain_trace_path():
    """scoring that does not fit the tagged trace encoding exercises the plain recorder."""
    names, contigs, cfg, n = sim.config_c1()
    rd = sim.make_reads(cfg, 0, 2000, contigs)
    with _ctx(gap_open=12, gap_extend=3, match=9, mismatch=-9) as ctx:
        ctx.load_reference(names, [c.tobytes() for c in contigs])
        b = run_gpu(ctx, rd)
        compare(b, rd, contigs, oracle_params(ctx.params))
        b.close()


def test_small_scratch_forces_many_launches():
    """a tiny checkpoint scratch splits the batch into many fill/trace launch pairs."""
    names, contigs, cfg, n = sim.config_c1()
    rd = sim.make_reads(cfg, 0, 4000, contigs)
    with _ctx(scratch_bytes=4 << 20) as ctx:
        ctx.load_reference(names, [c.tobytes() for c in contigs])
        b = run_gpu(ctx, rd)
        compare(b, rd, contigs, oracle_params(ctx.params))
        assert b.stats().kernel_launches > 6
        b.close()


def test_batch_reuse_and_double_buffering(gpu_ctx):
    names, contigs, cfg, n = sim.config_c1()
    gpu_ctx.load_reference(names, [c.tobytes() for c in contigs])
    bs = [gpu_ctx.alloc_batch(3000, 3000 * 75) for _ in range(2)]
    rds = [sim.make_reads(cfg, k * 3000, 3000 - 7 * k, contigs) for k in range(4)]
    for k, rd in enumerate(rds):            # submit k while k-1 is in flight
        b = bs[k & 1]
        b.fill(rd.seq4, rd.seq_off, rd.l_qseq, rd.tid, rd.pos, rd.aligned_len, rd.clip_left, rd.clip_right)
        b.submit()
        if k:
            bs[(k - 1) & 1].wait()
            compare(bs[(k - 1) & 1], rds[k - 1], contigs, oracle_params(gpu_ctx.params))
    bs[1].wait()
    compare(bs[1], rds[3], contigs, oracle_params(gpu_ctx.params))
    with pytest.raises(Exception):
        bs[0].wait()                         # not in flight -> FADEGPU_E_STATE, loudly
    for b in bs:
        b.close()


def test_record_level_tags_match_oracle(gpu_ctx):
    """rs / am / as / ar / ab of every record (anno.d:94-107) equal the oracle's."""
    from fade_b200 import Record, annotate_records
    names, contigs, cfg, n = sim.config_c1()
    gpu_ctx.load_reference(names, [c.tobytes() for c in contigs])
    rd = sim.make_reads(cfg, 0, 3000, contigs)
    L = rd.read_len
    stride = (L + 1) // 2
    recs = [Record(f"r{k}", int(rd.flag[k]), int(rd.tid[k]), int(rd.pos[k]), rd.cigar[k, : rd.n_cigar[k]].copy(),
                   rd.seq4[k * stride:(k + 1) * stride].copy(), rd.qual[k * L:(k + 1) * L].copy(), L,
                   bool(rd.has_sa[k])) for k in range(rd.n)]
    annotate_records(gpu_ctx, recs)
    n_art = 0
    refb = contigs[0].tobytes()
    for rec in recs:
        exp = orc.annotate_record(is_mapped=not (rec.flag & 4), has_sa=rec.has_sa, cigar=rec.cigar, seq4=rec.seq4,
                                  qual=rec.qual, l_qseq=rec.l_qseq, pos=rec.pos, contig_name=names[rec.tid],
                                  ref_seq=refb)
        assert rec.tags == exp, (rec.qname, rec.tags, exp)
        n_art += "am" in exp
    assert n_art > 100


def test_submit_inputs_from_caller_arrays(gpu_ctx):
    """fadegpu_submit_inputs on pageable caller arrays with absolute seq offsets == fadegpu_submit."""
    names, contigs, cfg, n = sim.config_c1()
    gpu_ctx.load_reference(names, [c.tobytes() for c in contigs])
    rd = sim.make_reads(cfg, 0, 6000, contigs)
    b = gpu_ctx.alloc_batch(2000, 2000 * 75)
    for a in (0, 2000, 4000):
        b.submit_arrays(2000, rd.seq4, rd.seq_off[a:], rd.l_qseq[a:], rd.tid[a:], rd.pos[a:], rd.aligned_len[a:],
                        rd.clip_left[a:], rd.clip_right[a:])
        b.wait()
        sub = sim.make_reads(cfg, a, 2000, contigs)
        compare(b, sub, contigs, oracle_params(gpu_ctx.params))
    b.close()


def test_compact_results_and_no_scatter():
    """fadegpu_get_results (compact records + per-read index) carries the same data as the per-read
    arrays; with FADEGPU_F_NO_SCATTER only flags[] and the compact results are filled."""
    names, contigs, cfg, n = sim.config_c1()
    rd = sim.make_reads(cfg, 0, 4000, contigs)
    with _ctx() as ctx:
        ctx.load_reference(names, [c.tobytes() for c in contigs])
        b = run_gpu(ctx, rd)
        compare(b, rd, contigs, oracle_params(ctx.params))
        rec, ws, ridx = b.results()
        al = np.where(b.flags[: rd.n] & 1)[0]
        assert len(rec) == len(al) == b.stats().n_aligned
        assert np.array_equal(np.sort(rec["read"]), al) and np.array_equal(np.where(ridx >= 0)[0], al)
        k = ridx[al]
        assert np.array_equal(rec["read"][k], al)
        for f in ("score", "beg_query", "end_query", "beg_ref", "end_ref", "n_ops"):
            assert np.array_equal(rec[f][k], getattr(b, f)[al]), f
        assert np.array_equal(ws[k], b.win_start[al]) and np.array_equal(rec["ops"][k], b.ops[al])
        assert np.array_equal(rec["flags"][k] & 0xff, b.flags[al])
        ref_flags = b.flags[: rd.n].copy()
        ref_rec = rec.copy()
        b.close()
    with _ctx(flags=api.F_NO_SCATTER) as ctx:
        ctx.load_reference(names, [c.tobytes() for c in contigs])
        b = ctx.alloc_batch(rd.n, int(rd.seq_off[rd.n]))
        assert b.score is None and b.ops is None          # the per-read arrays are not even allocated
        b.fill(rd.seq4, rd.seq_off, rd.l_qseq, rd.tid, rd.pos, rd.aligned_len, rd.clip_left, rd.clip_right).run()
        rec2, ws2, ridx2 = b.results()
        assert np.array_equal(b.flags[: rd.n], ref_flags)
        o1, o2 = np.argsort(ref_rec["read"]), np.argsort(rec2["read"])
        assert np.array_equal(ref_rec[o1], rec2[o2])
        b.close()


def test_no_shortcut_flag_gives_identical_results():
    """the ungapped-diagonal proof of the traceback is an optimisation only: with it disabled every
    block on the path is replayed and the records must be identical."""
    names, contigs, cfg, n = sim.config_c1()
    rd = sim.make_reads(cfg, 0, 6000, contigs)
    recs = []
    for fl in (0, api.F_NO_SHORTCUT):
        with _ctx(flags=fl) as ctx:
            ctx.load_reference(names, [c.tobytes() for c in contigs])
            b = run_gpu(ctx, rd)
            compare(b, rd, contigs, oracle_params(ctx.params))
            rec, ws, ridx = b.results()
            recs.append(rec[np.argsort(rec["read"])].copy())
            b.close()
    assert np.array_equal(recs[0], recs[1])


def test_share_reference_and_concurrent_contexts():
    """fadegpu_share_reference (device-to-device copy of the packed reference) and two contexts
    driven concurrently from two host threads (the C ABI's threading contract)."""
    import threading
    names, contigs, cfg, n = sim.config_c1()
    rds = [sim.make_reads(cfg, k * 5000, 5000, contigs) for k in range(2)]
    src = Context(0)
    src.load_reference(names, [c.tobytes() for c in contigs])
    dst = Context(0)
    dst.share_reference_from(src)
    assert dst.reference_info() == src.reference_info()
    errs = []

    def work(ctx, rd):
        try:
            for _ in range(3):
                b = run_gpu(ctx, rd)
                compare(b, rd, contigs, oracle_params(ctx.params))
                b.close()
        except Exception as e:  # noqa: BLE001
            errs.append(e)

    ts = [threading.Thread(target=work, args=(c, r)) for c, r in zip((src, dst), rds)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    src.close()
    dst.close()
    assert not errs, errs


def test_long_windows_use_generic_kernel_and_absurd_ones_are_reported():
    """spliced-style records (huge aligned_len): windows of thousands of columns stay on the packed kernels, those
    beyond a million columns go to the generic kernel on the device; a window of > 2^31 DP cells leaves THAT read unaligned with
    FADEGPU_R_OVERSIZE (counted in the stats) and the rest of the batch is served as usual."""
    rng = random.Random(31)
    contigs = [readsets.random_ref(rng, 60_000)]
    reads = readsets.ragged_reads(rng, contigs, 40, min_len=100, max_len=150)
    for r in reads[:20]:
        r["aligned_len"] = rng.randint(5_000, 12_000)      # an N-spanning CIGAR
        r["pos"] = rng.randint(0, 40_000)
    rd = readsets.build(reads)
    for flags in (0, api.F_HOST_BINNING):
        with _ctx(flags=flags) as ctx:
            ctx.load_reference(["c"], contigs)
            b = run_gpu(ctx, rd)
            compare(b, rd, contigs, oracle_params(ctx.params))
            assert b.stats().n_generic == 0      # the packed kernels restage the target chunk by chunk (1024 steps at a time)
            b.close()
    # windows beyond the packed kernels' million columns: the generic kernel on the device
    huge = [readsets.random_ref(rng, 1_300_000)]
    far = [dict(seq="".join(rng.choice("ACGT") for _ in range(60)), tid=0, pos=1000 + 50 * k, aligned_len=1_100_000 + 1000 * k,
                clip_left=10 + k, clip_right=0) for k in range(2)]
    near = readsets.ragged_reads(rng, huge, 30, min_len=100, max_len=150)
    rd3 = readsets.build(near[:15] + far + near[15:])
    with _ctx() as ctx:
        ctx.load_reference(["h"], huge)
        b = run_gpu(ctx, rd3)
        compare(b, rd3, huge, oracle_params(ctx.params))
        assert b.stats().n_generic == 2
        b.close()
    big = [bytes(40_000_000)]
    rnd = random.Random(32)
    small = [dict(seq="".join(rnd.choice("ACGT") for _ in range(120)), tid=0, pos=5000 + 10 * k, aligned_len=100, clip_left=20, clip_right=0)
             for k in range(30)]
    absurd = dict(seq="ACGT" * 30, tid=0, pos=100, aligned_len=39_000_000, clip_left=20, clip_right=0)
    rd2 = readsets.build(small[:10] + [absurd] + small[10:])
    for flags in (0, api.F_HOST_BINNING):
        with _ctx(flags=flags) as ctx:
            ctx.load_reference(["z"], big)
            b = ctx.alloc_batch(rd2.n, int(rd2.seq_off[rd2.n]))
            for path in ("view", "compact"):
                if path == "view":
                    b.fill(rd2.seq4, rd2.seq_off, rd2.l_qseq, rd2.tid, rd2.pos, rd2.aligned_len, rd2.clip_left, rd2.clip_right).run()
                else:
                    b.fill_compact(rd2.seq4, rd2.seq_off, rd2.l_qseq, rd2.tid, rd2.pos, rd2.aligned_len, rd2.clip_left, rd2.clip_right)
                    b.submit_compact()
                    b.wait()
                st = b.stats()
                assert st.n_oversize == 1 and st.n_aligned == 30
                assert b.flags[10] == api.R_OVERSIZE and (b.flags[:10] & 1).all() and (b.flags[11:31] & 1).all()
            b.close()


def test_compact_inputs_equal_view_inputs_and_oracle():
    """fadegpu_submit_compact (one gate byte per read uploaded, the 32-byte records and the bases of the reads
    past the length floor fetched by the GPU) against fadegpu_submit and the oracle: ragged lengths, several
    contigs, clips at / below / far above the floor (gate saturation at 255), several floors."""
    rng = random.Random(43)
    contigs = [readsets.random_ref(rng, n) for n in (9000, 2500, 600)]
    reads = readsets.ragged_reads(rng, contigs, 4000, max_len=320)
    for r in reads[:60]:          # clips beyond the gate's 8 bits
        r["clip_left"] = rng.choice([254, 255, 256, 300])
    rd = readsets.build(reads)
    for min_length in (5, 0, 254, 255, 290, -1):
        with _ctx(min_length=min_length) as ctx:
            ctx.load_reference(["a", "b", "c"], contigs)
            b = run_gpu(ctx, rd)
            rec1 = b.results()[0]
            rec1 = rec1[np.argsort(rec1["read"])].copy()
            fl1 = b.flags[: rd.n].copy()
            h2d_view = b.stats().h2d_bytes
            b.fill_compact(rd.seq4, rd.seq_off, rd.l_qseq, rd.tid, rd.pos, rd.aligned_len, rd.clip_left, rd.clip_right)
            b.submit_compact()
            b.wait()
            n_al = compare(b, rd, contigs, oracle_params(ctx.params))
            rec2 = b.results()[0]
            assert np.array_equal(rec1, rec2[np.argsort(rec2["read"])]) and np.array_equal(fl1, b.flags[: rd.n])
            st = b.stats()
            assert st.n_aligned == n_al
            if min_length == 5:
                assert n_al > 800 and st.h2d_bytes < h2d_view - 14 * rd.n      # half of the reads here pass the floor
            if min_length == -1:
                assert n_al == 0      # the floor compare is unsigned (analysis.d:34)
            ms = b.replay_kernels(1)  # replays run from the device mirrors of the fetched records
            assert ms > 0
            b.submit_compact()
            b.wait()
            rec3 = b.results()[0]
            assert np.array_equal(rec1, rec3[np.argsort(rec3["read"])])
            b.close()


@pytest.mark.parametrize("flags", [0, api.F_HOST_BINNING, api.F_SYNC_SUBMIT])
def test_device_and_host_binning_agree(flags):
    """By default the host only gathers the reads past the length floor and the device bins them, queued
    on the ctx thread; FADEGPU_F_SYNC_SUBMIT does that on the calling thread, FADEGPU_F_HOST_BINNING bins
    on the host.  Same records every way (ragged lengths, several contigs), from the view and from arrays, and
    the same plan as the default flags (every binning feeds one planner)."""
    rng = random.Random(41)
    contigs = [readsets.random_ref(rng, n) for n in (9000, 2500, 600)]
    rd = readsets.build(readsets.ragged_reads(rng, contigs, 4000, max_len=320))

    def plan_of(st):
        return st.n_aligned, st.n_generic, st.cells, st.scratch_bytes

    with _ctx() as ctx:
        ctx.load_reference(["a", "b", "c"], contigs)
        b = run_gpu(ctx, rd)
        want = plan_of(b.stats())
        b.close()
    with _ctx(flags=flags) as ctx:
        ctx.load_reference(["a", "b", "c"], contigs)
        b = run_gpu(ctx, rd)                       # fadegpu_submit (pinned view)
        compare(b, rd, contigs, oracle_params(ctx.params))
        st = b.stats()
        assert st.n_aligned > 800 and st.n_generic > 0
        assert plan_of(st) == want
        rec1 = b.results()[0]
        rec1 = rec1[np.argsort(rec1["read"])].copy()
        b.submit_arrays(rd.n, rd.seq4, rd.seq_off, rd.l_qseq, rd.tid, rd.pos, rd.aligned_len, rd.clip_left, rd.clip_right)
        b.wait()                                   # fadegpu_submit_inputs (caller-owned arrays)
        assert plan_of(b.stats()) == want
        rec2 = b.results()[0]
        assert np.array_equal(rec1, rec2[np.argsort(rec2["read"])])
        b.run(0)                                   # empty batch through the device path
        assert b.stats().n_aligned == 0
        b.close()


def test_many_batches_in_flight_and_replay_batches():
    """Asynchronous submits: six batches queued before the first wait (uploads, binning, fills and the
    traceback rounds of neighbouring batches overlap on the ctx's streams and its two scratch sets);
    every one equals the oracle.  fadegpu_replay_batches then re-runs only the kernels of all of them and
    leaves the results untouched."""
    rng = random.Random(77)
    contigs = [readsets.random_ref(rng, n) for n in (20000, 3000)]
    rds = [readsets.build(readsets.ragged_reads(random.Random(300 + k), contigs, 1500 + 200 * k, max_len=300)) for k in range(6)]
    with _ctx() as ctx:
        ctx.load_reference(["a", "b"], contigs)
        bs = [ctx.alloc_batch(r.n, int(r.seq_off[r.n])) for r in rds]
        for b, r in zip(bs, rds):
            b.fill(r.seq4, r.seq_off, r.l_qseq, r.tid, r.pos, r.aligned_len, r.clip_left, r.clip_right)
            b.submit()
        for b in bs:
            b.wait()
        for b, r in zip(bs, rds):
            compare(b, r, contigs, oracle_params(ctx.params))
        def by_read(b):                                      # the order of the records within a window length is unspecified
            rec = b.results()[0]
            return rec[np.argsort(rec["read"])].copy()
        before = [by_read(b) for b in bs]
        ms = ctx.replay_batches(bs, 2)
        assert ms > 0
        ms1 = sum(b.replay_kernels(1) for b in bs)
        assert ms1 > 0
        for b, r, rec in zip(bs, rds, before):
            b.run()                                          # fresh D2H of what the kernels left in HBM
            assert np.array_equal(by_read(b), rec)
        for b in bs:
            b.close()


def test_errors_of_a_queued_submit_surface_at_wait():
    """inconsistent seq_off, through fadegpu_submit (view), fadegpu_submit_compact and fadegpu_submit_inputs
    (arrays): FADEGPU_E_ARG from fadegpu_wait when the check runs in a queued submit, from the submit call itself
    with FADEGPU_F_SYNC_SUBMIT or FADEGPU_F_HOST_BINNING and for arrays (checked while they are gathered, on the
    calling thread); the batch and the ctx stay usable afterwards."""
    rng = random.Random(5)
    contigs = [readsets.random_ref(rng, 4000)]
    rd = readsets.build(readsets.ragged_reads(rng, contigs, 200, max_len=150))
    k = int(np.flatnonzero(rd.clip_left > 10)[0])
    bad_off = rd.seq_off.copy()
    bad_off[k] = int(rd.seq_off[rd.n]) + 5                   # points past the end of seq4
    fields = (rd.seq4, rd.seq_off, rd.l_qseq, rd.tid, rd.pos, rd.aligned_len, rd.clip_left, rd.clip_right)

    def submit(b, entry, seq_off):
        if entry == "view":
            b.fill(*fields)
            b.seq_off[:rd.n + 1] = seq_off
            b.submit()
        elif entry == "compact":
            b.fill_compact(*fields)
            b.meta["seq_off"][:rd.n] = seq_off[:rd.n]
            b.submit_compact()
        else:
            b.submit_arrays(rd.n, rd.seq4, seq_off, *fields[2:])

    for flags in (0, api.F_SYNC_SUBMIT, api.F_HOST_BINNING):
        with _ctx(flags=flags) as ctx:
            ctx.load_reference(["a"], contigs)
            b = ctx.alloc_batch(rd.n, int(rd.seq_off[rd.n]))
            for entry in ("view", "compact", "arrays"):
                if flags == 0 and entry != "arrays":
                    submit(b, entry, bad_off)
                    with pytest.raises(api.FadeGpuError) as e:
                        b.wait()
                else:
                    with pytest.raises(api.FadeGpuError) as e:
                        submit(b, entry, bad_off)
                assert e.value.code == -1 and "seq_off" in str(e.value), (flags, entry)   # FADEGPU_E_ARG
                submit(b, entry, rd.seq_off)
                b.wait()
                compare(b, rd, contigs, oracle_params(ctx.params))
            b.close()
