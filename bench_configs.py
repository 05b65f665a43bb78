#!/usr/bin/env python3
"""Measurements of the BASELINE.json configurations that `bench.py` does not time
(bench.py = configs[1], the one the headline metric is quoted on):

    python bench_configs.py build      configs[2]: motif --build, 750 motifs x 1e6 background samples
    python bench_configs.py genome     configs[3]: genome-wide scan, one GPU's share (1/8 of 3.1 Gbp)
    python bench_configs.py enrich     configs[4]: 200k target + 200k control 1 kb regions, 1900 motifs
    python bench_configs.py whole-genome --genome-scale 1 --gpus 8
                                       configs[3] genome with de-duplication (scan --whole-genome), tables and BED
    python bench_configs.py variants --genome-scale 0.1 --alleles 4000000 [--indel-fraction 0.15]
    python bench_configs.py haplotypes --genome-scale 0.1 --alleles 400000 --samples 16 [--indel-fraction 0.15]
                                       motifscan variant: SNVs / MNVs (and with --indel-fraction that share of
                                       deletions and insertions, scanned with --indels) of a seeded VCF against
                                       the resident genome

Each prints one JSON line: device-resident and end-to-end time, throughput, and a parity check of a
bounded sample against the reference's CPU implementation (oracle/_ref when it compiled, else the
oracle port).  Synthetic inputs (motifscan_b200/synth.py), nothing is read from /root/reference.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def cpu_ext():
    import oracle
    ref = oracle.load_reference_cscore()
    return ("reference", ref) if ref is not None else ("port", oracle)


def device_ms(ctx, *names):
    t = ctx.timings()
    return {k: t[k] for k in names}


def strs(blob, off, idx):
    raw = blob.tobytes()
    return [raw[off[i]:off[i + 1]].decode() for i in idx]


def bench_build(args):
    """cli/motif.py:119-153 at --n-random 1e6: score every sample at offset 0 on both strands, keep the
    order statistics for p = 1e-2 .. 1e-6."""
    from motifscan_b200 import engine, synth
    from motifscan_b200.motif import cutoff_ranks
    ctx = engine.default_context(0)
    _, pwms, _ = synth.motif_set(args.motifs, seed=2020)
    lmax = max(p.shape[1] for p in pwms)
    motifs = engine.MotifSet(ctx, pwms)
    blob, off = synth.background_samples(args.n_random, lmax, seed=1)
    ranks = cutoff_ranks(args.n_random)
    keys = list(ranks)
    times = []
    for _ in range(args.steps + 1):
        t0 = time.perf_counter()
        sset = engine.SequenceSet(ctx, blob=blob, seq_off=off)
        sel = engine.score_select(ctx, motifs, sset, 3, [ranks[k] for k in keys])
        times.append(time.perf_counter() - t0)
        dev = device_ms(ctx, "score", "select")
        sset.close()
    e2e = min(times[1:])
    counters = ctx.counters()
    # the plain form (every sample scored for every motif, select over the full rows) for comparison
    ctx.set_option("select_pilot", 0)
    sset = engine.SequenceSet(ctx, blob=blob, seq_off=off)
    t0 = time.perf_counter()
    plain = engine.score_select(ctx, motifs, sset, 3, [ranks[k] for k in keys])
    plain_s = time.perf_counter() - t0
    plain_dev = device_ms(ctx, "score", "select")
    sset.close()
    ctx.set_option("select_pilot", 1)
    same_as_plain = bool(np.array_equal(sel.view(np.uint64), plain.view(np.uint64)))
    # the real sampler in front (genome/__init__.py:159-176: legacy-numpy RNG on the host, N counts and window
    # extraction on the device out of a resident genome): `motif --build`'s whole step per repeat
    import bench
    from motifscan_b200.genome import DeviceGenome
    pg = bench.make_genome(0, 0.1)
    dg = DeviceGenome(pg, ctx)
    sampler = []
    for _ in range(3):
        t0 = time.perf_counter()
        sset = dg.random_sequence_set(args.n_random, lmax, 0, 1)
        t1 = time.perf_counter()
        engine.score_select(ctx, motifs, sset, 3, [ranks[k] for k in keys])
        t2 = time.perf_counter()
        sset.close()
        sampler.append((t2 - t0, t1 - t0))
    dg.close()
    with_sampler_s, sampler_s = min(sampler)
    # parity on a bounded sample: the same pipeline on the first n samples vs the CPU reference
    kind, ext = cpu_ext()
    n = args.cpu_samples
    sub_ranks = cutoff_ranks(n)
    sset = engine.SequenceSet(ctx, blob=blob[:off[n]], seq_off=off[:n + 1])
    got = engine.score_select(ctx, motifs, sset, 3, list(sub_ranks.values()))
    sset.close()
    t0 = time.perf_counter()
    scores = ext.c_score([p.tolist() for p in pwms], strs(blob, off, range(n)), 3, os.cpu_count() or 1)
    want = np.array([[sorted(row, reverse=True)[r] for r in sub_ranks.values()] for row in scores])
    cpu_s = time.perf_counter() - t0
    same = bool(np.array_equal(got.view(np.uint64), want.view(np.uint64)))
    units = args.motifs * args.n_random
    return {"config": f"configs[2]: motif --build cutoffs, {args.motifs} motifs x {args.n_random} samples x {lmax} bp, "
                      f"p=1e-2..1e-{len(keys) + 1}",
            "metric": "motif*samples scored and ranked per second", "e2e_s": e2e,
            "value": units / e2e, "device_ms": dev, "device_ms_total": dev["score"] + dev["select"],
            "candidate_sites": counters["hits"], "motifs_redone_the_plain_way": counters["retries"],
            "with_real_sampler": {"e2e_s": with_sampler_s, "sampler_s": sampler_s,
                                  "note": "DeviceGenome.random_sequence_set(n_random) on a 310 Mbp synthetic genome (7 % N: the rejected "
                                          "attempts are re-drawn with the reference's RNG sequence) + msb_score_select"},
            "plain_form": {"e2e_s": plain_s, "device_ms": plain_dev, "same_bits_as_pilot_form": same_as_plain},
            "cutoffs_p1e-4_head": np.around(sel[:3, keys.index("1e-4")], 8).tolist(),
            "cpu_baseline": {"kind": kind, "cores": os.cpu_count(), "sample": f"{n} samples (c_score + sort)",
                             "value": args.motifs * n / cpu_s, "seconds": cpu_s},
            "parity": {"order_statistics_bit_identical_on_sample": same}}


def bench_genome_sharded(args):
    """configs[3] over several GPUs of one box (SURVEY 8e): launched under torchrun, one process per
    GPU; every rank keeps the whole packed genome (world x genome_bp, 0.375 B/bp) in HBM and scans the
    position ranges dealt to it round-robin; no exchange step, only a barrier on both sides of the
    timed region and a max over ranks (gloo: NCCL is not on this path).  Weak scaling: genome_bp per
    GPU is fixed."""
    import torch.distributed as dist
    from motifscan_b200 import engine, synth
    from motifscan_b200.genome import DeviceGenome
    from motifscan_b200.genome_scan import scan_genome_resident
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    dist.init_process_group("gloo")
    ctx = engine.default_context(local)
    _, pwms, _ = synth.motif_set(args.motifs, seed=2020)
    motifs = engine.MotifSet(ctx, pwms)
    lmax = max(p.shape[1] for p in pwms)
    bblob, boff = synth.background_samples(100000, lmax, seed=1)
    bg = engine.SequenceSet(ctx, blob=bblob, seq_off=boff)
    cutoffs = np.maximum(np.around(engine.score_select(ctx, motifs, bg, 3, [int(100000 * 1e-4) - 1])[:, 0], 8), 1e-6)
    bg.close()
    motifs.set_cutoffs(cutoffs)
    n = args.genome_bp
    by_chrom = {}
    for c in range(world):                      # one synthetic chromosome of genome_bp per GPU, the same on every rank
        seq = synth.genome_chunk(n, seed=19 + c, n_block=(n // 3, int(n * 0.07)))
        seq[:10000] = ord("N")
        by_chrom[f"chr{c + 1:02d}"] = seq

    class Synthetic:
        pass

    Synthetic.chroms = sorted(by_chrom)
    Synthetic.chrom_sizes = {c: n for c in by_chrom}
    Synthetic.fetch_bytes = staticmethod(lambda chrom, a, b: by_chrom[chrom][a:b].tobytes())

    dg = DeviceGenome(Synthetic, ctx)
    times, counts = [], None
    for _ in range(args.steps + 1):
        dist.barrier()
        t0 = time.perf_counter()
        out = scan_genome_resident(dg, pwms, chunk_bp=args.chunk_bp, batch_bp=args.batch_bp, world=world, rank=rank,
                                   collect_sites=False, motifs=motifs)
        ctx.sync()
        dt = torch_max(dist, time.perf_counter() - t0)
        times.append(dt)
        counts = out.counts
    import torch
    total = torch.from_numpy(counts.copy())
    dist.all_reduce(total)                      # the final gather of the per-motif counts
    best = min(times[1:])
    if rank == 0:
        print(json.dumps({"config": f"configs[3] sharded: {world} GPUs x {n} bp x {args.motifs} motifs, both strands, resident genome, "
                                    f"ranges of {args.chunk_bp} bp round-robin", "n_gpus": world, "e2e_s": best,
                          "value": world * n * args.motifs / best, "metric": "motif*bp/s (aggregate, counts only)",
                          "sites": int(total.sum()), "scaling": "weak"}))
    dist.barrier()
    dist.destroy_process_group()
    return None


def torch_max(dist, x):
    import torch
    t = torch.tensor([x], dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t[0])


def bench_genome(args):
    """One GPU's share of the hg19-shaped genome (3.1 Gbp / 8): chunked counts-only scan."""
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        return bench_genome_sharded(args)
    from motifscan_b200 import engine, synth
    from motifscan_b200.genome_scan import scan_genome
    ctx = engine.default_context(0)
    _, pwms, _ = synth.motif_set(args.motifs, seed=2020)
    motifs = engine.MotifSet(ctx, pwms)
    lmax = max(p.shape[1] for p in pwms)
    bblob, boff = synth.background_samples(100000, lmax, seed=1)
    bg = engine.SequenceSet(ctx, blob=bblob, seq_off=boff)
    cutoffs = np.around(engine.score_select(ctx, motifs, bg, 3, [int(100000 * 1e-4) - 1])[:, 0], 8)
    bg.close(), motifs.close()
    n = args.genome_bp
    t0 = time.perf_counter()
    seq = synth.genome_chunk(n, seed=19, n_block=(n // 3, int(n * 0.07)))   # ~7 % N like the assembly gaps
    seq[:10000] = ord("N")
    gen_s = time.perf_counter() - t0

    class OneChrom:
        chroms = ["chrS"]
        chrom_sizes = {"chrS": n}

        @staticmethod
        def fetch_bytes(chrom, a, b):
            return seq[a:b].tobytes()

    # 51 of the 750 synthetic motifs get a NEGATIVE p=1e-4 cutoff on an iid background (long, very
    # specific columns: even the best of 1e5 random windows scores below 0).  By the reference's rule
    # (N adds 0, cscore.c:346) every all-N window then scores 0 >= cutoff and is a site: 27 M gap
    # positions x 51 motifs x 2 strands.  Motif sets built on real genomes have positive cutoffs, so
    # the headline run floors the cutoffs at 1e-6; the as-built run is reported beside it.
    from motifscan_b200.genome import DeviceGenome
    from motifscan_b200.genome_scan import scan_genome_resident
    t0 = time.perf_counter()
    dg = DeviceGenome(OneChrom, ctx)          # one-time: ASCII H2D + encode to 0.375 B/bp, stays in HBM
    load_s = time.perf_counter() - t0
    load_ms = device_ms(ctx, "h2d", "encode")

    t0 = time.perf_counter()
    mset = engine.MotifSet(ctx, pwms, cutoffs)        # one-time per motif set (prefilter tables are built on first scan)
    motifs_s = time.perf_counter() - t0

    def timed(cut, collect=False):
        runs = []
        mset.set_cutoffs(cut)
        for _ in range(args.steps + 1):
            stats = {}
            t0 = time.perf_counter()
            out = scan_genome_resident(dg, pwms, chunk_bp=args.chunk_bp, batch_bp=args.batch_bp,
                                       collect_sites=collect, stats=stats, motifs=mset)
            runs.append((time.perf_counter() - t0, stats))
        best = min(runs[1:], key=lambda r: r[0])
        return best[0], out, best[1]
    as_built_s, as_built, _ = timed(cutoffs)
    n_nonpos = int((cutoffs <= 1e-10).sum())
    cutoffs = np.maximum(cutoffs, 1e-6)
    e2e, sites, dev = timed(cutoffs)
    sites_s, with_sites, _ = timed(cutoffs, collect=True)
    n_collected = len(with_sites)
    del with_sites
    # the streamed path (host ASCII chunks with overlaps through PCIe every scan), one run for comparison
    t0 = time.perf_counter()
    streamed = scan_genome(OneChrom, pwms, cutoffs=cutoffs, chunk_bp=args.chunk_bp, batch_bp=1 << 27,
                           ctx=ctx, collect_sites=False, resident=False)
    streamed_s = time.perf_counter() - t0
    assert np.array_equal(streamed.counts, sites.counts)
    mset.close()
    dg.close()
    # parity: a 2 Mbp window with sites, vs the CPU reference
    kind, ext = cpu_ext()
    a = n // 3 - 1000000
    piece = seq[a:a + args.cpu_bp]

    class Piece:
        chroms = ["chrS"]
        chrom_sizes = {"chrS": len(piece)}

        @staticmethod
        def fetch_bytes(chrom, x, y):
            return piece[x:y].tobytes()

    got = scan_genome(Piece, pwms, cutoffs=cutoffs, chunk_bp=1 << 18, batch_bp=1 << 20, ctx=ctx)
    t0 = time.perf_counter()
    ref = ext.c_scan_motif([p.tolist() for p in pwms], cutoffs.tolist(), [piece.tobytes().decode()], 3, os.cpu_count() or 1)
    cpu_s = time.perf_counter() - t0
    ok = all(len(r) == c for r, c in zip(ref, got.counts))
    flat = [s for r in ref for s in r]
    ok = ok and np.array_equal(got.start, np.array([s[1] for s in flat], dtype=np.int64)) and \
        np.array_equal(got.score.view(np.uint64), np.array([s[2] for s in flat]).view(np.uint64)) and \
        np.array_equal(got.strand, np.array([s[3] for s in flat], dtype=np.int8))
    pwm_lens = np.array([p.shape[1] for p in pwms], dtype=np.int64)
    adds = 2.0 * float((np.maximum(n - pwm_lens + 1, 0) * pwm_lens).sum())       # SURVEY 8d OPS
    pre_s = dev.get("prefilter", 0.0) / 1e3
    return {"config": f"configs[3]: genome-wide scan, one GPU's share: {n} bp (7 % N, soft-masked) x {args.motifs} motifs, "
                      f"both strands, p=1e-4, resident genome, ranges of {args.chunk_bp} bp in batches of {args.batch_bp} bp",
            "metric": "motif*bp/s (resident packed genome, per-motif counts out)", "e2e_s": e2e, "value": args.motifs * n / e2e,
            "sites": int(sites.counts.sum()), "host_generation_s": gen_s,
            "genome_load": {"seconds": load_s, "device_ms": load_ms, "note": "one-time: host ASCII -> HBM, 2-bit + mask"},
            "motif_set_create_s": motifs_s,
            "with_sites": {"e2e_s": sites_s, "value": args.motifs * n / sites_s, "sites_copied": n_collected,
                           "note": "all site arrays copied to the host and merged motif-major"},
            "streamed": {"e2e_s": streamed_s, "value": args.motifs * n / streamed_s,
                         "note": "resident=False: ASCII chunks with overlaps through PCIe (the r1_b path), counts only"},
            "device_ms": dev,
            "prefilter_roofline": {"algorithmic_flops": 8.0 * adds, "tflops": 8.0 * adds / max(pre_s, 1e-9) / 1e12,
                                   "note": "8 x OPS (unpadded one-hot contraction, 2 flop per MAC) / summed prefilter "
                                           "event time; N windows are skipped, so this counts work not done as done "
                                           "for the 7 % of gap positions"},
            "cutoffs": f"p=1e-4 from 1e5 background samples, floored at 1e-6 ({n_nonpos} motifs had a cutoff <= 0)",
            "as_built_cutoffs": {"e2e_s": as_built_s, "value": args.motifs * n / as_built_s,
                                 "sites": int(as_built.counts.sum()),
                                 "note": "all-N windows are sites for the motifs with a non-positive cutoff"},
            "cpu_baseline": {"kind": kind, "cores": os.cpu_count(), "sample": f"{len(piece)} bp x all motifs",
                             "value": args.motifs * len(piece) / cpu_s, "seconds": cpu_s},
            "parity": {"sites_compared": len(flat), "identical": bool(ok)}}


def bench_enrich(args):
    """Scan target and control regions, count regions with a site per motif, Fisher tests."""
    from motifscan_b200 import engine, synth
    from motifscan_b200.scanner import MotifSites
    from motifscan_b200.stats import enrichment_from_counts
    ctx = engine.default_context(0)
    _, pwms, ids = synth.motif_set(args.motifs, seed=2020, n_long=20)     # 20 motifs of 33-40 columns: longer than the prefilter's 32
    motifs = engine.MotifSet(ctx, pwms)
    lmax = max(p.shape[1] for p in pwms)
    bblob, boff = synth.background_samples(100000, lmax, seed=1)
    bg = engine.SequenceSet(ctx, blob=bblob, seq_off=boff)
    cutoffs = np.around(engine.score_select(ctx, motifs, bg, 3, [int(100000 * 1e-4) - 1])[:, 0], 8)
    bg.close()
    motifs.set_cutoffs(cutoffs)
    pinned = []
    sets = []
    for seed in (200, 201):   # the region sequences sit in pinned host memory, as a loader would leave them
        blob, off = synth.peak_set(args.regions, 1000, seed=seed)
        pin = engine.PinnedArray(blob.size)
        pin.array[:] = blob
        sets.append((pin.array, off))
        pinned.append(pin)
    lengths = [p.shape[1] for p in pwms]

    def scan_hits(blob, off):
        """Regions with >= 1 site per motif; the regions go through in blocks that bound the site buffers."""
        hits = np.zeros(args.motifs, dtype=np.int64)
        n_sites = 0
        step = args.region_block
        for a in range(0, args.regions, step):
            b = min(args.regions, a + step)
            # only what the enrichment test needs leaves the device: per motif, the regions with a site
            sset = engine.SequenceSet(ctx, blob=blob[off[a]:off[b]], seq_off=off[a:b + 1] - off[a])
            n_sites += engine.scan_device(ctx, motifs, sset, 3, remove_dup=True)
            hits += ctx.region_counts(args.motifs)
            sset.close()
        return hits, n_sites

    runs = []
    for _ in range(args.steps + 1):
        t0 = time.perf_counter()
        (h_in, s_in), (h_ctl, s_ctl) = scan_hits(*sets[0]), scan_hits(*sets[1])
        t_scan = time.perf_counter() - t0
        results = enrichment_from_counts(ids, h_in, args.regions, h_ctl, args.regions)
        runs.append((time.perf_counter() - t0, t_scan))
    e2e, t_scan = min(runs[1:])
    # parity of the counts on a bounded sample of regions vs the CPU reference (dedup never empties a cell)
    kind, ext = cpu_ext()
    n = args.cpu_regions
    blob, off = sets[0]
    t0 = time.perf_counter()
    ref = ext.c_scan_motif([p.tolist() for p in pwms], cutoffs.tolist(), strs(blob, off, range(n)), 3, os.cpu_count() or 1)
    cpu_s = time.perf_counter() - t0
    want = np.array([len({s[0] for s in r}) for r in ref], dtype=np.int64)
    sset = engine.SequenceSet(ctx, blob=blob[:off[n]], seq_off=off[:n + 1])
    res = engine.scan(ctx, motifs, sset, 3, remove_dup=True)
    got = MotifSites(res, args.motifs, [0] * n, lengths).regions_with_sites()
    res.close(), sset.close()
    units = args.motifs * 2 * args.regions * 1000
    return {"config": f"configs[4]: {args.regions} target + {args.regions} control 1 kb regions x {args.motifs} motifs, "
                      "scan (dedup and regions-with-site counts on the device) + Fisher exact tests",
            "metric": "motif*bp/s (host ASCII in, enrichment table out)", "e2e_s": e2e, "scan_s": t_scan,
            "value": units / e2e, "sites": int(s_in + s_ctl),
            "top_result": list(min(results, key=lambda r: r.p_enriched))[:5],
            "cpu_baseline": {"kind": kind, "cores": os.cpu_count(), "sample": f"{n} regions x all motifs (scan only)",
                             "value": args.motifs * n * 1000 / cpu_s, "seconds": cpu_s},
            "parity": {"regions_with_site_counts_identical_on_sample": bool(np.array_equal(got, want))}}


def bench_cli(args):
    """configs[4] through the command line: `python -m motifscan_b200 scan` on 200k target + 200k control 1 kb regions x
    1,900 motifs (20 of them 33-40 columns long), a synthetic genome directory with a packed-genome cache next to
    the FASTA; wall time and peak RSS of the whole process (region parsing, scans, both site tables -- 1,900 columns
    x 200,000 rows each -- and the enrichment table).  The first `--cpu-regions` rows of the tables are compared with
    the reference pipeline (its extension on the CPU, its regrouping, de-duplication and writers restated)."""
    import resource
    import shutil
    import subprocess
    import tempfile
    import oracle
    import bench
    from motifscan_b200 import engine, synth
    from motifscan_b200 import io as msio
    from motifscan_b200.motif import MotifPwms, PositionWeightMatrix
    from motifscan_b200.scanner import MotifSite
    root = tempfile.mkdtemp(prefix="msb_cli_")
    gdir, mdir = os.path.join(root, "synth"), os.path.join(root, "jaspar_all")
    os.makedirs(gdir), os.makedirs(mdir)
    t0 = time.perf_counter()
    pg = bench.make_genome(0, args.genome_scale)
    with open(os.path.join(gdir, "synth.fa"), "wb") as fh:          # one line per chromosome
        for c in pg.chroms:
            fh.write(f">{c}\n".encode())
            fh.write(pg.decode_bytes(c, 0, pg.chrom_sizes[c]))
            fh.write(b"\n")
    pg.save(os.path.join(gdir, "synth.packed"))
    with open(os.path.join(gdir, "synth_bg_freq.txt"), "w") as fh:
        fh.write("Base\tFrequency\n" + "".join(f"{b}\t{v}\n" for b, v in synth.BG.items()))
    _, mats, ids = synth.motif_set(args.motifs, seed=2020, n_long=20)
    ctx = engine.default_context(0)
    mset = engine.MotifSet(ctx, mats)
    bblob, boff = synth.background_samples(100000, 40, seed=1)
    bg = engine.SequenceSet(ctx, blob=bblob, seq_off=boff)
    cutoffs = np.maximum(np.around(engine.score_select(ctx, mset, bg, 3, [int(100000 * 1e-4) - 1])[:, 0], 8), 1e-6)
    bg.close(), mset.close()
    pwms = MotifPwms(name="jaspar_all", genome="synth")
    for m, k, c in zip(mats, ids, cutoffs):
        pwms.append(PositionWeightMatrix(m, name="TF" + k[2:6], matrix_id=k, cutoffs={"1e-4": float(c)}))
    pwms.write_motifscan_pwms(os.path.join(mdir, "jaspar_all_synth_pwms.motifscan"))
    rng = np.random.default_rng(77)
    big = [c for c in pg.chroms if pg.chrom_sizes[c] > 20000]
    sizes = np.array([pg.chrom_sizes[c] for c in big], dtype=np.float64)
    for name in ("targets.bed", "controls.bed"):
        ci = rng.choice(len(big), size=args.regions, p=sizes / sizes.sum())
        st = (rng.random(args.regions) * (sizes[ci] - 2000)).astype(np.int64)
        with open(os.path.join(root, name), "w") as fh:
            for i in range(args.regions):
                fh.write(f"{big[ci[i]]}\t{st[i]}\t{st[i] + 1000}\tr{i}\t{1 + i % 50}\n")
    setup_s = time.perf_counter() - t0
    out = os.path.join(root, "out")
    cmd = [sys.executable, "-m", "motifscan_b200", "scan", "-i", os.path.join(root, "targets.bed"), "-c", os.path.join(root, "controls.bed"),
           "-m", mdir, "-g", gdir, "-o", out, "-w", "0", "-p", "1e-4", "--gpus", str(args.gpus)]
    runs = []
    for _ in range(2):
        shutil.rmtree(out, ignore_errors=True)
        before = resource.getrusage(resource.RUSAGE_CHILDREN).ru_maxrss
        t0 = time.perf_counter()
        proc = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True)
        dt = time.perf_counter() - t0
        if proc.returncode != 0:
            raise SystemExit("motifscan scan failed:\n" + proc.stderr[-2000:])
        runs.append((dt, max(resource.getrusage(resource.RUSAGE_CHILDREN).ru_maxrss, before) / 1024.0))
    wall_s, rss_mb = min(r[0] for r in runs), runs[-1][1]
    # parity sample: the first rows of the two tables vs the reference pipeline
    n = args.cpu_regions
    kind, ext = cpu_ext()
    regions = []
    with open(os.path.join(root, "targets.bed")) as fh:
        for line in fh:
            f = line.split("\t")
            regions.append((f[0], int(f[1]), int(f[2])))
            if len(regions) == n:
                break
    seqs = [pg.decode_bytes(c, a, b).decode() for c, a, b in regions]
    t0 = time.perf_counter()
    raw = ext.c_scan_motif([m.tolist() for m in mats], cutoffs.tolist(), seqs, 3, os.cpu_count() or 1)
    cpu_s = time.perf_counter() - t0
    nested = oracle.deduplicate_motif_sites(oracle.make_motif_sites(raw, [a for _, a, _ in regions]), [m.shape[1] for m in mats])
    nested = [[[MotifSite(*s) for s in cell] for cell in per] for per in nested]

    class Region:
        def __init__(self, c, a, b):
            self.chrom, self.start, self.end = c, a, b
    ref_dir = os.path.join(root, "ref")
    msio.write_sites_table(ref_dir, pwms, [Region(*r) for r in regions], nested)
    same, first_diff = True, None
    for name in ("motif_sites_number.xls", "motif_sites_score.xls"):
        with open(os.path.join(ref_dir, name)) as a, open(os.path.join(out, name)) as b:
            for row in range(n + 1):
                la, lb = a.readline(), b.readline()
                if la != lb:
                    same = False
                    if first_diff is None:
                        fa, fb = la.rstrip("\n").split("\t"), lb.rstrip("\n").split("\t")
                        cols = [k for k in range(min(len(fa), len(fb))) if fa[k] != fb[k]]
                        first_diff = {"table": name, "row": row, "n_fields": [len(fa), len(fb)], "columns": cols[:8],
                                      "reference": [fa[k] for k in cols[:8]], "ours": [fb[k] for k in cols[:8]],
                                      "motif_lengths": [int(mats[k - 3].shape[1]) for k in cols[:8] if k >= 3]}
    sizes_out = {name: os.path.getsize(os.path.join(out, name)) for name in sorted(os.listdir(out))}
    shutil.rmtree(root, ignore_errors=True)
    return {"config": f"configs[4] through the CLI: motifscan scan, {args.regions} target + {args.regions} control 1 kb regions x {args.motifs} motifs "
                      f"(20 of 33-40 columns), genome {sum(pg.chrom_sizes.values())} bp with a packed cache, --gpus {args.gpus}",
            "metric": "wall seconds of the whole command (parse, scan, 2 site tables, enrichment table)", "wall_s": wall_s,
            "runs_s": [r[0] for r in runs], "peak_rss_mb": rss_mb, "output_bytes": sizes_out, "setup_s": setup_s,
            "value": args.motifs * 2 * args.regions * 1000 / wall_s,
            "cpu_baseline": {"kind": kind, "cores": os.cpu_count(), "sample": f"{n} regions x all motifs (extension call only)",
                             "value": args.motifs * n * 1000 / cpu_s, "seconds": cpu_s},
            "parity": {f"first_{n}_rows_of_both_site_tables_identical_to_the_reference_pipeline": bool(same),
                       "first_difference": first_diff}}


def bench_whole_genome(args):
    """`scan --whole-genome` on the configs[3] genome and motif set (bench.py's: 750 motifs, cutoffs at p = 1e-4
    floored at 1e-6) with the reference's de-duplication over whole chromosomes: the tables alone (no site array
    leaves a device) and with every site gathered and written as BED, on one GPU and on `--gpus N` in the same
    process.  The BED files go to a temporary directory (`--out-dir`) that is deleted afterwards."""
    import shutil
    import subprocess
    import tempfile
    import bench
    from motifscan_b200 import _lib, engine
    from motifscan_b200 import io as msio
    from motifscan_b200.genome_scan import GenomeScanner
    from motifscan_b200.region import GenomicRegion

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    pg = bench.make_genome(0, args.genome_scale)
    mats = bench.motif_workload()
    ctx = engine.default_context(0)
    cutoffs = bench.scan_cutoffs(bench.cutoffs_gpu(engine, ctx, mats))

    class Pwm:
        def __init__(self, k, m):
            self.matrix_id, self.name, self.length = f"SYN{k:04d}.1", f"motif{k}", int(np.asarray(m).shape[1])
    pwms = [Pwm(k, m) for k, m in enumerate(mats)]
    regions = [GenomicRegion(c, 0, pg.chrom_sizes[c]) for c in pg.chroms]
    total_bp = sum(pg.chrom_sizes.values())
    out_root = tempfile.mkdtemp(prefix="msb_wg_", dir=args.out_dir)
    legs = []
    try:
        for n in sorted({1, args.gpus}):
            devices = list(range(n))
            gs = GenomeScanner(pg, mats, cutoffs=cutoffs, devices=devices, unit_bp=bench.UNIT_BP)
            raw = gs.scan(collect_sites=False)                  # sites before de-duplication (counts only)
            n_raw = int(raw.counts.sum())
            gs.close()
            for site in (False, True):
                gs = GenomeScanner(pg, mats, cutoffs=cutoffs, devices=devices, unit_bp=bench.UNIT_BP, remove_dup=True)
                out_dir = os.path.join(out_root, f"{n}gpu_{int(site)}")
                t0 = time.perf_counter()
                res = gs.scan(collect_sites=site)
                t_scan = time.perf_counter() - t0
                msio.write_cell_tables(out_dir, pwms, regions, res.cell_counts.T, res.cell_best.T)
                t_tables = time.perf_counter() - t0 - t_scan
                leg = {"gpus": n, "site": site, "scan_s": t_scan, "tables_s": t_tables, "sites_raw": n_raw,
                       "sites_dedup": int(res.counts.sum()), "stitch": gs.last_stitch,
                       "device_ms": {k: sum(st.get(k, 0.0) for st in gs.last_stats) for k in ("prefilter", "exact", "order")},
                       "note": "device_ms: summed over the GPUs; 'order' holds the sort, decode, de-duplication and boundary chains"}
                if site:
                    t1 = time.perf_counter()
                    _ = res.chrom_idx                            # gather + corrections
                    leg["gather_s"] = time.perf_counter() - t1
                    t1 = time.perf_counter()
                    msio.write_sites_bed(out_dir, pwms, regions, res)
                    leg["bed_write_s"] = time.perf_counter() - t1
                    leg["bed_bytes"] = sum(os.path.getsize(os.path.join(out_dir, "motif_sites", f))
                                           for f in os.listdir(os.path.join(out_dir, "motif_sites")))
                leg["wall_s"] = time.perf_counter() - t0
                leg["motif_bp_per_s_scan"] = len(mats) * total_bp / t_scan
                legs.append(leg)
                gs.close()
                shutil.rmtree(out_dir, ignore_errors=True)
    finally:
        shutil.rmtree(out_root, ignore_errors=True)
    return {"config": f"whole-genome scan with de-duplication: {total_bp} bp synthetic hg19-shaped genome "
                      f"(scale {args.genome_scale}) x {len(mats)} motifs, both strands, p=1e-4 cutoffs floored at 1e-6",
            "card": smi.stdout.strip().splitlines(), "devices_visible": _lib.device_count(), "legs": legs,
            "note": "wall_s = scan + tables (+ gather + BED write); the genome is generated and packed before the timed "
                    "region; one pass per leg, no warm-up besides the counts-only pass"}


def _oracle_trim(ref, alt):
    """(offset of the change in REF, r', inserted bases): an indel without its longest common prefix and then suffix
    (bases compared as scoring sees them); SNVs / MNVs as they are."""
    if len(ref) == len(alt):
        return 0, len(ref), alt
    code = lambda b: "ACGT".find(b.upper()) if b.upper() in "ACGT" else 4   # noqa: E731
    m, pre, suf = min(len(ref), len(alt)), 0, 0
    while pre < m and code(ref[pre]) == code(alt[pre]):
        pre += 1
    while suf < m - pre and code(ref[-1 - suf]) == code(alt[-1 - suf]):
        suf += 1
    return pre, len(ref) - pre - suf, alt[pre:len(alt) - suf]


def _oracle_variant_rows(pg, pwms, cutoffs, v, strand=3):
    """The reference's arithmetic on host-built contexts (oracle.scan_arrays on each allele's ref and alt context,
    windows that overlap the changed bases, the other allele's window scored with oracle.score_arrays): rows
    (allele, motif, chromosome start, strand, ref_score, alt_score, effect, paired) in the contract's order.  An indel's
    window with no counterpart on the other allele is unpaired, its other score NaN."""
    import oracle
    lens = [int(np.asarray(p).shape[1]) for p in pwms]
    lmax = max(lens)
    seqs, meta = [], []
    for a in range(len(v)):
        c = v.chroms[v.chrom[a]]
        pre, r, ins = _oracle_trim(v.ref[a], v.alt[a])
        p = int(v.pos[a]) + pre
        cs, ce = max(p - lmax + 1, 0), min(p + r + lmax - 1, pg.chrom_sizes[c])
        ref_ctx = pg.decode_bytes(c, cs, ce).decode()
        seqs += [ref_ctx, ref_ctx[:p - cs] + ins + ref_ctx[p - cs + r:]]
        meta.append((cs, p - cs, r, len(ins)))
    mats = [np.asarray(p).tolist() for p in pwms]
    counts, seq_idx, start, score, strd = oracle.scan_arrays(mats, list(cutoffs), seqs, strand, n_threads=os.cpu_count() or 1)
    hits = {}
    for m, q, s, sc, x in zip(np.repeat(np.arange(len(pwms)), counts).tolist(), seq_idx.tolist(), start.tolist(),
                              score.tolist(), strd.tolist()):
        a, side = divmod(q, 2)
        cs, c0, r, k_alt = meta[a]
        if s + lens[m] > c0 and s < c0 + (k_alt if side else r):
            paired = s < c0 + min(r, k_alt) and s + lens[m] <= len(seqs[2 * a + 1 - side])
            hits.setdefault((a, m, s, x) if paired else (a, m, s, x, side), [None, None])[side] = sc
    todo = {}
    for key, sides in hits.items():
        for side in (0, 1):
            if len(key) == 4 and sides[side] is None:
                todo.setdefault((key[1], key[3]), []).append((key, side, seqs[2 * key[0] + side][key[2]:key[2] + lens[key[1]]]))
    for (m, x), items in todo.items():
        for (key, side, _), val in zip(items, oracle.score_arrays([mats[m]], [w for _, _, w in items], x)[0].tolist()):
            hits[key][side] = val
    rows = []
    for key, (rs, al) in hits.items():
        a, m, s, x = key[:4]
        if len(key) == 5:
            rows.append((a, m, meta[a][0] + s, x, np.nan if rs is None else rs, np.nan if al is None else al,
                         1 if key[4] == 0 else 2, False))
            continue
        rh, ah = rs - cutoffs[m] >= -1e-10, al - cutoffs[m] >= -1e-10
        rows.append((a, m, meta[a][0] + s, x, rs, al, 3 if rh and ah else (1 if rh else 2), True))
    rows.sort(key=lambda t: t[:4])
    return rows


def _synthetic_vcf(path, pg, n_alleles, seed=31, indel_fraction=0.0):
    """A seeded VCF of about `n_alleles` scanned alleles on `pg`: positions uniform over the non-N bases, REF from the
    genome; ~90 % SNV records, ~8 % MNVs of 2-3 bases, ~2 % records with two ALTs, plus ~1 % records that are skipped
    (indels, an unknown chromosome, a REF that does not match).  `indel_fraction` of the other records become
    deletions or insertions (half each) of 1-50 bases, 1 % of them of 80-150 bases, longer than every motif (drawn
    from their own seeded stream, so 0 leaves the file as it is)."""
    rng = np.random.default_rng(seed)
    chroms = list(pg.chroms)
    sizes = np.array([pg.chrom_sizes[c] for c in chroms], dtype=np.int64)
    cum = np.concatenate([[0], np.cumsum(sizes)])
    n_rec = int(n_alleles / 1.02)
    kind = rng.random(n_rec)
    r = np.where(kind < 0.90, 1, np.where(kind < 0.98, rng.integers(2, 4, n_rec), 1)).astype(np.int64)
    two_alts = kind >= 0.98
    pos = np.zeros(0, dtype=np.int64)
    chrom = np.zeros(0, dtype=np.int64)
    while len(pos) < n_rec:                      # uniform over the bases, rejecting N (and windows running off the end)
        g = rng.integers(0, int(cum[-1]), 2 * n_rec)
        c = np.searchsorted(cum, g, side="right") - 1
        p = g - cum[c]
        b = pg.block_off[c] + p // 32
        ok = ((np.asarray(pg.nmask)[b] >> (p % 32).astype(np.uint32)) & 1) == 0
        ok &= p + 3 <= sizes[c]
        pos, chrom = np.concatenate([pos, p[ok]]), np.concatenate([chrom, c[ok]])
    pos, chrom = pos[:n_rec], chrom[:n_rec]
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    k = np.arange(3)
    q = pos[:, None] + k[None, :]
    b = pg.block_off[chrom][:, None] + q // 32
    word = np.asarray(pg.codes)[2 * b + (q % 32) // 16]
    code = ((word >> (2 * (q % 16)).astype(np.uint32)) & 3).astype(np.int64)
    isn = ((np.asarray(pg.nmask)[b] >> (q % 32).astype(np.uint32)) & 1) == 1
    ref_bytes = np.where(isn, ord("N"), acgt[code]).astype(np.uint8)
    alt_code = (code + rng.integers(1, 4, (n_rec, 3))) % 4
    alt2_code = (alt_code + rng.integers(1, 3, (n_rec, 3))) % 4
    alt2_code = np.where(alt2_code == code, (alt2_code + 1) % 4, alt2_code)
    alt_bytes, alt2_bytes = acgt[alt_code], acgt[alt2_code]
    skip = rng.random(n_rec) < 0.01
    indel = np.zeros(n_rec, dtype=bool)
    if indel_fraction > 0:
        irng = np.random.default_rng(seed + 1)
        indel = (irng.random(n_rec) < indel_fraction) & ~skip
        ilen = np.where(irng.random(n_rec) < 0.01, irng.integers(80, 151, n_rec), irng.integers(1, 51, n_rec))
        is_del = irng.random(n_rec) < 0.5
        ins_bases = acgt[irng.integers(0, 4, (n_rec, 150))]
    lines = []
    refs = [bytes(row).decode() for row in ref_bytes]
    alts = [bytes(row).decode() for row in alt_bytes]
    alts2 = [bytes(row).decode() for row in alt2_bytes]
    for i in range(n_rec):
        ri = int(r[i])
        ref, alt = refs[i][:ri], alts[i][:ri]
        if two_alts[i]:
            alt += "," + alts2[i][:ri]
        chrom_name = chroms[chrom[i]]
        if indel[i]:
            k = int(ilen[i])
            if is_del[i]:
                ref = pg.decode_bytes(chrom_name, int(pos[i]), min(int(pos[i]) + 1 + k, int(sizes[chrom[i]]))).decode()
                alt = ref[0]
            else:
                ref = refs[i][0]
                alt = ref + bytes(ins_bases[i, :k]).decode()
        if skip[i]:
            which = i % 3
            if which == 0:
                alt = alt.split(",")[0] + "T"                          # insertion: unsupported
            elif which == 1:
                chrom_name = "chrUnknown"
            else:
                ref = alt.split(",")[0]                                # REF differs from the genome: ref_mismatch
        lines.append(f"{chrom_name}\t{pos[i] + 1}\tv{i}\t{ref}\t{alt}\t.\tPASS\t.\n")
    with open(path, "w") as fh:
        fh.write("##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\n")
        fh.writelines(lines)
    return n_rec


def bench_variants(args):
    """`motifscan variant` on the configs[3]-shaped genome at `--genome-scale` with 750 motifs (cutoffs as `cli` makes
    them) and a seeded VCF of `--alleles` alleles (default 4e6 x scale): VCF parsing, the device phases of
    scan_variants, the native table writer, the whole command in a subprocess (wall time, peak RSS), and parity of a
    seeded sample of alleles with the oracle.  Everything is written to a temporary directory that is deleted."""
    import resource
    import shutil
    import subprocess
    import tempfile
    import bench
    from motifscan_b200 import engine, synth
    from motifscan_b200 import io as msio
    from motifscan_b200.genome import DeviceGenome
    from motifscan_b200.motif import MotifPwms, PositionWeightMatrix
    from motifscan_b200.variants import Variants, read_vcf, scan_variants

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    root = tempfile.mkdtemp(prefix="msb_var_", dir=args.out_dir)
    try:
        t0 = time.perf_counter()
        pg = bench.make_genome(0, args.genome_scale)
        gdir, mdir = os.path.join(root, "synth"), os.path.join(root, "jaspar_all")
        os.makedirs(gdir), os.makedirs(mdir)
        with open(os.path.join(gdir, "synth.fa"), "wb") as fh:
            for c in pg.chroms:
                fh.write(f">{c}\n".encode() + pg.decode_bytes(c, 0, pg.chrom_sizes[c]) + b"\n")
        pg.save(os.path.join(gdir, "synth.packed"))
        with open(os.path.join(gdir, "synth_bg_freq.txt"), "w") as fh:
            fh.write("Base\tFrequency\n" + "".join(f"{b}\t{v}\n" for b, v in synth.BG.items()))
        _, mats, ids = synth.motif_set(args.motifs, seed=2020)
        ctx = engine.default_context(0)
        mset = engine.MotifSet(ctx, mats)
        bblob, boff = synth.background_samples(100000, 40, seed=1)
        bg = engine.SequenceSet(ctx, blob=bblob, seq_off=boff)
        cutoffs = np.maximum(np.around(engine.score_select(ctx, mset, bg, 3, [int(100000 * 1e-4) - 1])[:, 0], 8), 1e-6)
        bg.close(), mset.close()
        pwms = MotifPwms(name="jaspar_all", genome="synth")
        for m, k, c in zip(mats, ids, cutoffs):
            pwms.append(PositionWeightMatrix(m, name="TF" + k[2:6], matrix_id=k, cutoffs={"1e-4": float(c)}))
        pwms.write_motifscan_pwms(os.path.join(mdir, "jaspar_all_synth_pwms.motifscan"))
        n_alleles = args.alleles or int(4e6 * args.genome_scale)
        vcf = os.path.join(root, "calls.vcf")
        indels = args.indel_fraction > 0
        n_rec = _synthetic_vcf(vcf, pg, n_alleles, indel_fraction=args.indel_fraction)
        setup_s = time.perf_counter() - t0

        t0 = time.perf_counter()
        v = read_vcf(vcf, pg, indels=indels)
        parse_s = time.perf_counter() - t0
        dg = DeviceGenome(pg, ctx)
        runs = []
        for _ in range(args.steps + 1):                                 # the first run warms up
            sites = scan_variants(dg, mats, cutoffs, v)
            runs.append((sites.seconds, sites.timings))
        best = min(runs[1:], key=lambda x: x[0])
        scan_s, dev = best
        dev_total = sum(dev.values())
        out = os.path.join(root, "tables")
        t0 = time.perf_counter()
        msio.write_variant_tables(out, pwms, v, sites)
        write_s = time.perf_counter() - t0
        out_bytes = {f: os.path.getsize(os.path.join(out, f)) for f in sorted(os.listdir(out))}
        # parity: a seeded sample of alleles, scanned on their own and compared with the oracle and with the full run
        rng = np.random.default_rng(5)
        idx = np.sort(rng.choice(len(v), size=min(args.cpu_alleles, len(v)), replace=False))
        sub = Variants(v.chroms, v.chrom[idx], v.pos[idx], [v.ref[i] for i in idx], [v.alt[i] for i in idx],
                       [v.id[i] for i in idx], v.record[idx], v.skipped, v.n_records, indels=v.indels)
        got = scan_variants(dg, mats, cutoffs, sub)
        t0 = time.perf_counter()
        want = _oracle_variant_rows(pg, mats, cutoffs, sub)
        cpu_s = time.perf_counter() - t0
        cols = list(zip(*want)) if want else [[]] * 8
        same = (len(got) == len(want) and np.array_equal(got.allele, np.array(cols[0], np.int32))
                and np.array_equal(got.motif, np.array(cols[1], np.int32)) and np.array_equal(got.start, np.array(cols[2], np.int64))
                and np.array_equal(got.strand, np.array(cols[3], np.int8))
                and np.array_equal(got.ref_score.view(np.uint64), np.array(cols[4], np.float64).view(np.uint64))
                and np.array_equal(got.alt_score.view(np.uint64), np.array(cols[5], np.float64).view(np.uint64))
                and np.array_equal(got.effect, np.array(cols[6], np.int8)) and np.array_equal(got.paired, np.array(cols[7], bool)))
        in_full = np.isin(sites.allele, idx)
        full_same = (np.array_equal(np.searchsorted(idx, sites.allele[in_full]), got.allele)
                     and np.array_equal(sites.start[in_full], got.start) and np.array_equal(sites.motif[in_full], got.motif)
                     and np.array_equal(sites.ref_score[in_full].view(np.uint64), got.ref_score.view(np.uint64))
                     and np.array_equal(sites.alt_score[in_full].view(np.uint64), got.alt_score.view(np.uint64))
                     and np.array_equal(sites.effect[in_full], got.effect) and np.array_equal(sites.paired[in_full], got.paired))
        dg.close()
        # the whole command, as a user runs it (the packed cache next to the FASTA is used)
        cmd = [sys.executable, "-m", "motifscan_b200", "variant", "-i", vcf, "-m", mdir, "-g", gdir, "-o",
               os.path.join(root, "cli"), "-p", "1e-4"] + (["--indels"] if indels else [])
        t0 = time.perf_counter()
        proc = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True)
        wall_s = time.perf_counter() - t0
        if proc.returncode != 0:
            raise SystemExit("motifscan variant failed:\n" + proc.stderr[-2000:])
        rss_mb = resource.getrusage(resource.RUSAGE_CHILDREN).ru_maxrss / 1024.0
        cli_same = all(open(os.path.join(root, "cli", f), "rb").read() == open(os.path.join(out, f), "rb").read()
                       for f in out_bytes)
        log = [line for line in proc.stderr.splitlines() if line.startswith("Scanned")]
    finally:
        shutil.rmtree(root, ignore_errors=True)
    extra = {}
    if indels:
        is_indel = np.fromiter((len(a) != len(r) for a, r in zip(v.alt, v.ref)), dtype=bool, count=len(v))
        extra = {"indel_fraction": args.indel_fraction, "indel_alleles": int(is_indel.sum()),
                 "sample_indel_alleles": int(is_indel[idx].sum()),
                 "rows_by_pairing": {"paired": int(sites.paired.sum()),
                                     "unpaired_loss": int((~sites.paired & (sites.effect == 1)).sum()),
                                     "unpaired_gain": int((~sites.paired & (sites.effect == 2)).sum())}}
    return {**extra, "config": f"motifscan variant: {n_rec} VCF records -> {len(v)} scanned alleles on a {sum(pg.chrom_sizes.values())} bp "
                      f"synthetic genome (scale {args.genome_scale}) x {args.motifs} motifs, both strands, p=1e-4 cutoffs floored at 1e-6",
            "card": smi.stdout.strip().splitlines(), "metric": "motif*bp/s over the context bases of both alleles",
            "scan_s": scan_s, "value": sites.motif_bp / scan_s, "alleles_per_s": len(v) / scan_s,
            "device_ms": dev, "device_ms_total": dev_total, "device_value": sites.motif_bp / max(dev_total / 1e3, 1e-12),
            "motif_bp": sites.motif_bp, "context_bp_per_set": sites.context_bp, "rows": len(sites),
            "rows_by_effect": sites.rows_by_effect(), "skipped": v.skipped, "vcf_parse_s": parse_s,
            "writer": {"seconds": write_s, "bytes": out_bytes}, "setup_s": setup_s,
            "cli": {"wall_s": wall_s, "peak_rss_mb": rss_mb, "tables_identical_to_the_library_run": bool(cli_same), "log": log},
            "parity": {"sample_alleles": int(len(idx)), "rows": len(want), "identical_to_oracle": bool(same),
                       "full_run_rows_of_the_sample_identical": bool(full_same), "oracle_s": cpu_s},
            "note": "scan_s: scan_variants wall time (extract both context sets, two scans, rows, sort, copy back), best of "
                    "--steps after one warm-up; device_ms per phase of that run"}


def _synthetic_phased_vcf(path, pg, n_alleles, n_samples, seed=37, indel_fraction=0.0):
    """A seeded phased VCF of about `n_alleles` alleles on `pg` and `n_samples` samples whose allele spacing makes
    multi-allele clusters: alleles come in bursts of 1-8 (positions uniform over the non-N bases), 1-20 bases apart;
    SNVs, and with `indel_fraction` deletions / insertions (half each) of 1-20 bases.  Each allele has a frequency
    drawn from Beta(0.5, 2) and each haplotype carries it with that probability, so haplotypes carry different subsets
    of a burst.  Returns (records, alleles)."""
    rng = np.random.default_rng(seed)
    chroms = list(pg.chroms)
    sizes = np.array([pg.chrom_sizes[c] for c in chroms], dtype=np.int64)
    cum = np.concatenate([[0], np.cumsum(sizes)])
    n_bursts = max(n_alleles // 4, 1)
    burst = rng.integers(1, 9, n_bursts)
    g = rng.integers(0, int(cum[-1]), n_bursts)
    c = np.searchsorted(cum, g, side="right") - 1
    start = g - cum[c]
    cs = np.cumsum(rng.integers(1, 21, int(burst.sum())))
    pos = np.repeat(start, burst) + cs - np.repeat(cs[np.cumsum(burst) - burst], burst)
    chrom = np.repeat(c, burst)
    ok = pos + 25 < sizes[chrom]
    pos, chrom = pos[ok], chrom[ok]
    order = np.lexsort((pos, chrom))
    pos, chrom = pos[order], chrom[order]
    keep = np.ones(len(pos), dtype=bool)
    keep[1:] = (pos[1:] != pos[:-1]) | (chrom[1:] != chrom[:-1])
    pos, chrom = pos[keep], chrom[keep]
    n = len(pos)
    b = pg.block_off[chrom] + pos // 32
    isn = ((np.asarray(pg.nmask)[b] >> (pos % 32).astype(np.uint32)) & 1) == 1
    pos, chrom, n = pos[~isn], chrom[~isn], int((~isn).sum())
    kind = rng.random(n)
    is_del = kind < indel_fraction / 2
    is_ins = (kind >= indel_fraction / 2) & (kind < indel_fraction)
    ilen = rng.integers(1, 21, n)
    acgt = "ACGT"
    af = rng.beta(0.5, 2.0, n)
    carry = rng.random((n, 2 * n_samples)) < af[:, None]
    lines = []
    for i in range(n):
        cn, p = chroms[chrom[i]], int(pos[i])
        if is_del[i]:
            ref = pg.decode_bytes(cn, p, p + 1 + int(ilen[i])).decode()
            alt = ref[0]
        else:
            ref = pg.decode_bytes(cn, p, p + 1).decode()
            alt = ref + "".join(rng.choice(list(acgt), int(ilen[i]))) if is_ins[i] else \
                acgt[(acgt.find(ref.upper()) + int(rng.integers(1, 4))) % 4]
        row = carry[i]
        gts = "\t".join(f"{int(row[2 * k])}|{int(row[2 * k + 1])}" for k in range(n_samples))
        lines.append(f"{cn}\t{p + 1}\th{i}\t{ref}\t{alt}\t.\tPASS\t.\tGT\t{gts}\n")
    with open(path, "w") as fh:
        fh.write("##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t" +
                 "\t".join(f"S{k}" for k in range(n_samples)) + "\n")
        fh.writelines(lines)
    return n


def bench_haplotypes(args):
    """`motifscan variant --haplotypes` on the configs[3]-shaped genome at `--genome-scale` with 750 motifs and a
    seeded phased VCF of `--alleles` alleles x `--samples` samples (_synthetic_phased_vcf): VCF + GT parsing, the
    clustering, the device phases of scan_haplotypes, rows by effect, the whole command in a subprocess (wall time,
    peak RSS) and parity of a seeded sample of clusters with the oracle of tests/test_gpu_haplotypes.py."""
    import resource
    import shutil
    import subprocess
    import tempfile
    import bench
    from motifscan_b200 import engine, synth
    from motifscan_b200.genome import DeviceGenome
    from motifscan_b200.motif import MotifPwms, PositionWeightMatrix
    from motifscan_b200.variants import Haplotypes, haplotype_clusters, read_vcf, scan_haplotypes
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_gpu_haplotypes import oracle_rows

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    root = tempfile.mkdtemp(prefix="msb_hap_", dir=args.out_dir)
    try:
        t0 = time.perf_counter()
        pg = bench.make_genome(0, args.genome_scale)
        gdir, mdir = os.path.join(root, "synth"), os.path.join(root, "jaspar_all")
        os.makedirs(gdir), os.makedirs(mdir)
        with open(os.path.join(gdir, "synth.fa"), "wb") as fh:
            for c in pg.chroms:
                fh.write(f">{c}\n".encode() + pg.decode_bytes(c, 0, pg.chrom_sizes[c]) + b"\n")
        pg.save(os.path.join(gdir, "synth.packed"))
        with open(os.path.join(gdir, "synth_bg_freq.txt"), "w") as fh:
            fh.write("Base\tFrequency\n" + "".join(f"{b}\t{v}\n" for b, v in synth.BG.items()))
        _, mats, ids = synth.motif_set(args.motifs, seed=2020)
        ctx = engine.default_context(0)
        mset = engine.MotifSet(ctx, mats)
        bblob, boff = synth.background_samples(100000, 40, seed=1)
        bg = engine.SequenceSet(ctx, blob=bblob, seq_off=boff)
        cutoffs = np.maximum(np.around(engine.score_select(ctx, mset, bg, 3, [int(100000 * 1e-4) - 1])[:, 0], 8), 1e-6)
        bg.close(), mset.close()
        pwms = MotifPwms(name="jaspar_all", genome="synth")
        for m, k, c in zip(mats, ids, cutoffs):
            pwms.append(PositionWeightMatrix(m, name="TF" + k[2:6], matrix_id=k, cutoffs={"1e-4": float(c)}))
        pwms.write_motifscan_pwms(os.path.join(mdir, "jaspar_all_synth_pwms.motifscan"))
        n_alleles = args.alleles or int(1e6 * args.genome_scale)
        vcf = os.path.join(root, "phased.vcf")
        indels = args.indel_fraction > 0
        n_rec = _synthetic_phased_vcf(vcf, pg, n_alleles, args.samples, indel_fraction=args.indel_fraction)
        setup_s = time.perf_counter() - t0
        lmax = max(m.shape[1] for m in mats)
        t0 = time.perf_counter()
        v = read_vcf(vcf, pg, indels=indels, samples="all")
        parse_s = time.perf_counter() - t0
        t0 = time.perf_counter()
        h = haplotype_clusters(v, lmax)
        cluster_s = time.perf_counter() - t0
        dg = DeviceGenome(pg, ctx)
        runs = []
        for _ in range(args.steps + 1):                                 # the first run warms up
            sites = scan_haplotypes(dg, mats, cutoffs, h)
            runs.append((sites.seconds, sites.timings))
        scan_s, dev = min(runs[1:], key=lambda x: x[0])
        # parity: a seeded sample of clusters, scanned on their own and compared with the oracle and the full run
        rng = np.random.default_rng(5)
        sel = np.sort(rng.choice(len(h), size=min(args.cpu_clusters, len(h)), replace=False))
        cnt = h.sizes()[sel]
        aoff = np.concatenate([[0], np.cumsum(cnt)])
        alle = h.allele[np.repeat(h.allele_off[sel], cnt) + np.arange(int(cnt.sum())) - np.repeat(aoff[:-1], cnt)]
        sub = Haplotypes(v, lmax, h.chrom[sel], aoff, alle, np.zeros(len(sel) + 1, np.int64), [], [], 0)
        got = scan_haplotypes(dg, mats, cutoffs, sub)
        dg.close()

        class _Chrom:
            def __init__(self, c):
                self.c = c

            def __len__(self):
                return int(pg.chrom_sizes[self.c])

            def __getitem__(self, sl):
                return pg.decode_bytes(self.c, sl.start, min(sl.stop, len(self))).decode()

        texts = {c: _Chrom(c) for c in pg.chroms}
        t0 = time.perf_counter()
        want = oracle_rows(texts, sub, mats, cutoffs, "both")
        cpu_s = time.perf_counter() - t0
        cols = list(zip(*want)) if want else [[]] * 9
        same = len(got) == len(want)
        for name, k, dt in (("cluster", 0, np.int32), ("motif", 1, np.int32), ("strand", 2, np.int8), ("ref_start", 3, np.int64),
                            ("alt_start", 4, np.int64), ("effect", 7, np.int8), ("paired", 8, bool)):
            same = same and np.array_equal(getattr(got, name), np.array(cols[k], dt))
        for name, k in (("ref_score", 5), ("alt_score", 6)):
            w = np.array(cols[k], np.float64)
            same = same and np.array_equal(np.isnan(getattr(got, name)), np.isnan(w)) and np.array_equal(
                getattr(got, name)[~np.isnan(w)].view(np.uint64), w[~np.isnan(w)].view(np.uint64))
        in_full = np.isin(sites.cluster, sel)
        full_same = (np.array_equal(np.searchsorted(sel, sites.cluster[in_full]), got.cluster)
                     and np.array_equal(sites.ref_start[in_full], got.ref_start)
                     and np.array_equal(sites.alt_start[in_full], got.alt_start)
                     and np.array_equal(sites.ref_score[in_full].view(np.uint64), got.ref_score.view(np.uint64)))
        cmd = [sys.executable, "-m", "motifscan_b200", "variant", "-i", vcf, "-m", mdir, "-g", gdir, "-o",
               os.path.join(root, "cli"), "-p", "1e-4", "--haplotypes"] + (["--indels"] if indels else [])
        t0 = time.perf_counter()
        proc = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True)
        wall_s = time.perf_counter() - t0
        if proc.returncode != 0:
            raise SystemExit("motifscan variant --haplotypes failed:\n" + proc.stderr[-2000:])
        rss_mb = resource.getrusage(resource.RUSAGE_CHILDREN).ru_maxrss / 1024.0
        out_bytes = {f: os.path.getsize(os.path.join(root, "cli", f)) for f in sorted(os.listdir(os.path.join(root, "cli")))}
        log = [line for line in proc.stderr.splitlines() if line.startswith(("Read", "Scanned"))]
    finally:
        shutil.rmtree(root, ignore_errors=True)
    sizes = h.sizes()
    hist = np.bincount(np.minimum(sizes, 16))
    return {"config": f"motifscan variant --haplotypes: {n_rec} VCF records x {args.samples} samples -> {len(v)} alleles, "
                      f"{len(v.call_allele)} haplotype calls, {len(h)} distinct clusters on a {sum(pg.chrom_sizes.values())} bp "
                      f"synthetic genome (scale {args.genome_scale}) x {args.motifs} motifs, both strands, p=1e-4 cutoffs "
                      f"floored at 1e-6, indel fraction {args.indel_fraction}",
            "card": smi.stdout.strip().splitlines(), "clusters": len(h),
            "cluster_size_hist": {(str(k) if k < 16 else "16+"): int(x) for k, x in enumerate(hist) if x},
            "max_cluster_size": int(sizes.max()), "call_skipped": {**v.call_skipped, "overlap": h.overlap},
            "context_bp_per_set": sites.context_bp, "motif_bp": sites.motif_bp, "scan_s": scan_s,
            "value": sites.motif_bp / scan_s, "device_ms": dev, "rows": len(sites), "rows_by_effect": sites.rows_by_effect(),
            "vcf_parse_s": parse_s, "cluster_s": cluster_s, "setup_s": setup_s,
            "cli": {"wall_s": wall_s, "peak_rss_mb": rss_mb, "bytes": out_bytes, "log": log},
            "parity": {"sample_clusters": int(len(sel)), "rows": len(want), "identical_to_oracle": bool(same),
                       "full_run_rows_of_the_sample_identical": bool(full_same), "oracle_s": cpu_s},
            "note": "scan_s: scan_haplotypes wall time (extract both context sets, two scans, rows, sort, copy back), best "
                    "of --steps after one warm-up; device_ms per phase of that run; value in motif*bp/s over the context "
                    "bases of both sides"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("which", choices=["build", "genome", "enrich", "cli", "whole-genome", "variants", "haplotypes"])
    ap.add_argument("--alleles", type=int, default=None)
    ap.add_argument("--samples", type=int, default=16)
    ap.add_argument("--cpu-clusters", dest="cpu_clusters", type=int, default=500)
    ap.add_argument("--cpu-alleles", dest="cpu_alleles", type=int, default=2000)
    ap.add_argument("--indel-fraction", dest="indel_fraction", type=float, default=0.0)
    ap.add_argument("--out-dir", dest="out_dir", default=None)
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--genome-scale", dest="genome_scale", type=float, default=0.1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--motifs", type=int, default=None)
    ap.add_argument("--n-random", dest="n_random", type=int, default=1000000)
    ap.add_argument("--cpu-samples", dest="cpu_samples", type=int, default=100000)
    ap.add_argument("--genome-bp", dest="genome_bp", type=int, default=388000000)
    ap.add_argument("--chunk-bp", dest="chunk_bp", type=int, default=1 << 23)
    ap.add_argument("--batch-bp", dest="batch_bp", type=int, default=1 << 29)
    ap.add_argument("--cpu-bp", dest="cpu_bp", type=int, default=2000000)
    ap.add_argument("--regions", type=int, default=200000)
    ap.add_argument("--region-block", dest="region_block", type=int, default=50000)
    ap.add_argument("--cpu-regions", dest="cpu_regions", type=int, default=4000)
    args = ap.parse_args()
    if args.motifs is None:
        args.motifs = 1900 if args.which in ("enrich", "cli") else 750
    out = {"build": bench_build, "genome": bench_genome, "enrich": bench_enrich, "cli": bench_cli,
           "whole-genome": bench_whole_genome, "variants": bench_variants, "haplotypes": bench_haplotypes}[args.which](args)
    if out is not None:
        print(json.dumps(out))


if __name__ == "__main__":
    main()
