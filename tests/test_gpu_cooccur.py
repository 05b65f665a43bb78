"""GPU tests of motif co-occurrence and anchor spacing (msb_scan_device_pair_counts / msb_scan_device_spacing,
Scanner.scan_motifs(pairs=...), `scan --cooccur --spacing-anchor`) against an oracle built from oracle.scan_arrays +
oracle.deduplicate_motif_sites on host strings: Python sets per motif for the pair counts and a double loop over the
sites of each region for the spacing.  Every count must be equal."""
import os

import numpy as np
import pytest

import oracle
from motifscan_b200 import cli, engine
from motifscan_b200 import io as msio
from motifscan_b200.cooccur import PairSpec, cooccur_table, spacing_rows
from motifscan_b200.genome import Genome
from motifscan_b200.motif import MotifPwms, PositionWeightMatrix
from motifscan_b200.region import GenomicRegion, generate_control_regions, load_motifscan_regions
from test_gpu_cli import _tree, oracle_build, oracle_sites, workspace  # noqa: F401
from test_gpu_parity import cutoffs_for, synth_pwms, synth_seqs

pytestmark = pytest.mark.gpu

STRAND = {"+": 1, "-": 2, "both": 3}


def final_sites(pwms, cutoffs, seqs, strand, dedup):
    """[motif][region] -> [(start, strand 1 / 2)], the final sites of the scan."""
    flat = oracle.c_scan_motif(pwms, cutoffs, seqs, strand, 4)
    nested = oracle.make_motif_sites(flat, [0] * len(seqs))
    if dedup:
        nested = oracle.deduplicate_motif_sites(nested, [len(p[0]) for p in pwms])
    return [[[(s.start, 1 if s.strand == "+" else 2) for s in cell] for cell in per] for per in nested]


def oracle_pairs(sites):
    hit = [{r for r, cell in enumerate(per) if cell} for per in sites]
    n = len(sites)
    return np.array([[len(hit[a] & hit[b]) for b in range(n)] for a in range(n)], dtype=np.int64)


def oracle_spacing(sites, lengths, anchors, D):
    n, W = len(sites), 2 * D + 1
    hist = np.zeros((len(anchors), n, 2, W), dtype=np.int64)
    for k, A in enumerate(anchors):
        LA = lengths[A]
        for r, cell in enumerate(sites[A]):
            for sA, tA in cell:
                for B in range(n):
                    LB = lengths[B]
                    for sB, tB in sites[B][r]:
                        if B == A and sB == sA and tB == tA:
                            continue                       # never a site with itself
                        d = sB - sA if tA == 1 else (sA + LA) - (sB + LB)
                        if -D <= d <= D:
                            hist[k, B, int(tA != tB), d + D] += 1
    return hist


def device_run(pwms, cutoffs, seqs, strand, dedup, anchors=None, D=0, pass_words=0, split_words=0):
    ctx = engine.Context(0)
    if pass_words:
        ctx.set_option("pair_pass_words", pass_words)
    if split_words:
        ctx.set_option("pair_split_words", split_words)
    motifs = engine.MotifSet(ctx, pwms, cutoffs)
    sset = engine.SequenceSet(ctx, seqs)
    try:
        engine.scan(ctx, motifs, sset, strand, remove_dup=dedup).close()
        counts = ctx.pair_counts(len(pwms), len(seqs))
        hist = ctx.spacing(motifs, anchors, D) if anchors else None
        return counts, hist
    finally:
        sset.close(), motifs.close(), ctx.close()


def dense_case(seed, n_motifs, n_regions, lo=80, hi=400, rate=0.01, lmin=5, lmax=20):
    rng = np.random.default_rng(seed)
    pwms = synth_pwms(rng, n_motifs, lmin, lmax)
    seqs = synth_seqs(rng, n_regions, lo, hi, p_n=0.002) if n_regions else []
    cut_seqs = seqs if n_regions and max(len(s) for s in seqs) > lmax + 1 else synth_seqs(rng, 20, 200, 300)
    return pwms, cutoffs_for(pwms, cut_seqs, rate), seqs


@pytest.mark.parametrize("n_regions", [0, 1, 31, 32, 33, 64, 65])
def test_region_counts_at_the_bit_tails(n_regions):
    pwms, cutoffs, seqs = dense_case(11 + n_regions, 20, n_regions)
    if n_regions >= 3:
        seqs[1] = "N" * 50          # regions without any site
        seqs[-1] = "ACG"
    counts, hist = device_run(pwms, cutoffs, seqs, 3, True, anchors=[0, 7], D=30)
    sites = final_sites(pwms, cutoffs, seqs, 3, True)
    assert np.array_equal(counts, oracle_pairs(sites))
    assert np.array_equal(hist, oracle_spacing(sites, [len(p[0]) for p in pwms], [0, 7], 30))
    if n_regions >= 31:
        assert counts.sum() > 0


@pytest.mark.parametrize("n_motifs", [1, 127, 128, 129, 257])
def test_motif_counts_at_the_tile_edges(n_motifs):
    pwms, cutoffs, seqs = dense_case(100 + n_motifs, n_motifs, 70, rate=0.003)
    counts, hist = device_run(pwms, cutoffs, seqs, 3, True, anchors=[0, n_motifs - 1], D=12)
    sites = final_sites(pwms, cutoffs, seqs, 3, True)
    want = oracle_pairs(sites)
    assert np.array_equal(counts, want)
    assert np.array_equal(counts, counts.T)
    assert np.array_equal(hist, oracle_spacing(sites, [len(p[0]) for p in pwms], [0, n_motifs - 1], 12))
    assert (np.diagonal(want) > 0).sum() > n_motifs // 2


@pytest.mark.parametrize("pass_words", [1, 2, 3])
def test_word_range_passes(pass_words):
    pwms, cutoffs, seqs = dense_case(7, 140, 200, lo=60, hi=200, rate=0.003)
    counts, _ = device_run(pwms, cutoffs, seqs, 3, True, pass_words=pass_words)
    assert np.array_equal(counts, oracle_pairs(final_sites(pwms, cutoffs, seqs, 3, True)))


@pytest.mark.parametrize("split_words, pass_words", [(64, 0), (96, 0), (32, 0), (64, 80)])
def test_ctas_over_several_chunks(split_words, pass_words):
    """3,000 regions = 94 words: CTAs that loop over 2 or 3 32-word chunks (the last one partial), alone and inside
    word-range passes, over a diagonal and an off-diagonal motif tile."""
    pwms, cutoffs, seqs = dense_case(17, 130, 3000, lo=40, hi=120, rate=0.002)
    counts, _ = device_run(pwms, cutoffs, seqs, 3, True, pass_words=pass_words, split_words=split_words)
    want = oracle_pairs(final_sites(pwms, cutoffs, seqs, 3, True))
    assert np.array_equal(counts, want)
    assert (want[:128, 128:] > 0).any() and want.max() > 64


@pytest.mark.parametrize("strand", ["+", "-", "both"])
@pytest.mark.parametrize("dedup", [True, False])
def test_strands_and_dedup(strand, dedup):
    pwms, cutoffs, seqs = dense_case(3, 24, 40, rate=0.02)
    anchors = [2, 5, 2]
    counts, hist = device_run(pwms, cutoffs, seqs, STRAND[strand], dedup, anchors=anchors, D=25)
    sites = final_sites(pwms, cutoffs, seqs, STRAND[strand], dedup)
    assert np.array_equal(counts, oracle_pairs(sites))
    want = oracle_spacing(sites, [len(p[0]) for p in pwms], anchors, 25)
    assert np.array_equal(hist, want)
    assert want.sum() > 0


@pytest.mark.parametrize("D", [0, 1, 40])
def test_spacing_edges_self_pairs_and_mirror(D):
    """D = 0 and offsets at exactly +-D, overlapping windows, A == B, reverse anchors and anchor sites at both region
    ends, each present in the oracle's histogram."""
    pwms, cutoffs, seqs = dense_case(21, 12, 60, lo=40, hi=120, rate=0.05, lmin=4, lmax=10)
    lengths = [len(p[0]) for p in pwms]
    anchors = list(range(6))
    counts, hist = device_run(pwms, cutoffs, seqs, 3, False, anchors=anchors, D=D)
    sites = final_sites(pwms, cutoffs, seqs, 3, False)
    want = oracle_spacing(sites, lengths, anchors, D)
    assert np.array_equal(hist, want)
    assert np.array_equal(counts, oracle_pairs(sites))
    self_pairs = sum(want[k, a].sum() for k, a in enumerate(anchors))
    assert self_pairs > 0                                        # A == B
    assert want[..., 0].sum() > 0 and want[..., -1].sum() > 0    # -D and +D
    assert want[:, :, 1].sum() > 0                               # opposite orientation: reverse anchors and partners
    ends = {(s == 0, s + lengths[a] == len(seqs[r])) for a in anchors for r, cell in enumerate(sites[a]) for s, _ in cell}
    assert (True, False) in ends and (False, True) in ends      # anchor sites at both region ends


def toy_genome(tmp_path, rng):
    alphabet = np.frombuffer(b"ACGTacgt", dtype=np.uint8)
    sizes = {"chr1": 20000, "chr2": 9000}
    with open(tmp_path / "g.fa", "w") as fh:
        for chrom, n in sizes.items():
            seq = alphabet[rng.choice(8, size=n, p=[.2, .15, .15, .2, .09, .06, .06, .09])].copy()
            seq[500:560] = ord("N")
            fh.write(f">{chrom}\n{bytes(seq).decode()}\n")
    regions = []
    for _ in range(90):
        chrom = ["chr1", "chr2"][int(rng.integers(2))]
        a = int(rng.integers(0, sizes[chrom] - 600))
        regions.append(GenomicRegion(chrom, a, a + int(rng.integers(50, 600))))
    return Genome("g", str(tmp_path), bg_freq=dict(A=0.29, C=0.21, G=0.21, T=0.29)), regions


def test_scanner_paths(tmp_path):
    """ASCII, resident-genome and Scanner(devices=[0, 0, 0]) paths: counts and histograms summed over the blocks equal
    the oracle; the diagonal equals regions_with_sites(); pairs=None leaves the result as it was."""
    from motifscan_b200.genome import DeviceGenome
    from motifscan_b200.scanner import Scanner
    rng = np.random.default_rng(8)
    genome, regions = toy_genome(tmp_path, rng)
    mats = synth_pwms(rng, 30, 5, 16)
    probe = Scanner(genome=genome, regions=regions, window_size=0)
    cut = cutoffs_for(mats, [s for s in probe.sequences if len(s) > 20], 0.01)
    pwms = MotifPwms()
    for i, (m, c) in enumerate(zip(mats, cut)):
        pwms.append(PositionWeightMatrix(m, name=f"TF{i}", matrix_id=f"M{i}", cutoffs={"1e-4": c}))
    spec = PairSpec(cooccur=True, anchors=[3, 0], max_offset=20)
    sites = final_sites(mats, cut, probe.sequences, 3, True)
    want_counts = oracle_pairs(sites)
    want_hist = oracle_spacing(sites, [len(m[0]) for m in mats], [3, 0], 20)
    dg = DeviceGenome(genome)
    try:
        for src, devices in ((genome, None), (dg, None), (genome, [0, 0, 0])):
            sc = Scanner(genome=src, regions=regions, window_size=0, devices=devices)
            got = sc.scan_motifs(pwms, pairs=spec)
            assert np.array_equal(got.pairs.counts, want_counts)
            assert np.array_equal(np.diagonal(got.pairs.counts), got.regions_with_sites())
            assert np.array_equal(got.pairs.spacing, want_hist)
            assert got.pairs.n_regions == len(regions)
            plain = sc.scan_motifs(pwms)
            assert plain.pairs is None
            assert np.array_equal(plain.regions_with_sites(), got.regions_with_sites())
    finally:
        dg.close()


def test_einval_cases():
    pwms, cutoffs, seqs = dense_case(5, 10, 20)
    ctx = engine.Context(0)
    motifs = engine.MotifSet(ctx, pwms, cutoffs)
    other = engine.MotifSet(ctx, pwms[:5], cutoffs[:5])
    sset = engine.SequenceSet(ctx, seqs)
    try:
        engine.scan(ctx, motifs, sset, 3, remove_dup=True).close()
        for call in (lambda: ctx.pair_counts(9, 20), lambda: ctx.pair_counts(10, 19),
                     lambda: ctx.spacing(motifs, [10], 5), lambda: ctx.spacing(motifs, [-1], 5),
                     lambda: ctx.spacing(motifs, [0], -1), lambda: ctx.spacing(motifs, [0], 501),
                     lambda: ctx.spacing(motifs, [], 5), lambda: ctx.spacing(motifs, [0] * 17, 5),
                     lambda: ctx.spacing(other, [0], 5)):
            with pytest.raises(ValueError):
                call()
        assert ctx.spacing(motifs, [0] * 16, 500).shape == (16, 10, 2, 1001)
        engine.scan_device(ctx, motifs, sset, 3, counts_only=True)
        with pytest.raises(ValueError):
            ctx.pair_counts(10, 20)
        with pytest.raises(ValueError):
            ctx.spacing(motifs, [0], 5)
        engine.scan(ctx, motifs, sset, 3, compact=True).close()
        with pytest.raises(ValueError):
            ctx.pair_counts(10, 20)
        with pytest.raises(ValueError):
            ctx.spacing(motifs, [0], 5)
    finally:
        sset.close(), motifs.close(), other.close(), ctx.close()


def test_cli_tables_against_the_oracle(workspace, tmp_path):  # noqa: F811
    gdir, mdir = workspace / "toyg", workspace / "toym"
    if not (mdir / "toym_toyg_pwms.motifscan").exists():
        assert cli.main(["motif", "--build", str(mdir), "-g", str(gdir), "--n-random", "20000", "--seed", "1"]) == 0
    base = ["scan", "-i", str(workspace / "peaks.bed"), "-m", str(mdir), "-g", str(gdir), "-p", "1e-3", "-w", "400",
            "--site", "--n-random", "2", "--seed", "3"]
    assert cli.main(base + ["-o", str(tmp_path / "plain")]) == 0
    assert cli.main(base + ["-o", str(tmp_path / "pairs"), "--cooccur", "--spacing-anchor", "MA0003.1,TF7",
                            "--spacing-max", "30"]) == 0
    plain, pairs = _tree(tmp_path / "plain"), _tree(tmp_path / "pairs")
    assert set(pairs) == set(plain) | {"motif_cooccurrence.xls", "motif_spacing.xls"}
    assert all(pairs[k] == v for k, v in plain.items())            # the other files are byte-identical

    genome, _ = oracle_build(gdir, mdir, 20000, 1)
    pwms = MotifPwms(name="toym", genome="toyg")
    pwms.read_motifscan_pwms(str(mdir / "toym_toyg_pwms.motifscan"))
    regions = load_motifscan_regions(str(workspace / "peaks.bed"), "bed")
    controls = generate_control_regions(2, regions, genome.chrom_sizes, random_seed=3)

    def as_sites(nested):
        return [[[(s.start, 1 if s.strand == "+" else 2) for s in cell] for cell in per] for per in nested]
    sites = as_sites(oracle_sites(genome, regions, pwms, 400, "both", "1e-3"))
    ctl = as_sites(oracle_sites(genome, controls, pwms, 400, "both", "1e-3"))
    table = cooccur_table(oracle_pairs(sites), len(regions), oracle_pairs(ctl), len(controls))
    anchors = [3, 7]
    rows = spacing_rows(oracle_spacing(sites, [p.length for p in pwms], anchors, 30), anchors, [p.length for p in pwms])
    ref = tmp_path / "ref"
    msio.write_cooccur_table(str(ref), pwms, table)
    msio.write_spacing_table(str(ref), pwms, anchors, rows)
    for name in ("motif_cooccurrence.xls", "motif_spacing.xls"):
        assert pairs[name] == (ref / name).read_bytes(), name
    assert len(rows) > 10 and table.n_both.sum() > 0

    assert cli.main(base + ["-o", str(tmp_path / "noenrich"), "--cooccur", "--no-enrich"]) == 0
    body = (tmp_path / "noenrich" / "motif_cooccurrence.xls").read_text().splitlines()[1:]
    assert body and all(line.endswith("\tNA\tNA\tNA\tNA\tNA") for line in body)
    assert os.path.getsize(tmp_path / "noenrich" / "motif_cooccurrence.xls") > 0
