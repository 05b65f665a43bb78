"""Whole-genome scans with the reference's de-duplication (`GenomeScanner(remove_dup=True)`, `scan --whole-genome`)
against the oracle bit for bit: whole-chromosome `c_scan_motif`, `make_motif_sites`, `deduplicate_motif_sites`.
Units as small as 64 bases cut chains of overlapping sites at many boundaries; the genome holds the cases that
make stitching hard (tandem repeats, chains on both strands, N runs under a cutoff <= 0)."""
import os

import numpy as np
import pytest

import oracle
from motifscan_b200 import _lib, cli, engine, synth
from motifscan_b200.genome import PackedGenome
from motifscan_b200.genome_scan import GenomeScanner, scan_genome
from motifscan_b200.region import GenomicRegion
from motifscan_b200.scanner import Scanner
from test_gpu_cli import _tree, workspace  # noqa: F401  (module fixture)
from test_gpu_parity import cutoffs_for, synth_pwms

pytestmark = pytest.mark.gpu
STRAND = {"+": 1, "-": 2, "both": 3}


def _at_motif(L=10):
    """A motif that hits ATATAT... at every other position on both strands (the repeat is its own reverse complement)."""
    pfm = np.full((4, L), 2, dtype=np.int64)
    pfm[0, 0::2] = 200
    pfm[3, 1::2] = 200
    return oracle.pfm_to_pwm(pfm, dict(A=0.295, C=0.205, G=0.205, T=0.295)).tolist()


@pytest.fixture(scope="module")
def genome():
    rng = np.random.default_rng(7)
    texts = {}
    for name, n in [("chr1", 9000), ("chr2", 5200), ("chr3", 33), ("chrM", 1571)]:
        s = bytearray(synth.random_bases(rng, n).tobytes())
        if n > 5000:
            s[1000:1400] = b"AT" * 200                       # tandem repeat over more than three 64-base units
            s[2000:2600] = b"N" * 600                        # N run: a chain of equal scores under a cutoff <= 0
            s[3000:3500] = bytes(s[3000:3500]).lower()       # soft-masked
        texts[name] = bytes(s)
    chroms = sorted(texts)
    packed = [synth.pack_ascii(np.frombuffer(texts[c], dtype=np.uint8)) for c in chroms]
    pg = PackedGenome(chroms, {c: len(texts[c]) for c in chroms}, np.concatenate([p[0] for p in packed]),
                      np.concatenate([p[1] for p in packed]), name="wg")
    whole = [texts[c].decode() for c in chroms]
    pwms = synth_pwms(rng, 62) + synth_pwms(rng, 6, lmin=33, lmax=40) + [_at_motif()] + synth_pwms(rng, 1, lmin=8, lmax=8)
    cutoffs = cutoffs_for(pwms, whole[:2], 3e-3)
    cutoffs[-2] = 0.9
    cutoffs[-1] = 0.0                                        # every all-N window scores 0 and hits
    return pg, pwms, cutoffs, whole


def expect(genome, strand):
    pg, pwms, cutoffs, whole = genome
    flat = oracle.c_scan_motif(pwms, cutoffs, whole, STRAND[strand], 8)
    nested = oracle.deduplicate_motif_sites(oracle.make_motif_sites(flat, [0] * len(whole)), [len(p[0]) for p in pwms])
    rows = [(m, c, s.start, s.score, 1 if s.strand == "+" else 2)
            for m, per in enumerate(nested) for c, cell in enumerate(per) for s in cell]
    cols = list(zip(*rows)) if rows else [[]] * 5
    counts = np.array([[len(cell) for cell in per] for per in nested], dtype=np.int64)
    best = np.array([[max(s.score for s in cell) if cell else np.nan for cell in per] for per in nested])
    return flat, dict(motif=np.array(cols[0], np.int32), chrom=np.array(cols[1], np.int32), start=np.array(cols[2], np.int32),
                      score=np.array(cols[3], np.float64), strand=np.array(cols[4], np.int8), counts=counts, best=best)


def assert_sites(sites, want):
    assert np.array_equal(sites.counts, want["counts"].sum(axis=1))
    assert np.array_equal(sites.motif, want["motif"])
    assert np.array_equal(sites.chrom_idx, want["chrom"]) and np.array_equal(sites.start, want["start"])
    assert np.array_equal(sites.strand, want["strand"])
    assert np.array_equal(np.asarray(sites.score).view(np.uint64), want["score"].view(np.uint64))


def assert_cells(sites, want):
    assert np.array_equal(sites.cell_counts, want["counts"])
    assert np.array_equal(sites.cell_best.view(np.uint64), want["best"].view(np.uint64))


def test_the_hard_cases_occur(genome):
    pg, pwms, cutoffs, whole = genome
    flat, want = expect(genome, "both")
    at = [s for s in flat[-2] if s[0] == 0 and 1000 <= s[1] < 1400]
    for x in (1, 2):                                          # both strands hit the repeat at consecutive even offsets
        starts = sorted(s[1] for s in at if s[3] == x)
        assert starts and starts[-1] - starts[0] >= 3 * 64 and max(np.diff(starts)) < len(pwms[-2][0])
    assert cutoffs[-1] <= 0
    nrun = [s for s in flat[-1] if s[0] == 0 and 2000 <= s[1] < 2600 - 8]
    assert len(nrun) >= 2 * (600 - 8) and all(s[2] == 0.0 for s in nrun)
    assert max(c for c in want["counts"].sum(axis=1)) > 0 and want["counts"].sum() > 500


@pytest.mark.parametrize("strand", ["+", "-", "both"])
@pytest.mark.parametrize("unit_bp", [1 << 26, 50000, 4096, 64])
def test_dedup_genome_scan_equals_reference(genome, unit_bp, strand):
    pg, pwms, cutoffs, _ = genome
    _, want = expect(genome, strand)
    for devices in ([0], [0, 0, 0]):
        gs = GenomeScanner(pg, pwms, cutoffs=cutoffs, strand=strand, devices=devices, unit_bp=unit_bp, remove_dup=True)
        try:
            sites = gs.scan()
            assert_cells(sites, want)
            assert_sites(sites, want)
            if unit_bp == 64:
                st = gs.last_stitch
                assert st["joined_chains"] > 0 and st["corrections"] > 0
                assert st["removed"] > 0                       # a right piece's site beat the left piece's survivor
            only = gs.scan(collect_sites=False)
            assert_cells(only, want)
            assert np.array_equal(only.counts, want["counts"].sum(axis=1)) and len(only.start) == 0
        finally:
            gs.close()


def test_dedup_genome_scan_equals_region_scanner(genome):
    pg, pwms, cutoffs, _ = genome
    regions = [GenomicRegion(c, 0, pg.chrom_sizes[c]) for c in pg.chroms]

    class P:
        def __init__(self, m, c):
            self.matrix, self.cutoffs, self.length = np.asarray(m), {"1e-4": c}, len(m[0])
    ps = [P(m, c) for m, c in zip(pwms, cutoffs)]
    ref = Scanner(genome=pg, regions=regions, window_size=0, remove_dup=True).scan_motifs(ps)
    gs = GenomeScanner(pg, pwms, cutoffs=cutoffs, unit_bp=64, remove_dup=True)
    try:
        got = gs.scan()
        assert np.array_equal(got.counts, ref.n_sites())
        assert np.array_equal(got.chrom_idx, ref._seq_idx) and np.array_equal(got.start, ref._start)
        assert np.array_equal(got.strand, ref._strand) and np.array_equal(got.score.view(np.uint64), ref._score.view(np.uint64))
    finally:
        gs.close()


def test_without_dedup_unchanged_and_scan_genome_routes(genome):
    pg, pwms, cutoffs, whole = genome
    counts, seq_idx, start, score, strand = oracle.scan_arrays(pwms, cutoffs, whole, 3, n_threads=8)
    gs = GenomeScanner(pg, pwms, cutoffs=cutoffs, unit_bp=64)
    try:
        sites = gs.scan()
        assert np.array_equal(sites.counts, counts) and np.array_equal(sites.start, start.astype(np.int32))
        assert np.array_equal(sites.score.view(np.uint64), score.view(np.uint64))
    finally:
        gs.close()
    _, want = expect(genome, "both")
    assert_sites(scan_genome(pg, pwms, cutoffs=cutoffs, remove_dup=True), want)
    with pytest.raises(ValueError):
        scan_genome(pg, pwms, cutoffs=cutoffs, remove_dup=True, resident=False)
    with pytest.raises(ValueError):
        GenomeScanner(pg, pwms, cutoffs=cutoffs, world=2, remove_dup=True)


def test_range_dedup_needs_one_range_per_sequence(genome):
    pg, pwms, cutoffs, whole = genome
    ctx = engine.default_context(0)
    motifs = engine.MotifSet(ctx, pwms, cutoffs)
    sset = engine.SequenceSet(ctx, whole)
    try:
        with pytest.raises(ValueError, match="not defined across range boundaries"):
            engine.scan_ranges(ctx, motifs, sset, 3, [(0, 0, 100), (0, 100, 200)], remove_dup=True)
        with pytest.raises(ValueError, match="not defined across range boundaries"):
            engine.scan_ranges_device(ctx, motifs, sset, 3, [(1, 0, 100), (1, 300, 400)], remove_dup=True)
        res = engine.scan_ranges(ctx, motifs, sset, 3, [(k, 0, len(w)) for k, w in enumerate(whole)], remove_dup=True)
        _, want = expect(genome, "both")
        assert np.array_equal(res.counts, want["counts"].sum(axis=1))
        res.close()
    finally:
        sset.close()
        motifs.close()


def test_cli_whole_genome_equals_chromosome_regions(workspace, tmp_path, monkeypatch):  # noqa: F811
    gdir, mdir = workspace / "toyg", workspace / "toym"
    if not (mdir / "toym_toyg_pwms.motifscan").exists():
        assert cli.main(["motif", "--build", str(mdir), "-g", str(gdir), "--n-random", "20000", "--seed", "1"]) == 0
    for stale in gdir.glob("toyg.packed.*"):
        stale.unlink()
    sizes = {"chr1": 60000, "chr2": 45000, "chrX": 30011}
    bed = tmp_path / "chroms.bed"
    bed.write_text("".join(f"{c}\t0\t{n}\n" for c, n in sorted(sizes.items())))
    common = ["-m", str(mdir), "-g", str(gdir), "-p", "1e-3"]
    for site in ([], ["--site"]):
        monkeypatch.setattr(cli, "PACKED_MIN_BP", 1 << 40)
        ref = tmp_path / f"ref{len(site)}"
        assert cli.main(["scan", "-i", str(bed), "-w", "0", "--no-enrich", "-o", str(ref)] + common + site) == 0
        want = _tree(ref)
        assert len(want) == 2 + (24 if site else 0)
        plain = tmp_path / f"plain{len(site)}"                       # no cache: packs from the FASTA
        assert cli.main(["scan", "--whole-genome", "-o", str(plain)] + common + site) == 0
        assert (gdir / "toyg.packed.chroms.tsv").exists()
        cached = tmp_path / f"cached{len(site)}"                     # from the cache it wrote
        assert cli.main(["scan", "--whole-genome", "-o", str(cached), "-w", "77", "--seed", "5"] + common + site) == 0
        assert _tree(plain) == want and _tree(cached) == want
        n = min(_lib.device_count(), 8)
        if n >= 2:
            multi = tmp_path / f"multi{len(site)}"
            assert cli.main(["scan", "--whole-genome", "-o", str(multi), "--gpus", str(n)] + common + site) == 0
            assert _tree(multi) == want
        for stale in gdir.glob("toyg.packed.*"):
            stale.unlink()
    with pytest.raises(SystemExit):
        cli.main(["scan", "--whole-genome", "-i", str(bed), "-o", str(tmp_path / "x")] + common)
    with pytest.raises(SystemExit):
        cli.main(["scan", "--whole-genome", "-c", str(bed), "-o", str(tmp_path / "y")] + common)
    assert not os.path.exists(tmp_path / "x") and not os.path.exists(tmp_path / "y")
