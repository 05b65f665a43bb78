"""GPU tests of the positional-centrality histograms (msb_scan_device_centrality, Scanner.scan_motifs(centrality=B),
`scan --centrality`) against an oracle built from oracle.c_scan_motif + oracle.deduplicate_motif_sites on host strings,
with d2, the bins and each cell's best site computed in Python.  Every count must be equal."""
import ctypes

import numpy as np
import pytest

import oracle
from motifscan_b200 import _lib, cli, engine
from motifscan_b200 import io as msio
from motifscan_b200.centrality import CentralityResult, centrality_rows, half_bins
from motifscan_b200.motif import MotifPwms, PositionWeightMatrix
from motifscan_b200.region import GenomicRegion, load_motifscan_regions
from motifscan_b200.scanner import Scanner
from test_gpu_cli import _tree, oracle_build, workspace  # noqa: F401
from test_gpu_cooccur import toy_genome
from test_gpu_parity import cutoffs_for, synth_pwms, synth_seqs

pytestmark = pytest.mark.gpu

STRAND = {"+": 1, "-": 2, "both": 3}


def oracle_hists(pwms, cutoffs, seqs, strand, dedup, mid2, B, H):
    """(hist_all, hist_best) int64[n_motifs, 2H + 1] of the final sites by the definitions."""
    lengths = [len(p[0]) for p in pwms]
    nested = oracle.make_motif_sites(oracle.c_scan_motif(pwms, cutoffs, seqs, strand, 4), [0] * len(seqs))
    if dedup:
        nested = oracle.deduplicate_motif_sites(nested, lengths)
    hist_all = np.zeros((len(pwms), 2 * H + 1), dtype=np.int64)
    hist_best = np.zeros_like(hist_all)

    def add(hist, m, d2):
        k = (d2 + B) // (2 * B)
        if -H <= k <= H:
            hist[m, k + H] += 1
    for m, per in enumerate(nested):
        for s, cell in enumerate(per):
            if mid2[s] < 0 or not cell:
                continue
            cell = sorted(cell, key=lambda x: (x.start, x.strand != "+"))    # the final order: start, then +
            best = cell[0]
            for site in cell:
                add(hist_all, m, 2 * site.start + lengths[m] - mid2[s])
                if site.score > best.score:
                    best = site
            add(hist_best, m, 2 * best.start + lengths[m] - mid2[s])
    return hist_all, hist_best


def device_hists(pwms, cutoffs, seqs, strand, dedup, mid2, B, H, shared=1):
    ctx = engine.Context(0)
    if not shared:
        ctx.set_option("centrality_shared", 0)
    motifs = engine.MotifSet(ctx, pwms, cutoffs)
    sset = engine.SequenceSet(ctx, seqs)
    try:
        engine.scan(ctx, motifs, sset, strand, remove_dup=dedup).close()
        return ctx.centrality(motifs, mid2, B, H)
    finally:
        sset.close(), motifs.close(), ctx.close()


def check(pwms, cutoffs, seqs, strand, dedup, mid2, B, H, min_sites=1):
    want = oracle_hists(pwms, cutoffs, seqs, strand, dedup, mid2, B, H)
    for shared in (1, 0):
        got = device_hists(pwms, cutoffs, seqs, strand, dedup, mid2, B, H, shared)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
    assert want[0].sum() >= min_sites
    return want


def dyadic_pwm(rng, L):
    return (rng.integers(-8, 9, size=(4, L)) / 4.0).tolist()


def tie_motifs(rng):
    """A reverse-complement palindrome (equal scores on both strands at one start) and a period-2 motif (equal scores
    at every other start of a tandem repeat), with dyadic entries so that the sums are exact."""
    half = np.array(dyadic_pwm(rng, 5))
    pal = np.concatenate([half, half[::-1, ::-1]], axis=1)          # column L-1-i = complement of column i
    a, b = np.array(dyadic_pwm(rng, 1)), np.array(dyadic_pwm(rng, 1))
    rep = np.concatenate([a, b] * 4, axis=1)
    return [pal.tolist(), rep.tolist()]


def consensus(pwm):
    return "".join("ACGT"[int(i)] for i in np.argmax(np.array(pwm), axis=0))


def route_case(seed, n_regions=60, lo=150, hi=420, rate=0.01):
    """Motifs on the three scan routes (<= 32, 33..64 and > 64 columns) plus the two tie motifs; sequences with N
    runs, some shorter than a motif, and planted palindromes and tandem repeats."""
    rng = np.random.default_rng(seed)
    pwms = synth_pwms(rng, 4, 6, 32) + synth_pwms(rng, 2, 33, 64) + synth_pwms(rng, 2, 65, 90) + tie_motifs(rng)
    seqs = synth_seqs(rng, n_regions, lo, hi, p_n=0.003)
    seqs[1] = "ACG"
    seqs[2] = "N" * 30 + seqs[2][30:]
    seqs[3] = seqs[3][:50]                                          # shorter than the long motifs
    pal, rep = consensus(pwms[-2]), consensus(pwms[-1])
    for r in range(4, n_regions, 3):
        s = list(seqs[r])
        at = int(rng.integers(0, len(s) - 60))
        s[at:at + 10] = pal
        s[at + 20:at + 44] = rep * 3
        seqs[r] = "".join(s)
    cutoffs = cutoffs_for(pwms, seqs, rate)
    return pwms, cutoffs, seqs


@pytest.mark.parametrize("B", [1, 3, 7, 10, 400, 1000])
def test_bins_and_routes(B):
    """Centred reference points: B = 1, odd B, and B > E (with B > 2E - 1 a single bin holds everything)."""
    pwms, cutoffs, seqs = route_case(1)
    mid2 = [len(s) for s in seqs]
    E = max(len(s) for s in seqs) // 2
    H = half_bins(E, B)
    got = check(pwms, cutoffs, seqs, 3, True, mid2, B, H, min_sites=100)
    lengths = [len(p[0]) for p in pwms]
    routes = [m for m in range(len(pwms)) if got[0][m].sum()]
    assert any(lengths[m] <= 32 for m in routes) and any(33 <= lengths[m] <= 64 for m in routes)
    assert any(lengths[m] > 64 for m in routes)
    assert got[0].shape[1] == 2 * H + 1 and (H == 0) == (B > 2 * E - 1)


@pytest.mark.parametrize("H", [0, 2, 5])
def test_half_bins_too_small_drop_sites(H):
    pwms, cutoffs, seqs = route_case(2)
    mid2 = [len(s) for s in seqs]
    want = check(pwms, cutoffs, seqs, 3, True, mid2, 10, H, min_sites=10)
    full = oracle_hists(pwms, cutoffs, seqs, 3, True, mid2, 10, 30)
    assert want[0].sum() < full[0].sum()


def test_excluded_and_off_centre_reference_points():
    """mid2 < 0 leaves a sequence out; mid2 = 0 and 2 len + 31 give the extreme d2 of both signs."""
    pwms, cutoffs, seqs = route_case(3)
    rng = np.random.default_rng(3)
    mid2 = []
    for s in seqs:
        kind = int(rng.integers(4))
        mid2.append([-1, 0, 2 * len(s) + 31, int(rng.integers(0, 2 * len(s) + 1))][kind])
    B = 3
    H = (2 * max(len(s) for s in seqs) + 120 + B) // (2 * B)
    want = check(pwms, cutoffs, seqs, 3, True, mid2, B, H, min_sites=100)
    assert want[0][:, :H - 20].sum() > 0 and want[0][:, H + 20:].sum() > 0


@pytest.mark.parametrize("strand", ["+", "-", "both"])
@pytest.mark.parametrize("dedup", [True, False])
def test_strands_dedup_and_ties(strand, dedup):
    pwms, cutoffs, seqs = route_case(4, rate=0.02)
    mid2 = [len(s) + 7 for s in seqs]
    got = check(pwms, cutoffs, seqs, STRAND[strand], dedup, mid2, 2, 120, min_sites=50)
    assert got[1][-2:].sum() > 10                                   # the tie motifs have best sites
    if strand == "both":
        nested = oracle.make_motif_sites(oracle.c_scan_motif(pwms, cutoffs, seqs, 3, 4), [0] * len(seqs))
        if dedup:
            nested = oracle.deduplicate_motif_sites(nested, [len(p[0]) for p in pwms])

        def best_ties(cell, same_start):
            top = max(x.score for x in cell)
            return any(a is not b and a.score == b.score == top and (a.start == b.start) == same_start
                       for a in cell for b in cell)
        assert any(best_ties(cell, True) for cell in nested[-2] if cell)     # palindrome: + and - at one start
        assert any(best_ties(cell, False) for cell in nested[-1] if cell)    # tandem repeat: several starts


def test_zero_sites_and_many_motifs_per_tile():
    """No site at all; and 300 motifs with few sites each, so that one CTA's tile spans more motifs than its shared
    histograms hold."""
    pwms, cutoffs, seqs = route_case(5)
    mid2 = [len(s) for s in seqs]
    got = device_hists(pwms, [1e9] * len(pwms), seqs, 3, True, mid2, 5, 40)
    assert got[0].shape == (len(pwms), 81) and not got[0].any() and not got[1].any()
    rng = np.random.default_rng(6)
    many = synth_pwms(rng, 300, 6, 14)
    seqs = synth_seqs(rng, 40, 200, 300)
    check(many, cutoffs_for(many, seqs, 0.003), seqs, 3, True, [len(s) for s in seqs], 1, 150, min_sites=300)


def pwm_set(mats, cut):
    pwms = MotifPwms()
    for i, (m, c) in enumerate(zip(mats, cut)):
        pwms.append(PositionWeightMatrix(m, name=f"TF{i}", matrix_id=f"M{i}", cutoffs={"1e-4": c}))
    return pwms


def test_scanner_paths_and_clipped_windows(tmp_path):
    """ASCII, resident-genome and Scanner(devices=[0, 0, 0]) paths over summit-centred windows, some clipped at both
    ends of a chromosome: equal to the oracle with the clipped windows left out."""
    from motifscan_b200.genome import DeviceGenome
    rng = np.random.default_rng(8)
    genome, regions = toy_genome(tmp_path, rng)
    regions += [GenomicRegion("chr1", 0, 40), GenomicRegion("chr1", 19900, 20000), GenomicRegion("chr2", 8950, 9000),
                GenomicRegion("chr2", 100, 300, summit=150)]
    mats = synth_pwms(rng, 30, 5, 16) + synth_pwms(rng, 2, 40, 70)
    W, B = 300, 7
    E = W // 2
    probe = Scanner(genome=genome, regions=regions, window_size=W)
    cut = cutoffs_for(mats, [s for s in probe.sequences if len(s) > 80], 0.01)
    pwms = pwm_set(mats, cut)
    lens = [len(s) for s in probe.sequences]
    mid2 = [2 * E if n == 2 * E else -1 for n in lens]
    assert 2 <= mid2.count(-1) < len(mid2) - 50
    H = half_bins(E, B)
    want = oracle_hists(mats, cut, probe.sequences, 3, True, mid2, B, H)
    assert want[1].sum() > 100
    dg = DeviceGenome(genome)
    try:
        for src, devices in ((genome, None), (dg, None), (genome, [0, 0, 0])):
            sc = Scanner(genome=src, regions=regions, window_size=W, devices=devices)
            got = sc.scan_motifs(pwms, centrality=B)
            c = got.centrality
            assert np.array_equal(c.hist_all, want[0]) and np.array_equal(c.hist_best, want[1])
            assert (c.n_tested, c.extend, c.bin) == (mid2.count(2 * E), E, B)
            plain = sc.scan_motifs(pwms)
            assert plain.centrality is None
            assert np.array_equal(plain.n_sites(), got.n_sites())
        with pytest.raises(ValueError):
            Scanner(genome=genome, regions=regions, window_size=0).scan_motifs(pwms, centrality=B)
    finally:
        dg.close()


def test_einval_cases():
    pwms, cutoffs, seqs = route_case(9, n_regions=20)
    n = len(seqs)
    mid2 = [len(s) for s in seqs]
    ctx, other_ctx = engine.Context(0), engine.Context(0)
    motifs = engine.MotifSet(ctx, pwms, cutoffs)
    foreign = engine.MotifSet(other_ctx, pwms, cutoffs)
    fewer = engine.MotifSet(ctx, pwms[:5], cutoffs[:5])
    sset = engine.SequenceSet(ctx, seqs)
    lib = ctx._lib
    try:
        engine.scan(ctx, motifs, sset, 3, remove_dup=True).close()
        m2 = np.asarray(mid2, dtype=np.int32)
        out = np.zeros((len(pwms), 3), dtype=np.int64)
        p32, p64 = _lib.ptr(m2, ctypes.c_int32), _lib.ptr(out, ctypes.c_int64)
        for args in ((None, p64, p64), (p32, None, p64), (p32, p64, None)):
            assert lib.msb_scan_device_centrality(ctx._h, motifs._h, n, args[0], 1, 1, args[1], args[2]) == _lib.MSB_EINVAL
        assert lib.msb_scan_device_centrality(ctx._h, None, n, p32, 1, 1, p64, p64) == _lib.MSB_EINVAL
        big = (_lib.CENTRALITY_MAX_CELLS // len(pwms) - 1) // 2 + 1   # the smallest half_bins over the cell cap
        for call in (lambda: ctx.centrality(foreign, mid2, 1, 1), lambda: ctx.centrality(fewer, mid2, 1, 1),
                     lambda: ctx.centrality(motifs, mid2[:-1], 1, 1), lambda: ctx.centrality(motifs, mid2 + [0], 1, 1),
                     lambda: ctx.centrality(motifs, mid2, 0, 1), lambda: ctx.centrality(motifs, mid2, -3, 1),
                     lambda: ctx.centrality(motifs, mid2, 1, -1), lambda: ctx.centrality(motifs, mid2, 1, big)):
            with pytest.raises(ValueError):
                call()
        engine.scan_device(ctx, motifs, sset, 3, counts_only=True)
        with pytest.raises(ValueError):
            ctx.centrality(motifs, mid2, 1, 1)
        engine.scan(ctx, motifs, sset, 3, compact=True).close()
        with pytest.raises(ValueError):
            ctx.centrality(motifs, mid2, 1, 1)
    finally:
        sset.close(), motifs.close(), foreign.close(), fewer.close(), ctx.close(), other_ctx.close()


def test_cli_tables_against_the_oracle(workspace, tmp_path):  # noqa: F811
    gdir, mdir = workspace / "toyg", workspace / "toym"
    if not (mdir / "toym_toyg_pwms.motifscan").exists():
        assert cli.main(["motif", "--build", str(mdir), "-g", str(gdir), "--n-random", "20000", "--seed", "1"]) == 0
    base = ["scan", "-i", str(workspace / "peaks.bed"), "-m", str(mdir), "-g", str(gdir), "-p", "1e-3", "-w", "400",
            "--site", "--n-random", "2", "--seed", "3"]
    assert cli.main(base + ["-o", str(tmp_path / "plain")]) == 0
    assert cli.main(base + ["-o", str(tmp_path / "cent"), "--centrality", "--centrality-bin", "5"]) == 0
    plain, cent = _tree(tmp_path / "plain"), _tree(tmp_path / "cent")
    assert set(cent) == set(plain) | {"motif_centrality.xls", "motif_site_distribution.xls"}
    assert all(cent[k] == v for k, v in plain.items())              # the other files are byte-identical

    genome, _ = oracle_build(gdir, mdir, 20000, 1)
    pwms = MotifPwms(name="toym", genome="toyg")
    pwms.read_motifscan_pwms(str(mdir / "toym_toyg_pwms.motifscan"))
    regions = load_motifscan_regions(str(workspace / "peaks.bed"), "bed")
    sc = Scanner(genome=genome, regions=regions, window_size=400)
    mid2 = [400 if len(s) == 400 else -1 for s in sc.sequences]
    H = half_bins(200, 5)
    hist_all, hist_best = oracle_hists([p.matrix.tolist() for p in pwms], [p.cutoffs["1e-3"] for p in pwms],
                                       sc.sequences, 3, True, mid2, 5, H)
    res = CentralityResult(hist_all, hist_best, sum(m >= 0 for m in mid2), 200, 5)
    ref = tmp_path / "ref"
    msio.write_centrality_tables(str(ref), pwms, res, centrality_rows(res, [p.length for p in pwms]))
    for name in ("motif_centrality.xls", "motif_site_distribution.xls"):
        assert cent[name] == (ref / name).read_bytes(), name
    assert hist_best.sum() > 50
