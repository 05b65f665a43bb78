"""Host tests of the positional-centrality statistics (motifscan_b200/centrality.py), its tables and the
`scan --centrality` flag validation."""
import numpy as np
import pytest
from scipy.stats import binom

from motifscan_b200 import cli
from motifscan_b200 import io as msio
from motifscan_b200.centrality import CentralityResult, centrality_rows, half_bins, null_counts
from motifscan_b200.motif import MotifPwms, PositionWeightMatrix


def brute_null(L, E, B):
    """Per j = 0..K, the starts s in 0..2E - L whose d2 = 2s + L - 2E is in bins -j..j, by the bin formula."""
    K = half_bins(E, B)
    bins = [(2 * s + L - 2 * E + B) // (2 * B) for s in range(2 * E - L + 1)]
    return [sum(abs(k) <= j for k in bins) for j in range(K + 1)], 2 * E - L + 1


@pytest.mark.parametrize("E", [1, 2, 7, 50, 51])
@pytest.mark.parametrize("B", [1, 2, 3, 10])
@pytest.mark.parametrize("L", [1, 2, 5, 6, 13, 14])
def test_null_counts_equal_enumeration(L, E, B):
    counts, starts = null_counts(L, E, B)
    want, want_starts = brute_null(L, E, B)
    assert starts == want_starts
    if starts > 0:
        assert counts.tolist() == want
        assert counts[-1] == starts                       # bins -K..K hold every start
        # every site's bin is in -K..K, and |d2| <= 2E - L
        assert all(abs(2 * s + L - 2 * E) <= 2 * E - L for s in range(starts))


def synth_result(rng, lengths, E, B, n_regions, central_frac=None):
    """Best-site histograms of uniform starts (plus, for motif 0, `central_frac` of regions within +-15 bp of the
    centre), and all-site histograms."""
    K = half_bins(E, B)
    best = np.zeros((len(lengths), 2 * K + 1), dtype=np.int64)
    for m, L in enumerate(lengths):
        for _ in range(n_regions):
            if rng.random() < 0.7:                    # a region with a site of m
                if m == 0 and central_frac and rng.random() < central_frac:
                    c = int(rng.integers(-15, 16))    # centre offset in bases
                    s = E + c - L // 2
                else:
                    s = int(rng.integers(0, 2 * E - L + 1))
                best[m, (2 * s + L - 2 * E + B) // (2 * B) + K] += 1
    return CentralityResult(best * 3, best, n_regions, E, B)


def test_rows_equal_direct_binom_calls():
    rng = np.random.default_rng(2)
    lengths = [8, 11, 20, 499, 500, 1000]
    E, B = 250, 10
    res = synth_result(rng, lengths[:3], E, B, 300)
    K = half_bins(E, B)
    best = np.zeros((len(lengths), 2 * K + 1), dtype=np.int64)
    best[:3] = res.hist_best
    best[3, K] = 4                                       # L = 2E - 1: J = 0 at B = 10
    best[5] = 0                                          # does not fit: no sites
    res = CentralityResult(best, best, 300, E, B)
    rows = centrality_rows(res, lengths)
    by = {r.motif: r for r in rows}
    M = 3
    for m in range(3):
        L = lengths[m]
        counts, starts = brute_null(L, E, B)
        J = sum(c < starts for c in counts)
        n = int(best[m].sum())
        ps = []
        for j in range(J):
            k = int(best[m, K - j:K + j + 1].sum())
            ps.append(float(binom.sf(k - 1, n, counts[j] / starts)))
        j = int(np.argmin(ps))
        r = by[m]
        assert r.n_regions == n and r.n_tested == 300 and r.length == L
        assert r.half_width == (j + 0.5) * B
        assert r.central == int(best[m, K - j:K + j + 1].sum())
        assert r.expected == n * (counts[j] / starts)
        assert r.ratio == r.central / r.expected
        assert r.p_value == ps[j]
        assert r.p_corrected == min(1.0, ps[j] * J * M)
    for m in (3, 4, 5):                                  # J = 0 (L = 2E - 1 with B > 1, L = 2E) or n = 0
        assert by[m].half_width is None and np.isnan(by[m].p_value) and np.isnan(by[m].p_corrected)
    assert by[3].n_regions == 4 and by[5].n_regions == 0
    assert [r.motif for r in rows[-3:]] == [3, 4, 5]     # NA last, by motif index
    finite = [(r.p_value, -r.ratio, r.motif) for r in rows[:3]]
    assert finite == sorted(finite)


def test_na_and_tie_rules():
    E, B = 10, 1
    K = half_bins(E, B)
    # L = 2E - 1 with B = 1: two starts, d2 = -1 (bin 0) and +1 (bin 1): J = 1
    best = np.zeros((4, 2 * K + 1), dtype=np.int64)
    best[0, K] = 3
    best[0, K + 1] = 3
    # motif 1 and 2: identical histograms -> equal p and ratio: ordered by motif index
    best[1, K] = best[2, K] = 5
    best[1, K + 4] = best[2, K + 4] = 2
    rows = centrality_rows(CentralityResult(best, best, 9, E, B), [19, 6, 6, 4])
    by = {r.motif: r for r in rows}
    assert by[0].half_width == 0.5 and by[0].central == 3 and by[0].expected == 3.0
    assert np.isnan(by[3].p_value) and by[3].central is None       # n = 0
    order = [r.motif for r in rows]
    assert order.index(1) + 1 == order.index(2)
    # p ties across widths: the smaller j wins (all sites at the extremes: p = 1 at every j)
    best = np.zeros((1, 2 * K + 1), dtype=np.int64)
    best[0, 0] = 2
    r = centrality_rows(CentralityResult(best, best, 2, E, B), [1])[0]
    assert r.p_value == 1.0 and r.half_width == 0.5


def test_planted_motif_ranks_first():
    rng = np.random.default_rng(7)
    lengths = [12, 8, 10, 15, 20, 9]
    E, B = 500, 10
    res = synth_result(rng, lengths, E, B, 400, central_frac=0.6)
    rows = centrality_rows(res, lengths)
    assert rows[0].motif == 0 and rows[0].p_corrected < 1e-6
    assert rows[0].half_width <= 25
    assert all(r.p_corrected > 0.01 for r in rows[1:])


def pwm_set(n):
    pwms = MotifPwms()
    for i in range(n):
        pwms.append(PositionWeightMatrix([[1, 0], [0, 1], [0, 0], [0, 0]], name=f"TF-{i}", matrix_id=f"MA{i}"))
    return pwms


def test_tables(tmp_path):
    E, B = 20, 10
    K = half_bins(E, B)
    assert K == 2
    best = np.array([[0, 1, 4, 1, 0], [0, 0, 0, 0, 0]], dtype=np.int64)
    res = CentralityResult(best * 2, best, 7, E, B)
    rows = centrality_rows(res, [2, 2])
    msio.write_centrality_tables(str(tmp_path), pwm_set(2), res, rows)
    lines = (tmp_path / "motif_centrality.xls").read_text().splitlines()
    assert lines[0] + "\n" == msio.CENTRALITY_HEADER
    r = rows[0]
    assert lines[1] == "\t".join(str(x) for x in ["MA0", "TF-0", 2, 7, 6, r.half_width, r.central, r.expected, r.ratio,
                                                  r.p_value, r.p_corrected])
    assert lines[2] == "MA1\tTF-1\t2\t7\t0\tNA\tNA\tNA\tNA\tNA\tNA"
    dist = (tmp_path / "motif_site_distribution.xls").read_text().splitlines()
    assert dist == ["Motif_ID\tMotif_name\tSites\t-20\t-10\t0\t10\t20", "MA0\tTF-0\tall\t0\t2\t8\t2\t0",
                    "MA0\tTF-0\tbest\t0\t1\t4\t1\t0", "MA1\tTF-1\tall\t0\t0\t0\t0\t0", "MA1\tTF-1\tbest\t0\t0\t0\t0\t0"]


def test_flag_validation():
    base = ["scan", "-i", "a.bed", "-m", "x", "-g", "y", "-o", "z", "--centrality"]
    with pytest.raises(SystemExit, match="--centrality"):
        cli.main(["scan", "--whole-genome", "-m", "x", "-g", "y", "-o", "z", "--centrality"])
    for w in ("0", "1"):
        with pytest.raises(SystemExit, match="-w 2 or more"):
            cli.main(base + ["-w", w])
    with pytest.raises(SystemExit, match="1..50"):
        cli.main(base + ["-w", "100", "--centrality-bin", "51"])
    with pytest.raises(SystemExit):
        cli.main(base + ["--centrality-bin", "0"])


def test_scanner_rejects_bad_geometry():
    from motifscan_b200.scanner import Scanner

    class G:
        chrom_sizes = {"c": 100}

        def fetch_sequence(self, chrom, a, b):
            return "A" * (b - a)
    for w, b in ((0, 1), (1, 1), (10, 6), (10, 0)):
        sc = Scanner(genome=G(), regions=[], window_size=w)
        with pytest.raises(ValueError, match="centrality"):
            sc.scan_motifs([], centrality=b)
