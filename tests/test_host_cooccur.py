"""Host tests of the co-occurrence statistics (motifscan_b200/cooccur.py), the native co-occurrence writer and the
`scan --cooccur` / `--spacing-anchor` flag validation."""
import numpy as np
import pytest
from scipy.stats import binom, fisher_exact, hypergeom

from motifscan_b200 import cli
from motifscan_b200 import io as msio
from motifscan_b200.cooccur import cooccur_order, cooccur_table, fisher_greater_less, spacing_rows
from motifscan_b200.motif import MotifPwms, PositionWeightMatrix


def bits(x):
    return np.asarray(x, dtype=np.float64).view(np.uint64)


def seeded_tables(rng, k):
    N, Nc = int(rng.integers(1, 400)), int(rng.integers(1, 400))
    a = rng.integers(0, N + 1, k)
    c = rng.integers(0, Nc + 1, k)
    a[:4] = [0, N, 0, N]                 # n_ab = 0 and n_ab = N, with empty and full control columns
    c[:4] = [0, Nc, Nc, 0]
    return a, N, c, Nc


@pytest.mark.parametrize("seed", range(6))
def test_vectorised_fisher_equals_fisher_exact(seed):
    rng = np.random.default_rng(seed)
    a, N, c, Nc = seeded_tables(rng, 300)
    up, down = fisher_greater_less(a, N, c, Nc)
    want_up = [fisher_exact([[x, N - x], [y, Nc - y]], "greater")[1] for x, y in zip(a, c)]
    want_down = [fisher_exact([[x, N - x], [y, Nc - y]], "less")[1] for x, y in zip(a, c)]
    assert np.array_equal(bits(up), bits(want_up))
    assert np.array_equal(bits(down), bits(want_down))


@pytest.mark.parametrize("N, Nc", [(0, 5), (5, 0), (0, 0)])
def test_fisher_with_an_empty_row(N, Nc):
    a, c = np.array([0, 0]), np.array([0, min(Nc, 1)])
    up, down = fisher_greater_less(a, N, c, Nc)
    assert np.array_equal(up, [1.0, 1.0]) and np.array_equal(down, [1.0, 1.0])
    for x, y, p in zip(a, c, up):
        assert fisher_exact([[x, N - x], [y, Nc - y]], "greater")[1] == p


def random_counts(rng, n, N):
    hits = rng.random((n, N)) < rng.uniform(0, 1, (n, 1))
    hits[0] = False                       # a motif without sites
    if n > 2:
        hits[1] = True                    # a motif in every region: n_ab = n_b
    h = hits.astype(np.int64)
    return h @ h.T


def test_cooccur_table_equals_scalar_scipy():
    rng = np.random.default_rng(3)
    n, N, Nc = 9, 120, 80
    counts, ctl = random_counts(rng, n, N), random_counts(rng, n, Nc)
    t = cooccur_table(counts, N, ctl, Nc)
    n_pairs = n * (n - 1) // 2
    assert len(t.a) == n_pairs
    for i, (a, b) in enumerate(zip(t.a, t.b)):
        na, nb, nab = counts[a, a], counts[b, b], counts[a, b]
        p_co = hypergeom.sf(nab - 1, N, na, nb)
        p_ex = hypergeom.cdf(nab, N, na, nb)
        assert bits(t.p_cooccur[i]) == bits(p_co) and bits(t.p_exclusive[i]) == bits(p_ex)
        assert bits(t.q_cooccur[i]) == bits(min(min(p_co, p_ex) * n_pairs, 1))
        c = ctl[a, b]
        up = fisher_exact([[nab, N - nab], [c, Nc - c]], "greater")[1]
        down = fisher_exact([[nab, N - nab], [c, Nc - c]], "less")[1]
        assert bits(t.p_enriched[i]) == bits(up) and bits(t.p_depleted[i]) == bits(down)
        assert bits(t.p_corrected[i]) == bits(min(min(up, down) * n_pairs, 1))
        fold = nab * Nc / c / N if c > 0 else np.nan
        assert bits(t.fold_change[i]) == bits(fold) or (np.isnan(fold) and np.isnan(t.fold_change[i]))
        assert t.expected[i] == na * nb / N
    order = cooccur_order(t)
    keys = [(t.p_cooccur[i], -t.ratio[i], t.a[i], t.b[i]) for i in order]
    finite = [k for k in keys if not np.isnan(k[1])]
    assert finite == sorted(finite)


def test_threaded_statistics_equal_single_threaded():
    rng = np.random.default_rng(4)
    counts = random_counts(rng, 420, 300)
    one = cooccur_table(counts, 300, counts, 300, n_threads=1)
    many = cooccur_table(counts, 300, counts, 300, n_threads=8)
    for x, y in zip(one, many):
        assert np.array_equal(bits(x), bits(y)) if x.dtype == np.float64 else np.array_equal(x, y)


def test_spacing_peak_tie_rule_and_no_free_bins():
    D = 4
    lengths = [2, 3, 9]
    hist = np.zeros((2, 3, 2, 2 * D + 1), dtype=np.int64)
    # anchor 0 (length 2) vs partner 1 (length 3): free offsets d <= -3 or d >= 2
    hist[0, 1, 0, -3 + D] = 5
    hist[0, 1, 0, 3 + D] = 5                # tie at |d| = 3: -3 wins (smallest d)
    hist[0, 1, 0, 0 + D] = 9                # overlapping: counted in Pairs, not tested
    hist[0, 1, 1, 2 + D] = 4
    hist[0, 1, 1, -4 + D] = 4               # tie: |d| = 2 wins
    hist[1, 2, 0, 1 + D] = 3                # anchor and partner of length 9: every offset in +-4 overlaps
    rows = {(r.anchor, r.partner, r.orientation): r for r in spacing_rows(hist, [0, 2], lengths)}
    rows = {(k[1], k[2]) if k[0] == 0 else (2, 0): r for k, r in rows.items()}
    assert len(rows) == 3 and set(rows) == {(1, 0), (1, 1), (2, 0)}
    r = rows[(1, 0)]
    n_bins = 2 + 3                           # d in {-4, -3} and {2, 3, 4}
    assert (r.pairs, r.peak_offset, r.peak_pairs) == (19, -3, 5)
    assert r.expected == 10 / n_bins
    assert r.p_value == min(1.0, n_bins * float(binom.sf(4, 10, 1 / n_bins)))
    assert rows[(1, 1)].peak_offset == 2
    r = rows[(2, 0)]
    assert r.peak_offset is None and np.isnan(r.p_value) and r.pairs == 3
    got = spacing_rows(hist, [0, 2], lengths)
    assert [x.p_value for x in got[:2]] == sorted(x.p_value for x in got[:2])
    assert np.isnan(got[-1].p_value)


def pwm_set(names):
    pwms = MotifPwms()
    for mid, name in names:
        pwms.append(PositionWeightMatrix([[1, 0], [0, 1], [0, 0], [0, 0]], name=name, matrix_id=mid))
    return pwms


def test_native_writer_equals_str(tmp_path):
    rng = np.random.default_rng(9)
    n, N = 7, 50
    pwms = pwm_set([(f"MA{i:04d}.1", f"TF-{i}") for i in range(n)])
    counts = random_counts(rng, n, N)
    for ctl in (random_counts(rng, n, 40), None):
        t = cooccur_table(counts, N, ctl, 40 if ctl is not None else None)
        msio.write_cooccur_table(str(tmp_path), pwms, t)
        got = (tmp_path / "motif_cooccurrence.xls").read_text()
        lines = [msio.COOCCUR_HEADER]
        names = [f"{p.matrix_id},{p.name}" for p in pwms]
        for i in cooccur_order(t):
            a, b = t.a[i], t.b[i]
            cells = [names[a], names[b], int(t.n_a[i]), int(t.n_b[i]), int(t.n_both[i])]
            cells += [float(getattr(t, f)[i]) for f in ("expected", "ratio", "p_cooccur", "p_exclusive", "q_cooccur")]
            if ctl is None:
                cells += ["NA"] * 5
            else:
                cells += [int(t.n_both_control[i])]
                cells += [float(getattr(t, f)[i]) for f in ("fold_change", "p_enriched", "p_depleted", "p_corrected")]
            lines.append("\t".join(str(x) for x in cells) + "\n")
        assert got == "".join(lines)
    # special values: nan, inf, exponents, integral floats
    t = cooccur_table(np.zeros((2, 2), np.int64), 0)
    msio.write_cooccur_table(str(tmp_path), pwm_set([("A", "a"), ("B", "b")]), t)
    assert (tmp_path / "motif_cooccurrence.xls").read_text().splitlines()[1].startswith("A,a\tB,b\t0\t0\t0\tnan\tnan\t")


def test_anchor_resolution():
    pwms = pwm_set([("MA1", "FOS"), ("MA2", "JUN"), ("MA3", "JUN"), ("MA4", "MA1")])
    assert cli.resolve_anchors(pwms, "MA2,FOS") == [1, 0]
    assert cli.resolve_anchors(pwms, "MA1") == [0]         # a matrix_id wins over a name
    with pytest.raises(SystemExit, match="ambiguous.*MA2,JUN.*MA3,JUN"):
        cli.resolve_anchors(pwms, "JUN")
    with pytest.raises(SystemExit, match="unknown"):
        cli.resolve_anchors(pwms, "NFAT")
    with pytest.raises(SystemExit, match="1 to 16"):
        cli.resolve_anchors(pwms, ",".join(["MA1"] * 17))


def test_flag_validation():
    with pytest.raises(SystemExit, match="--cooccur"):
        cli.main(["scan", "--whole-genome", "-m", "x", "-g", "y", "-o", "z", "--cooccur"])
    with pytest.raises(SystemExit, match="--spacing-anchor"):
        cli.main(["scan", "--whole-genome", "-m", "x", "-g", "y", "-o", "z", "--spacing-anchor", "MA1"])
    with pytest.raises(SystemExit):
        cli.main(["scan", "-i", "a.bed", "-m", "x", "-g", "y", "-o", "z", "--spacing-anchor", "MA1", "--spacing-max", "501"])
