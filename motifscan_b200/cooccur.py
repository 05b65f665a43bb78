"""Motif co-occurrence and anchor spacing (`motifscan scan --cooccur` / `--spacing-anchor`): host statistics on the
counts the device reduces from a region scan's final sites (engine.Context.pair_counts / spacing).

    Pair counts   n_ab = regions with at least one site of motif a and one of motif b; n_aa = regions with a site of a.
    Within the input set, per pair a < b of N regions:
        expected = n_a n_b / N, ratio = n_ab / expected,
        p_cooccur = hypergeom.sf(n_ab - 1, N, n_a, n_b), p_exclusive = hypergeom.cdf(n_ab, N, n_a, n_b),
        q_cooccur = min(min(p_cooccur, p_exclusive) * n (n - 1) / 2, 1).
    Against the control regions: stats.py's enrichment test on the "has both" bit -- the 2 x 2 table
        [[n_ab, N - n_ab], [n_ab_control, N_control - n_ab_control]], fold change as stats.py:33, the one-sided Fisher
        tests as the exact hypergeom.cdf calls scipy.stats.fisher_exact makes (so the values equal it bit for bit), and
        Bonferroni over the n (n - 1) / 2 pairs.
    Spacing       hist[anchor][partner][orientation][d + D], orientation 0 same strand, 1 opposite, d in the anchor's
        frame (DESIGN section 5.6).  Per (anchor, partner, orientation) with at least one pair, only the offsets where the
        two windows do not overlap (d <= -L_partner or d >= L_anchor) are tested: n_bins such offsets within +-D hold T
        pairs, the peak is the fullest of them (ties: smallest |d|, then smallest d) with k pairs, and
        p_peak = min(1, n_bins * binom.sf(k - 1, T, 1 / n_bins)) (NaN when n_bins = 0).

The statistics are vectorised scipy calls over all pairs at once; `n_threads` > 1 cuts the arrays into chunks over a
thread pool.
"""
import concurrent.futures
from collections import namedtuple

import numpy as np
from scipy.stats import binom, hypergeom

PairSpec = namedtuple("PairSpec", ["cooccur", "anchors", "max_offset"], defaults=(False, (), 50))
PairSpec.__doc__ = """What `Scanner.scan_motifs(pwms, pairs=...)` reduces on the device after the scan: the pair counts
(`cooccur`) and the spacing histograms around the motifs at indices `anchors` (1..16 of them) up to |d| <= `max_offset`
(0..500)."""

PairResult = namedtuple("PairResult", ["counts", "n_regions", "spacing"])
PairResult.__doc__ = """`MotifSites.pairs`: `counts` int64[n, n] (None without `cooccur`), `n_regions`, and `spacing`
int64[n_anchors, n, 2, 2 D + 1] (None without anchors)."""

CooccurTable = namedtuple("CooccurTable", [
    "a", "b", "n_a", "n_b", "n_both", "expected", "ratio", "p_cooccur", "p_exclusive", "q_cooccur",
    "n_both_control", "fold_change", "p_enriched", "p_depleted", "p_corrected"])

SpacingRow = namedtuple("SpacingRow", ["anchor", "partner", "orientation", "pairs", "peak_offset", "peak_pairs", "expected",
                                       "p_value", "counts"])


def _chunked(fn, arrays, n_threads, min_chunk=1 << 16):
    """fn(*arrays) elementwise, on chunks of the arrays over `n_threads` threads when they are long enough."""
    n = len(arrays[0])
    if n_threads <= 1 or n < 2 * min_chunk:
        return fn(*arrays)
    bounds = np.linspace(0, n, min(n_threads, n // min_chunk) + 1).astype(np.int64)
    with concurrent.futures.ThreadPoolExecutor(max_workers=len(bounds) - 1) as pool:
        parts = list(pool.map(lambda k: fn(*[x[bounds[k]:bounds[k + 1]] for x in arrays]), range(len(bounds) - 1)))
    return np.concatenate(parts)


def fisher_greater_less(a, n_total, c, n_control_total, n_threads=1):
    """(p_greater, p_less) of scipy.stats.fisher_exact([[a, N - a], [c, Nc - c]], 'greater' / 'less') for arrays a, c:
    the same hypergeom.cdf calls, its p = 1.0 for a table with an empty row or column, and min(p, 1.0)."""
    a = np.asarray(a, dtype=np.int64)
    c = np.asarray(c, dtype=np.int64)
    n1, n2 = int(n_total), int(n_control_total)
    degenerate = (a + c == 0) | ((n1 - a) + (n2 - c) == 0) | (n1 == 0) | (n2 == 0)
    less = _chunked(lambda x, y: hypergeom.cdf(x, n1 + n2, n1, x + y), [a, c], n_threads)
    greater = _chunked(lambda x, y: hypergeom.cdf(n1 - x, n1 + n2, n1, (n1 - x) + (n2 - y)), [a, c], n_threads)
    greater = np.where(degenerate, 1.0, np.minimum(greater, 1.0))
    less = np.where(degenerate, 1.0, np.minimum(less, 1.0))
    return greater, less


def cooccur_table(counts, n_regions, control_counts=None, n_control_regions=None, n_threads=1):
    """Statistics of every motif pair a < b (CooccurTable of arrays in (a, b) order); the control columns are None
    without `control_counts`."""
    counts = np.asarray(counts, dtype=np.int64)
    n = counts.shape[0]
    a, b = np.triu_indices(n, k=1)
    single = np.diagonal(counts)
    n_a, n_b, n_ab = single[a], single[b], counts[a, b]
    N = int(n_regions)
    with np.errstate(divide="ignore", invalid="ignore"):
        expected = n_a * n_b / N if N > 0 else np.full(len(a), np.nan)
        ratio = n_ab / expected
    p_co = _chunked(lambda k, x, y: hypergeom.sf(k - 1, N, x, y), [n_ab, n_a, n_b], n_threads)
    p_ex = _chunked(lambda k, x, y: hypergeom.cdf(k, N, x, y), [n_ab, n_a, n_b], n_threads)
    n_pairs = n * (n - 1) // 2
    q = np.minimum(np.minimum(p_co, p_ex) * n_pairs, 1.0)
    ctl = [None] * 5
    if control_counts is not None:
        c = np.asarray(control_counts, dtype=np.int64)[a, b]
        Nc = int(n_control_regions)
        with np.errstate(divide="ignore", invalid="ignore"):
            fold = np.where((c > 0) & (N > 0), n_ab * Nc / np.maximum(c, 1) / max(N, 1), np.nan)   # stats.py:33
        p_up, p_down = fisher_greater_less(n_ab, N, c, Nc, n_threads)
        ctl = [c, fold, p_up, p_down, np.minimum(np.minimum(p_up, p_down) * n_pairs, 1.0)]
    return CooccurTable(a.astype(np.int32), b.astype(np.int32), n_a, n_b, n_ab, expected, ratio, p_co, p_ex, q, *ctl)


def cooccur_order(table):
    """Row order of motif_cooccurrence.xls: by (P_cooccur, -Ratio, a, b)."""
    return np.lexsort((table.b, table.a, -table.ratio, table.p_cooccur))


def spacing_rows(hist, anchors, lengths):
    """One SpacingRow per (anchor k, partner, orientation) with at least one pair, ordered by (P_value, k, partner,
    orientation); `anchors` are motif indices, `lengths` the motif lengths."""
    hist = np.asarray(hist, dtype=np.int64)
    n_anchors, n_motifs, _, width = hist.shape
    D = (width - 1) // 2
    d = np.arange(-D, D + 1)
    lengths = np.asarray(lengths, dtype=np.int64)
    rows = []
    for k in range(n_anchors):
        la = int(lengths[anchors[k]])
        for m in range(n_motifs):
            free = (d <= -int(lengths[m])) | (d >= la)      # the windows do not overlap
            n_bins = int(free.sum())
            order = np.flatnonzero(free)
            order = order[np.lexsort((d[order], np.abs(d[order])))]   # ties: smallest |d|, then smallest d
            for o in range(2):
                h = hist[k, m, o]
                total = int(h.sum())
                if total == 0:
                    continue
                if n_bins == 0:
                    rows.append(SpacingRow(k, m, o, total, None, None, float("nan"), float("nan"), h))
                    continue
                vals = h[order]
                best = int(order[int(np.argmax(vals))])
                t = int(vals.sum())
                peak = int(h[best])
                p = min(1.0, n_bins * float(binom.sf(peak - 1, t, 1.0 / n_bins)))
                rows.append(SpacingRow(k, m, o, total, int(d[best]), peak, t / n_bins, p, h))
    rows.sort(key=lambda r: (np.inf if np.isnan(r.p_value) else r.p_value, r.anchor, r.partner, r.orientation))
    return rows
