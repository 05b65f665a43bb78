"""Positional centrality of motif sites around the region summits (`motifscan scan --centrality`): host statistics on
the histograms the device reduces from a region scan's final sites (engine.Context.centrality; DESIGN section 5.7).

    Every region is scanned in the window [summit - E, summit + E), E = window_size // 2.  A region is tested when its
    window is not clipped by a chromosome end (2E bases); the others are left out.  A site of motif m (length L) at
    start s has the doubled offset d2 = 2s + L - 2E from the window midpoint and lies in bin k = floor((d2 + B) / (2B))
    (centre offsets [kB - B/2, kB + B/2)); bins -K..K, K = floor((2E - 1 + B) / (2B)), hold every site.
    hist_all counts every site, hist_best each tested region's best-scoring site (ties: the first in start, strand +
    order), n_m = sum(hist_best[m]).
    Null: the best site's start is uniform over the 2E - L + 1 starts; p_m(j) is the exact fraction of starts whose d2
    falls in bins -j..j.  For j < J_m (the j with p_m(j) < 1), k_mj best sites in bins -j..j give
    p_mj = binom.sf(k_mj - 1, n_m, p_m(j)); the reported width is the j of the smallest p_mj (ties: smaller j), and
    p_corrected = min(1, p J_m M) over the M motifs with n_m > 0 and J_m > 0.  NA when n_m = 0 or J_m = 0.
"""
from collections import namedtuple

import numpy as np
from scipy.stats import binom

CentralityResult = namedtuple("CentralityResult", ["hist_all", "hist_best", "n_tested", "extend", "bin"])
CentralityResult.__doc__ = """`MotifSites.centrality`: `hist_all` / `hist_best` int64[n_motifs, 2K + 1] (bin k at column
k + K), the number of tested regions `n_tested`, the half-window E (`extend`) and the bin width B (`bin`)."""

CentralityRow = namedtuple("CentralityRow", ["motif", "length", "n_tested", "n_regions", "half_width", "central",
                                             "expected", "ratio", "p_value", "p_corrected"])


def half_bins(extend, bin):
    """K: bins -K..K hold every site of a 2E-base window."""
    return (2 * int(extend) - 1 + int(bin)) // (2 * int(bin))


def null_counts(length, extend, bin):
    """(counts int64[K + 1], starts): of the 2E - L + 1 starts of a motif of length L, the number whose d2 falls in
    bins -j..j, for j = 0..K (starts <= 0 when the motif does not fit)."""
    L, E, B = int(length), int(extend), int(bin)
    starts = 2 * E - L + 1
    j = np.arange(half_bins(E, B) + 1, dtype=np.int64)
    lo, hi = -(2 * j + 1) * B, (2 * j + 1) * B                 # lo <= d2 < hi, d2 = 2s + L - 2E
    s_lo = np.maximum(0, -((L - 2 * E - lo) // 2))             # ceil((lo - L + 2E) / 2)
    s_hi = np.minimum(starts - 1, (hi - L + 2 * E - 1) // 2)
    return np.maximum(s_hi - s_lo + 1, 0), starts


def centrality_rows(result, lengths):
    """One CentralityRow per motif, ordered like motif_centrality.xls: by (p_value with NaN last, -ratio, motif)."""
    best = np.asarray(result.hist_best, dtype=np.int64)
    n_motifs, width = best.shape
    K = (width - 1) // 2
    E, B = int(result.extend), int(result.bin)
    n = best.sum(axis=1)
    # central[m, j] = best sites in bins -j..j
    central = best[:, K:].copy()
    central[:, 1:] += best[:, K - 1::-1] if K else 0
    central = np.cumsum(central, axis=1)
    p_null = np.ones((n_motifs, K + 1))
    J = np.zeros(n_motifs, dtype=np.int64)
    by_length = {}
    for m, L in enumerate(lengths):
        if int(L) not in by_length:
            counts, starts = null_counts(L, E, B)
            by_length[int(L)] = (counts / starts, int((counts < starts).sum())) if starts > 0 else (None, 0)
        frac, J[m] = by_length[int(L)]
        if frac is not None:
            p_null[m] = frac
    tested = (n > 0) & (J > 0)
    M = int(tested.sum())
    cols = np.arange(K + 1)
    live = tested[:, None] & (cols[None, :] < J[:, None])
    p = np.full((n_motifs, K + 1), np.inf)
    p[live] = binom.sf(central[live] - 1, np.broadcast_to(n[:, None], live.shape)[live], p_null[live])
    rows = []
    for m in range(n_motifs):
        if not tested[m]:
            rows.append(CentralityRow(m, int(lengths[m]), int(result.n_tested), int(n[m]), None, None, float("nan"),
                                      float("nan"), float("nan"), float("nan")))
            continue
        j = int(np.argmin(p[m]))
        expected = float(n[m] * p_null[m, j])
        pv = float(p[m, j])
        rows.append(CentralityRow(m, int(lengths[m]), int(result.n_tested), int(n[m]), (j + 0.5) * B, int(central[m, j]),
                                  expected, int(central[m, j]) / expected, pv, min(1.0, pv * int(J[m]) * M)))
    rows.sort(key=lambda r: (np.isnan(r.p_value), 0.0 if np.isnan(r.p_value) else r.p_value,
                             0.0 if np.isnan(r.ratio) else -r.ratio, r.motif))
    return rows
