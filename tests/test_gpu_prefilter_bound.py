"""The tensor-core prefilter's superset guarantee (DESIGN §3) at the edges of its bound and of its table layout.

A window the prefilter does not flag is never re-scored, so a site it loses is gone without a trace.  These
tests aim at the places where the bound in `tc_fill_column` and the tile / batch layout of `ensure_tc_tables`
could go wrong: N bases behind column 32 of long motifs, lengths at every K-step edge, tiles and batches filled
exactly and overflowed by one, both tile orders, N runs at every alignment, and matrices of extreme magnitude.

Bar: bit-exact against the oracle (the discipline of test_gpu_parity.py), no tolerance.  Every test also checks
that the case it is about occurs in the oracle's result, so a change of seed or shape cannot turn it into a
plain random test.
"""
import numpy as np
import pytest

import oracle
from test_gpu_parity import assert_scan_equal, cutoffs_for, synth_pwms, synth_seqs

pytestmark = pytest.mark.gpu

ACGT = "ACGT"
K_STEP_EDGES = [1, 2, 7, 8, 9, 15, 16, 17, 23, 24, 25, 31, 32, 33, 40, 56, 63, 64, 65]


@pytest.fixture(scope="module")
def eng():
    from motifscan_b200 import engine
    return engine


# ---- helpers -----------------------------------------------------------------------------------------------
def strand_matrix(pwm, rev):
    """V[b][c]: what base b at window offset c adds on one strand (forward M[b][c], reverse M[3-b][L-1-c])."""
    m = np.asarray(pwm, dtype=np.float64)
    return m[::-1, ::-1] if rev else m


def best_bases(pwm, rev):
    return np.argmax(strand_matrix(pwm, rev), axis=0)


def window_score(pwm, window, rev):
    """The oracle's score of one window on one strand (the scan's arithmetic, cscore.c:344-357)."""
    return float(oracle.score_arrays([pwm], [window], 2 if rev else 1)[0, 0])


def is_site(score, cutoff):
    return score - cutoff >= -1e-10


def prefix(expect, n):
    """The oracle's result for the first n motifs of a set (sites are motif-major)."""
    counts, seq_idx, start, score, strand = expect
    k = int(counts[:n].sum())
    return counts[:n], seq_idx[:k], start[:k], score[:k], strand[:k]


def select_sites(expect, keep):
    counts, seq_idx, start, score, strand = expect
    motif = np.repeat(np.arange(len(counts)), counts)
    return (np.bincount(motif[keep], minlength=len(counts)).astype(counts.dtype), seq_idx[keep], start[keep],
            score[keep], strand[keep])


def site_windows(pwms, seqs, expect):
    """(motif, window text, strand is reverse, score) of every site of the oracle's result."""
    counts, seq_idx, start, score, strand = expect
    motif = np.repeat(np.arange(len(pwms)), counts)
    for k in range(len(score)):
        m = int(motif[k])
        L = len(pwms[m][0])
        yield m, seqs[seq_idx[k]][start[k]:start[k] + L], strand[k] == 2, float(score[k])


def trailing_n_traps(pwms, cutoffs, seqs, expect):
    """Sites of motifs longer than 32 columns whose window has A/C/G/T in its first 32 bases and non-ACGT bases
    only behind them, and which are no site once each of those bases is replaced by its column's best base: the
    sites a budget that counted the columns behind 32 at colmax would lose."""
    n = 0
    for m, w, rev, _ in site_windows(pwms, seqs, expect):
        if len(w) <= 32:
            continue
        bad = [i for i, ch in enumerate(w.upper()) if ch not in ACGT]
        if not bad or bad[0] < 32:
            continue
        bb = best_bases(pwms[m], rev)
        w2 = "".join(ACGT[bb[i]] if i in bad else ch for i, ch in enumerate(w))
        n += not is_site(window_score(pwms[m], w2, rev), cutoffs[m])
    return n


def expected_batches(lens, strand, interleave):
    """Prefilter launches of one scan of one range: mirrors the tile order and batching of ensure_tc_tables
    (motifs of 1..64 columns, sorted by length; 128 motifs per tile on strand 3, 256 otherwise; tiles of
    min(L, 32) / 8 K steps, rounded up; at most 24 K steps and 24 tiles per batch)."""
    fast = sorted(L for L in lens if 1 <= L <= 64)
    per = 128 if strand == 3 else 256
    tiles = [fast[k:k + per] for k in range(0, len(fast), per)]
    n_full = len(fast) // per
    if interleave and len(tiles) > 2:
        order, lo, hi, i = [], 0, n_full, 0
        while lo < hi:
            if i & 1:
                hi -= 1
                order.append(hi)
            else:
                order.append(lo)
                lo += 1
            i += 1
        tiles = [tiles[g] for g in order] + tiles[n_full:]
    batches, n_tiles, units = 0, 0, 0
    for t in tiles:
        ks = max(1, max((min(L, 32) + 7) // 8 for L in t))
        if n_tiles == 24 or units + ks > 24:
            batches, n_tiles, units = batches + 1, 0, 0
        n_tiles, units = n_tiles + 1, units + ks
    return batches + (n_tiles > 0)


def check_launches(ctx, n_batches):
    c = ctx.counters()
    if c["retries"] == 0:
        assert c["prefilter_launches"] == n_batches
    else:   # a buffer retry repeats the prefilter: every attempt launches every batch
        assert c["prefilter_launches"] % n_batches == 0 and c["prefilter_launches"] >= n_batches


def assert_sites(res, expect):
    """assert_scan_equal, with the site counts in the message when they differ."""
    assert res.n_sites == len(expect[3]), f"{len(expect[3])} oracle sites, {res.n_sites} returned"
    assert_scan_equal(res, expect)


def scan_equal(eng, ctx, pwms, cutoffs, seqs, strand, expect, limit=None):
    motifs = eng.MotifSet(ctx, pwms, cutoffs)
    sset = eng.SequenceSet(ctx, seqs)
    if limit is not None:
        sset.set_start_limit(limit)
    res = eng.scan(ctx, motifs, sset, strand)
    try:
        assert_sites(res, expect)
    finally:
        res.close(), sset.close(), motifs.close()


# ---- a. N behind column 32 of a 33-64-column motif ---------------------------------------------------------
def hand_built():
    """The three windows of the defect: an N at a column whose four entries are all negative, behind the 32
    columns the prefilter looks at, adds 0 -- more than the column's best base."""
    L = 40
    fwd = np.zeros((4, L))
    fwd[0, :32] = 2
    fwd[0, 32:39] = 1
    fwd[:, 39] = -10          # forward column 39: strand-1 window offset 39
    rev = np.zeros((4, L))
    rev[3, 1:] = 2
    rev[:, 0] = -10           # forward column 0: strand-2 window offset 39
    pwms = [fwd.tolist(), fwd.tolist(), rev.tolist()]
    cutoffs = [0.9, 0.75, 0.9]
    seqs = ["CCCCC" + "A" * 39 + "N" + "CCCCC",
            "CCCCC" + "AC" * 5 + "A" * 29 + "N" + "CCCCC",
            "GGGGG" + "A" * 39 + "N" + "GGGGG"]
    return pwms, cutoffs, seqs


@pytest.mark.parametrize("strand", [1, 2, 3])
def test_hand_built_trailing_n_sites(eng, strand):
    pwms, cutoffs, seqs = hand_built()
    expect = oracle.scan_arrays(pwms, cutoffs, seqs, strand)
    sites = {(m, w, rev, s) for m, w, rev, s in site_windows(pwms, seqs, expect)}
    if strand & 1:
        assert (0, "A" * 39 + "N", False, 1.0) in sites                         # 71 / 71; no site at all before
        assert (1, "AC" * 5 + "A" * 29 + "N", False, 61 / 71) in sites          # 51 / 71 with an A for the N
        assert window_score(pwms[1], "AC" * 5 + "A" * 30, False) < 0.75
    if strand & 2:
        assert (2, "A" * 39 + "N", True, 1.0) in sites
    assert trailing_n_traps(pwms, cutoffs, seqs, expect) >= {1: 2, 2: 1, 3: 3}[strand]
    ctx = eng.default_context(0)
    scan_equal(eng, ctx, pwms, cutoffs, seqs, strand, expect)


@pytest.fixture(scope="module")
def trailing():
    """36 motifs of 33-64 columns (log-odds and normal-valued) with one or two all-negative columns behind
    column 32 of each strand, 21 motifs of at most 32 columns beside them (one with an all-negative column at
    31), and windows planted for every long motif and strand: the strand's best bases, 0-3 substitutions among
    the first 32, N on the all-negative columns behind them.  Cutoffs: two thirds of the long motifs sit exactly
    on one planted window's score, the rest come from quantiles."""
    rng = np.random.default_rng(2401)
    pwms = []
    for i in range(36):
        L = int(rng.integers(33, 65))
        mat = np.round(rng.normal(0, 2, size=(4, L)), 3) if i % 2 else np.asarray(synth_pwms(rng, 1, L, L)[0])
        for lo, hi in ((32, L), (0, L - 32)):       # forward columns >= 32 serve strand 1, <= L - 33 strand 2
            for c in rng.choice(np.arange(lo, hi), size=min(2, hi - lo), replace=False):
                mat[:, c] = -np.round(rng.uniform(4.0, 10.0, size=4), 3)
        pwms.append(mat.tolist())
    short = synth_pwms(rng, 20, lmin=6, lmax=32)
    m32 = np.round(rng.normal(0, 2, size=(4, 32)), 3)
    m32[:, 31] = -5.0
    pwms += short + [m32.tolist()]
    planted = []                                    # (motif, reverse, window)
    for m in range(36):
        for rev in (0, 1):
            V = strand_matrix(pwms[m], rev)
            L = V.shape[1]
            behind = [c for c in range(32, L) if V[:, c].max() < 0]
            assert behind
            for k in range(4):
                b = best_bases(pwms[m], rev).copy()
                for c in rng.choice(32, size=k, replace=False):
                    b[c] = (b[c] + int(rng.integers(1, 4))) % 4
                w = [ACGT[x] for x in b]
                for c in (behind if k < 3 else behind[:1]):
                    w[c] = "N"
                w = "".join(w)
                planted.append((m, rev, w.lower() if k == 1 else w))
    order = rng.permutation(len(planted))
    seqs = synth_seqs(rng, 60, 800, 1200, p_n=0.001)
    bg = synth_seqs(rng, 400, 3, 40)
    starts = []                                     # (sequence, start) of every planted window
    for g in range(24):
        s = ""
        for j in order[g * 12:(g + 1) * 12]:
            s += bg[int(rng.integers(len(bg)))]
            starts.append((len(seqs), len(s)))
            s += planted[j][2]
        seqs.append(s + bg[int(rng.integers(len(bg)))])
    cutoffs = cutoffs_for(pwms, seqs, 2e-3)
    for m in range(36):
        if m % 3 != 2:
            w = [p[2] for p in planted if p[0] == m and p[1] == m % 2]
            cutoffs[m] = window_score(pwms[m], w[2], m % 2)
    return pwms, cutoffs, seqs, starts


@pytest.mark.parametrize("strand", [1, 2, 3])
def test_trailing_n_scan_and_ranges(eng, trailing, strand):
    pwms, cutoffs, seqs, starts = trailing
    expect = oracle.scan_arrays(pwms, cutoffs, seqs, strand, n_threads=8)
    assert trailing_n_traps(pwms, cutoffs, seqs, expect) >= 20
    ctx = eng.default_context(0)
    motifs = eng.MotifSet(ctx, pwms, cutoffs)
    sset = eng.SequenceSet(ctx, seqs)
    res = eng.scan(ctx, motifs, sset, strand)
    assert_sites(res, expect)
    res.close()
    # the same windows as ranges cut at and right behind every planted window's start: each such window is the
    # first start of one range and the last of another (a one-position range)
    cuts = {}
    for s, a in starts:
        cuts.setdefault(s, set()).update((a, a + 1))
    ranges = []
    for s, seq in enumerate(seqs):
        edges = [0] + sorted(cuts.get(s, ())) + [len(seq)]
        ranges += [(s, a, b) for a, b in zip(edges[:-1], edges[1:]) if b > a]
    res = eng.scan_ranges(ctx, motifs, sset, strand, ranges)
    assert_sites(res, expect)
    res.close(), sset.close(), motifs.close()


def test_trailing_n_score_select_pilot(eng):
    """msb_score_select's pilot path scans all samples with the pilot scores as cutoffs, through the same tables.
    Motifs of 33-48 columns with an all-negative column behind column 32 of each strand; 2000 samples per motif
    carry N there.  Those samples outscore their clean neighbours and reach the top ranks."""
    from motifscan_b200 import synth
    rng = np.random.default_rng(2402)
    n, width = 300000, 48
    pwms, n_offsets = [], []
    for L in (33, 40, 47, 48):
        mat = np.asarray(synth_pwms(rng, 1, L, L)[0])
        cf, cr = int(rng.integers(32, L)), int(rng.integers(0, L - 32))
        mat[:, cf] = -np.round(rng.uniform(8.0, 12.0, size=4), 3)
        mat[:, cr] = -np.round(rng.uniform(8.0, 12.0, size=4), 3)
        pwms.append(mat.tolist())
        n_offsets.append((cf, L - 1 - cr))           # window offsets >= 32 of the two columns
    pwms += synth_pwms(rng, 2, lmin=8, lmax=20)
    blob, off = synth.background_samples(n, width, seed=9)
    blob = blob.copy()
    picks = rng.permutation(n)[:2000 * 4].reshape(4, 2000)
    for j, offs in enumerate(n_offsets):
        for o in offs:
            blob[picks[j] * width + o] = ord("N")
    seqs = [blob[off[i]:off[i + 1]].tobytes().decode() for i in range(n)]
    ranks = [int(n * 0.1 ** e) - 1 for e in range(2, 6)] + [0]
    deepest = max(ranks)
    ctx = eng.Context(0)
    motifs = eng.MotifSet(ctx, pwms)
    sset = eng.SequenceSet(ctx, blob=blob, seq_off=off)
    try:
        for strand in (1, 2, 3):
            scores = oracle.score_arrays(pwms, seqs, strand)
            order = np.argsort(-scores, axis=1, kind="stable")
            want = np.take_along_axis(scores, order, axis=1)[:, ranks]
            if strand != 3:
                # trap: N samples in the top ranks that would fall below the depth the pilot sizes the candidate
                # set for (1.5 x the deepest rank) with the N replaced by the column's best base
                rev = strand == 2
                for j in range(4):
                    floor = scores[j, order[j, int(1.5 * (deepest + 1))]]
                    bb = best_bases(pwms[j], rev)
                    lost = 0
                    for i in set(order[j, :deepest + 1].tolist()) & set(picks[j].tolist()):
                        w = list(seqs[i][:len(pwms[j][0])])
                        o = n_offsets[j][rev]
                        w[o] = ACGT[bb[o]]
                        lost += window_score(pwms[j], "".join(w), rev) < floor
                    assert lost >= 30, (strand, j, lost)
            got = eng.score_select(ctx, motifs, sset, strand, ranks)
            assert ctx.counters()["retries"] == 0                       # the pilot path served every motif
            assert np.array_equal(got.view(np.uint64), np.ascontiguousarray(want).view(np.uint64)), strand
    finally:
        sset.close(), motifs.close(), ctx.close()


# ---- b. layout edges of the tables ---------------------------------------------------------------------------
def test_motif_lengths_at_every_k_step_edge(eng):
    """Motifs of every length at a K-step edge (8 bases per step) and at the prefilter's limits (32 columns seen,
    64 taken, 65 scored at every position): 30 of each -- log-odds, normal-valued, small integers -- so both tile
    orders have more than two tiles and a partial last one on every strand."""
    rng = np.random.default_rng(2403)
    pwms = []
    for L in K_STEP_EDGES:
        pwms += synth_pwms(rng, 10, L, L)
        pwms += np.round(rng.normal(0, 2, size=(10, 4, L)), 3).tolist()
        pwms += rng.integers(-3, 4, size=(10, 4, L)).astype(float).tolist()
    seqs = synth_seqs(rng, 60, 600, 1400, p_n=0.003, n_blocks=True)
    cutoffs = cutoffs_for(pwms, seqs, 3e-3)
    lens = [len(p[0]) for p in pwms]
    expect = {s: oracle.scan_arrays(pwms, cutoffs, seqs, s, n_threads=8) for s in (1, 2, 3)}
    for s in (1, 2, 3):
        per_len = np.bincount(np.repeat(lens, expect[s][0]), minlength=66)
        assert (per_len[K_STEP_EDGES] > 0).all(), s
    fast = sum(L <= 64 for L in lens)
    assert fast // 128 > 2 and fast % 128 and fast // 256 >= 2 and fast % 256
    for inter in (1, 0):
        ctx = eng.Context(0)             # tables are cached per motif set: a fresh context per tile order
        try:
            ctx.set_option("tc_interleave", inter)
            for s in (1, 2, 3):
                scan_equal(eng, ctx, pwms, cutoffs, seqs, s, expect[s])
                check_launches(ctx, expected_batches(lens, s, inter))
        finally:
            ctx.close()


def test_tiles_and_batches_filled_exactly_and_overflowed(eng):
    """25-32-column motifs: 4 K steps per tile, so six tiles are exactly one batch of 24 K steps.  Motif counts that
    fill one tile (128 on strand 3, 256 on strands 1 and 2) or six, and one more; and 3073 motifs, several batches on
    every strand.  Both tile orders.  The prefilter launch count proves the second batch."""
    rng = np.random.default_rng(2404)
    pool = synth_pwms(rng, 2800, lmin=25, lmax=32) + np.round(rng.normal(0, 2, size=(273, 4, 28)), 3).tolist()
    perm = rng.permutation(len(pool))
    pool = [pool[i] for i in perm]
    seqs = synth_seqs(rng, 20, 700, 1300, p_n=0.002, n_blocks=True)
    cutoffs = cutoffs_for(pool, seqs, 2e-3)
    counts = {3: [128, 129, 768, 769, 3073], 1: [256, 257, 1536, 1537, 3073], 2: [256, 257, 1536, 1537, 3073]}
    lens = [len(p[0]) for p in pool]
    assert [expected_batches(lens[:n], 3, 1) for n in counts[3]] == [1, 1, 1, 2, 5]
    assert [expected_batches(lens[:n], 1, 1) for n in counts[1]] == [1, 1, 1, 2, 3]
    expect = {s: oracle.scan_arrays(pool, cutoffs, seqs, s, n_threads=8) for s in (1, 2, 3)}
    for s in (1, 2, 3):
        assert (expect[s][0] > 0).sum() > 0.5 * len(pool)
    for inter in (1, 0):
        ctx = eng.Context(0)
        try:
            ctx.set_option("tc_interleave", inter)
            for s in (3, 1, 2):
                for n in counts[s]:
                    scan_equal(eng, ctx, pool[:n], cutoffs[:n], seqs, s, prefix(expect[s], n))
                    check_launches(ctx, expected_batches(lens[:n], s, inter))
        finally:
            ctx.close()


# ---- c. N runs at every alignment ------------------------------------------------------------------------------
def n_run_layout(rng):
    """Sequence 0 (64 position tiles of 512): N runs that start at every offset 0..31 of a 32-base block and end at
    every offset, short ones, ones longer than the 32-base horizon and ones longer than the longest motif; runs that
    end on a tile's last position, start on a tile's first, straddle a tile edge, and one that covers a tile and the
    horizon behind it.  Then 8 tiles of 8 sequences of 64 bases with start limits: in tile A_s only positions = s
    (mod 4) are live (N at 0..s-1, limit s + 1), in tile B_s only shifts s+1..3 (N at s, limit 4)."""
    n0 = 64 * 512
    s0 = np.frombuffer(synth_seqs(rng, 1, n0, n0, p_n=0.0)[0].encode(), dtype=np.uint8).copy()
    runs = []
    for a in range(32):
        for k, length in enumerate((1 + (7 * a) % 31, 33 + (11 * a) % 32, 130 + (30 - 2 * a) % 32)):   # the last ends at 31 - a
            start = 256 * (3 * a + k) + 64 + a
            runs.append((start, start + length))
    for e in range(50, 62, 2):
        E = 512 * e
        runs += [(E - 1 - e, E), (E, E + 1 + e), (E - 20, E + 20)]
    runs.append((512 * 62, 512 * 63 + 40))
    for a, b in runs:
        s0[a:b] = ord("N")
    starts = {a % 32 for a, _ in runs}
    ends = {(b - 1) % 32 for _, b in runs}
    assert starts == set(range(32)) and ends == set(range(32))
    seqs, limits = [s0.tobytes().decode()], [n0]
    for s in range(4):
        for tile in ("A", "B"):
            for _ in range(8):
                w = list(synth_seqs(rng, 1, 64, 64)[0])
                if tile == "A":
                    w[:s] = "N" * s
                    limits.append(s + 1)
                else:
                    w[s] = "N"
                    limits.append(4)
                seqs.append("".join(w))
    return seqs, np.array(limits, dtype=np.int32)


@pytest.mark.parametrize("cutoff_kind", ["positive", "zero", "negative_long"])
def test_n_runs_at_every_alignment(eng, cutoff_kind):
    """The producer's dirty / ignore bits, the shift skip (s_skip) and the all-N drop (taken when no cutoff admits a
    zero score, not taken when one does) at every alignment of an N run to the 32-base blocks and the 512-position
    tiles.  Sites behind the start limits are not reported, so the oracle's sites there are dropped."""
    rng = np.random.default_rng(2405)
    seqs, limits = n_run_layout(rng)
    pwms = synth_pwms(rng, 30, lmin=1, lmax=32) + synth_pwms(rng, 6, lmin=33, lmax=64)
    pwms.append(np.round(rng.normal(0, 2, size=(4, 48)), 3).tolist())
    cutoffs = [max(c, 0.05) for c in cutoffs_for(pwms, synth_seqs(rng, 20, 500, 800), 3e-3)]   # no all-N window is a site
    if cutoff_kind == "zero":
        cutoffs[0] = 0.0
    elif cutoff_kind == "negative_long":
        cutoffs[-1] = -0.3
    ctx = eng.default_context(0)
    for strand in (1, 2, 3):
        full = oracle.scan_arrays(pwms, cutoffs, seqs, strand, n_threads=8)
        expect = select_sites(full, full[2] < limits[full[1]])
        windows = list(site_windows(pwms, seqs, expect))
        all_n = [m for m, w, _, _ in windows if not set(w.upper()) & set(ACGT)]
        if cutoff_kind == "positive":
            assert not all_n
        elif cutoff_kind == "zero":
            assert len(all_n) > 500 and set(all_n) == {0}
        else:
            head_n = [s for m, w, _, s in windows if m == len(pwms) - 1 and not set(w[:32].upper()) & set(ACGT)]
            assert len(head_n) > 100 and min(head_n) < 0 < max(head_n)
        assert (expect[0] > 0).sum() > 20
        scan_equal(eng, ctx, pwms, cutoffs, seqs, strand, expect, limit=limits)


# ---- d. magnitude extremes ------------------------------------------------------------------------------------
def plant_consensus(rng, pwms, seqs, copies=2):
    """Append sequences holding each motif's best window on both strands (and lower-case copies)."""
    out = list(seqs)
    for p in pwms:
        s = ""
        for rev in (0, 1):
            w = "".join(ACGT[b] for b in best_bases(p, rev))
            for k in range(copies):
                s += synth_seqs(rng, 1, 3, 30)[0] + (w.lower() if k else w)
        out.append(s + "ACGT")
    return out


@pytest.mark.parametrize("scale", [2.0 ** -1000, 1e-30, 1e25, 1e30, 1e150])
def test_magnitude_extremes(eng, scale):
    """Production PWMs (4-64 columns) scaled so that the prefilter's budget hits its 1e-300 floor (2^-1000), the
    scale factor its 1e30 clamp (1e-30), and the dirty-window kernel's fp32 screen runs at a large magnitude (1e25)
    or is off (1e30, 1e150: the column maxima sum past 1e30).  A quarter of the motifs get a cutoff 0.5 raw units
    below their best window, so the budget is tiny."""
    rng = np.random.default_rng(2406)
    base = synth_pwms(rng, 40, lmin=4, lmax=64)
    seqs = plant_consensus(rng, base, synth_seqs(rng, 30, 600, 1200, p_n=0.003, n_blocks=True))
    pwms = [(np.asarray(p) * scale).tolist() for p in base]
    cutoffs = cutoffs_for(pwms, seqs, 3e-3)
    tight = list(range(0, 40, 4))
    for m in tight:
        cutoffs[m] = 1.0 - 0.5 / oracle.max_raw_score(base[m])
    abs_sum = np.array([np.abs(np.asarray(p)).max(axis=0).sum() for p in pwms])
    # the prefilter's budget sum colmax - T of the tight motifs (log-odds columns: colmax >= 0)
    budget = np.array([np.asarray(pwms[m]).max(axis=0).sum() - oracle.max_raw_score(pwms[m]) * (cutoffs[m] - 1e-10)
                       for m in tight])
    assert (budget > 0).all()
    if scale == 2.0 ** -1000:
        assert (budget < 1e-300).all()
    elif scale == 1e-30:
        assert ((384 - 6) / budget > 1e30).all()
    elif scale == 1e25:
        assert abs_sum.max() <= 1e30
    else:
        assert abs_sum.min() > 1e30
    ctx = eng.default_context(0)
    for strand in (1, 2, 3):
        expect = oracle.scan_arrays(pwms, cutoffs, seqs, strand, n_threads=8)
        assert all(expect[0][m] > 0 for m in tight)
        assert expect[0].sum() > 1000
        scan_equal(eng, ctx, pwms, cutoffs, seqs, strand, expect)


def test_cutoffs_at_one(eng):
    """Cutoffs 1.0 and 1 + 0.99e-10 keep a motif's best windows (score exactly 1.0 forward) as sites, 1 + 1.01e-10 keeps
    none.  Production PWMs and small-integer matrices whose columns tie for their maximum (any of the tied bases is a
    best window)."""
    rng = np.random.default_rng(2407)
    pwms = synth_pwms(rng, 20, lmin=4, lmax=64)
    for _ in range(16):
        L = int(rng.integers(3, 45))
        m = rng.integers(-3, 4, size=(4, L)).astype(float)
        mx = np.maximum(m.max(axis=0), 1.0)
        for c in range(L):
            rows = rng.choice(4, size=int(rng.integers(2, 4)), replace=False)
            m[rows, c] = mx[c]
        pwms.append(m.tolist())
    seqs = synth_seqs(rng, 20, 500, 900, p_n=0.003)
    for p in pwms:               # best windows with the tie broken at random
        for rev in (0, 1):
            W = strand_matrix(p, rev)
            w = "".join(ACGT[int(rng.choice(np.flatnonzero(W[:, c] == W[:, c].max())))] for c in range(W.shape[1]))
            seqs.append("TT" + w + "GA" + w.lower())
    ctx = eng.default_context(0)
    for cut, sites in ((1.0, True), (1.0 + 0.99e-10, True), (1.0 + 1.01e-10, False)):
        cutoffs = [cut] * len(pwms)
        for strand in (1, 2, 3):
            expect = oracle.scan_arrays(pwms, cutoffs, seqs, strand, n_threads=8)
            if sites:
                assert (expect[0] >= 2).all()
                if strand == 1:
                    assert (expect[3] == 1.0).all()
            else:
                assert expect[0].sum() == 0
            scan_equal(eng, ctx, pwms, cutoffs, seqs, strand, expect)
